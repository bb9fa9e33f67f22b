// twr_forward_generic.cu -- K2 for general layer stacks (SURVEY.md 8f row f4): batched Policy::_raw_predict
// (rust/src/nn/policy.rs:79-100) for policies whose `common`, `action_net` and `value_net` are arbitrary
// Sequentials of Linears (rust/src/nn/modules.rs:23-34, nn/layers.rs:24-38) -- BasicPolicy(common_layers=(256,128),
// policy_layers=(64,), value_layers=(64,)) and the like.  The configurations the reference ships (one common layer,
// single-Linear heads) run the tcgen05 / fp32 tile kernels instead; this one is plain fp32 SIMT: a CTA owns 16 envs,
// the activations of a layer live in shared memory, thread (env, o) accumulates out[o] = sum_i W[i][o] x[i] in
// ascending i and adds the bias afterwards (layers.rs:31-37), W reads coalesced along o.
#include "twr_kernels.cuh"

#include <atomic>
extern std::atomic<long long> g_twr_launches;

namespace {

constexpr int GT = 16;          // envs per CTA
constexpr int GTHREADS = 256;

__global__ void __launch_bounds__(GTHREADS) k_forward_generic(PolicyDev p, ForwardArgs a) {
    extern __shared__ __align__(16) float gsm[];
    const int64_t n = a.n_live_ptr ? (int64_t)*a.n_live_ptr : a.n;
    const int64_t tile0 = (int64_t)blockIdx.x * GT;
    if (tile0 >= n) return;
    const int tid = threadIdx.x;
    const int n_obs = p.n_obs, obs_size = p.obs_size, E = p.E, W = p.max_width;
    float* buf0 = gsm;                       // three activation buffers [GT][W]: input, output, and the trunk's result
    float* buf1 = gsm + GT * W;              // kept for the second head
    float* buf2 = gsm + 2 * GT * W;
    uint16_t* rows_s = reinterpret_cast<uint16_t*>(gsm + 3 * GT * W);   // [GT][n_obs]
    int8_t* perm_s = reinterpret_cast<int8_t*>(rows_s + GT * n_obs);    // [GT]

    // ---- observation rows (twist-in applied), one thread per env of the tile
    if (tid < GT) {
        const int64_t pos = tile0 + tid;
        int perm = -1;
        EnvState s = env_from_cells(make_uint4(0, 0, 0, 0));
        if (pos < n) {
            const int64_t e = a.live ? a.live[pos] : pos;
            if (!a.obs_rows) s = env_from_cells(a.cells[e]);
            if (a.perm_idx) {
                perm = a.perm_idx[pos];
            } else if (p.n_perms > 0 && a.t >= 0) {       // get_perm_id, nn/policy.rs:67-77
                uint32_t w[4];
                philox4x32_10(a.ids.gid((uint32_t)e), (uint32_t)a.t, TWR_RNG_PERM, a.cid, (uint32_t)a.seed,
                              (uint32_t)(a.seed >> 32), w);
                perm = (int)mulhi_u32(w[0], (uint32_t)p.n_perms);
            }
        }
        perm_s[tid] = (int8_t)perm;
        for (int i = 0; i < n_obs; ++i) {
            int row = 0;
            if (pos < n) row = a.obs_rows ? a.obs_rows[pos * n_obs + i] : i * a.env.N + (int)env_board(a.env, s, i);
            if (perm >= 0) row = p.obs_perms[(size_t)perm * obs_size + row];
            rows_s[tid * n_obs + i] = (uint16_t)row;
        }
    }
    __syncthreads();

    // ---- EmbeddingBag: bias, then the rows in observation order (layers.rs:57-62), optional ReLU
    for (int idx = tid; idx < GT * E; idx += GTHREADS) {
        const int env = idx / E, f = idx % E;
        float v = p.emb_b[f];
        const uint16_t* rr = rows_s + env * n_obs;
        for (int i = 0; i < n_obs; ++i) v += p.emb[(size_t)rr[i] * E + f];
        if (p.emb_relu) v = v > 0.f ? v : 0.f;
        buf0[env * W + f] = v;
    }
    __syncthreads();

    auto linear = [&](const PolicyDev::Lin& L, const float* in, float* out) {
        for (int idx = tid; idx < GT * L.out; idx += GTHREADS) {
            const int env = idx / L.out, o = idx % L.out;
            const float* x = in + env * W;
            float acc = 0.0f;
            for (int i = 0; i < L.in; ++i) acc = fmaf(L.w[(size_t)i * L.out + o], x[i], acc);
            acc += L.b[o];
            if (L.relu) acc = acc > 0.f ? acc : 0.f;
            out[env * W + o] = acc;
        }
        __syncthreads();
    };
    // trunk: ping-pong between buf0 and buf1; its result stays where it lands, the heads use the other two buffers
    float* cur = buf0;
    float* other = buf1;
    int li = 0;
    for (int k = 0; k < p.n_common; ++k, ++li) { linear(p.lin[li], cur, other); float* t = cur; cur = other; other = t; }
    float* trunk = cur;
    float* ha = other;          // scratch pair for the heads
    float* hb = buf2;
    const float* x = trunk;
    for (int k = 0; k < p.n_action; ++k, ++li) { float* out = (k & 1) ? hb : ha; linear(p.lin[li], x, out); x = out; }
    const float* logits_s = x;  // [GT][A] in the first A slots of each row
    // the value stack must not overwrite the logits: it alternates between the two buffers that do not hold them
    float* vfree0 = (logits_s == ha) ? hb : ha;
    float* vfree1 = trunk;      // the trunk is dead once the first value layer has read it
    x = trunk;
    for (int k = 0; k < p.n_value; ++k, ++li) { float* out = (k & 1) ? vfree1 : vfree0; linear(p.lin[li], x, out); x = out; }
    const float* value_s = x;

    if (tid < GT) {
        const int64_t pos = tile0 + tid;
        if (pos < n) {
            float l[4] = {0.f, 0.f, 0.f, 0.f};
            for (int o = 0; o < p.A; ++o) l[o] = logits_s[tid * W + o];
            float out[4] = {l[0], l[1], l[2], l[3]};
            const int perm = perm_s[tid];
            if (perm >= 0) {                                 // twist-out, nn/policy.rs:95-97
                for (int o = 0; o < p.A; ++o) {
                    const int src = p.act_perms[perm * p.A + o];
                    out[o] = src == 0 ? l[0] : src == 1 ? l[1] : src == 2 ? l[2] : l[3];
                }
            }
            a.logits[pos] = make_float4(out[0], out[1], out[2], out[3]);
            a.values[pos] = value_s[tid * W];               // value_net(h).sum() of a 1-wide output (policy.rs:88)
        }
    }
}

}  // namespace

size_t forward_generic_smem(const PolicyDev& p) {
    size_t b = sizeof(float) * 3 * (size_t)GT * p.max_width + sizeof(uint16_t) * (size_t)GT * (p.n_obs > 0 ? p.n_obs : TWR_MAX_CELLS) + GT;
    return (b + 15) & ~(size_t)15;
}

void launch_forward_generic(cudaStream_t st, const PolicyDev& p, const ForwardArgs& a) {
    if (a.n <= 0) return;
    const size_t sm = forward_generic_smem(p);
    cudaFuncSetAttribute(k_forward_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    k_forward_generic<<<(unsigned)((a.n + GT - 1) / GT), GTHREADS, sm, st>>>(p, a);
    g_twr_launches.fetch_add(1, std::memory_order_relaxed);
}
