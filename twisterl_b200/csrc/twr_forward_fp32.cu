// twr_forward_fp32.cu -- K2, fp32 SIMT variant: batched Policy::_raw_predict
// (rust/src/nn/policy.rs:79-100; EmbeddingBag/Linear rust/src/nn/layers.rs:31-86) for a tile of 128
// envs per CTA.
//
//   obs rows   : row_i = twist(i*N + board[i])                      (policy.rs:81-83)
//   embedding  : h1 = relu(bias + sum_i E[row_i])  in obs order     (layers.rs:57-62,81-84)
//   common     : h2 = relu(W1 h1 + b1), fp32 FMA, k ascending       (layers.rs:31-37)
//   heads      : logits = Wa h2 + ba ; value = wv.h2 + bv ; twist-out (policy.rs:89-97)
//
// The E dimension is streamed in chunks of KC features: the table slice E[:, kc] and W1[kc, :]
// are staged in shared memory with cp.async (double buffered), the h1 slice is produced by a
// conflict-free shared-memory gather, and the 128 x H output tile lives in registers
// (8 envs x H/16 columns per thread).  Bound: fp32 FMA pipe (2*E*H flop per env) -- this variant
// exists for the 1e-5 parity bar; the tensor-core variant is twr_forward_tc2.cu.
//
// COMPACT (GridWorld boards of 33..64 cells, PolicyDev::compact_n = N): a GridWorld observation only reaches table
// rows i*N + v with v in 0..3 (examples/grid_world/src/lib.rs:74-81), so each KC slice stages those 4N rows alone, row
// i*N + v at i*4 + v.  The cells are summed in the same order from the same values: the full-table arithmetic, bit for bit.
#include "twr_kernels.cuh"

#include <atomic>
extern std::atomic<long long> g_twr_launches;

namespace {

constexpr int TM = 128;       // envs per CTA
constexpr int NTHREADS = 256;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

template <int H, int KC, bool COMPACT>
__global__ void __launch_bounds__(NTHREADS, 1) k_forward_fp32(PolicyDev p, ForwardArgs a) {
    constexpr int TN = H / 16;      // output columns per thread
    constexpr int LPF = KC / 4;     // lanes covering one env's KC features with float4
    constexpr int EG = 32 / LPF;    // envs handled per warp instruction in the gather
    extern __shared__ __align__(16) unsigned char smem_raw[];

    const int64_t n = a.n_live_ptr ? (int64_t)*a.n_live_ptr : a.n;
    const int64_t tile0 = (int64_t)blockIdx.x * TM;
    if (tile0 >= n) return;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_obs = p.n_obs, obs_size = p.obs_size, E = p.E;
    const int cn = COMPACT ? p.compact_n : 0;
    const int tab_rows = COMPACT ? 4 * cn : obs_size;              // staged rows of the table

    float* Es = reinterpret_cast<float*>(smem_raw);                 // [2][tab_rows*KC]
    float* Ws = Es + 2 * (size_t)tab_rows * KC;                     // [2][KC*H]
    float* As = Ws + 2 * (size_t)KC * H;                            // [TM][KC]
    uint16_t* rows_s = reinterpret_cast<uint16_t*>(As + TM * KC);   // [TM][n_obs]
    int8_t* perm_s = reinterpret_cast<int8_t*>(rows_s + TM * n_obs); // [TM]

    auto issue_chunk = [&](int kc, int buf) {
        float* es = Es + (size_t)buf * tab_rows * KC;
        const int e_pieces = tab_rows * LPF;
        for (int q = tid; q < e_pieces; q += NTHREADS) {
            const int row = q / LPF, c4 = q % LPF;
            const int src = COMPACT ? (row >> 2) * cn + (row & 3) : row;
            cp_async16(es + row * KC + c4 * 4, p.emb + (size_t)src * E + kc * KC + c4 * 4);
        }
        float* ws = Ws + (size_t)buf * KC * H;
        const float* wsrc = p.w1 + (size_t)kc * KC * H;
        for (int q = tid; q < KC * H / 4; q += NTHREADS) cp_async16(ws + q * 4, wsrc + q * 4);
        cp_async_commit();
    };
    issue_chunk(0, 0);

    // ---- observation rows (twist-in applied), one thread per env of the tile
    if (tid < TM) {
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
            if (COMPACT) row = (row / cn) * 4 + row % cn;             // the twists keep v in 0..3 (twr_policy_create)
            rows_s[tid * n_obs + i] = (uint16_t)row;
        }
    }

    const int mg = tid >> 4, ng = tid & 15;
    float acc[8][TN];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < TN; ++c) acc[i][c] = 0.0f;

    const int n_chunks = E / KC;
    for (int kc = 0; kc < n_chunks; ++kc) {
        const int buf = kc & 1;
        cp_async_wait<0>();
        __syncthreads();   // chunk kc landed for everyone; FMA phase kc-1 is done with As and buffer buf^1
        if (kc + 1 < n_chunks) issue_chunk(kc + 1, buf ^ 1);   // overlaps this chunk's gather + FMA

        // ---- embedding slice: As[env][f] = relu(bias[f] + sum_i Es[row_i][f])
        {
            const float* es = Es + (size_t)buf * tab_rows * KC;
            const int f4 = lane % LPF, eg = lane / LPF;
            const float4 bias = *reinterpret_cast<const float4*>(p.emb_b + kc * KC + f4 * 4);
#pragma unroll 2
            for (int it = 0; it < 16 / EG; ++it) {
                const int env = warp * 16 + it * EG + eg;
                float4 v = bias;
                const uint16_t* rr = rows_s + env * n_obs;
                for (int i = 0; i < n_obs; ++i) {
                    const float4 r = *reinterpret_cast<const float4*>(es + (int)rr[i] * KC + f4 * 4);
                    v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
                }
                v.x = v.x > 0.f ? v.x : 0.f; v.y = v.y > 0.f ? v.y : 0.f;
                v.z = v.z > 0.f ? v.z : 0.f; v.w = v.w > 0.f ? v.w : 0.f;
                *reinterpret_cast<float4*>(As + env * KC + f4 * 4) = v;
            }
        }
        __syncthreads();

        // ---- acc[128 x H] += As[128 x KC] * Ws[KC x H]
        {
            const float* ws = Ws + (size_t)buf * KC * H;
#pragma unroll 2
            for (int k = 0; k < KC; k += 4) {
                float4 av[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) av[i] = *reinterpret_cast<const float4*>(As + (mg * 8 + i) * KC + k);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    float w[TN];
#pragma unroll
                    for (int j = 0; j < TN / 4; ++j) {
                        const float4 t = *reinterpret_cast<const float4*>(ws + (k + kk) * H + j * 64 + ng * 4);
                        w[j * 4 + 0] = t.x; w[j * 4 + 1] = t.y; w[j * 4 + 2] = t.z; w[j * 4 + 3] = t.w;
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float x = kk == 0 ? av[i].x : kk == 1 ? av[i].y : kk == 2 ? av[i].z : av[i].w;
#pragma unroll
                        for (int c = 0; c < TN; ++c) acc[i][c] = fmaf(x, w[c], acc[i][c]);
                    }
                }
            }
        }
    }

    // ---- heads: bias + ReLU, then 4 logits + value as partial dots reduced over the 16 column lanes
    float part[8][5];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int o = 0; o < 5; ++o) part[i][o] = 0.0f;
#pragma unroll
    for (int c = 0; c < TN; ++c) {
        const int col = (c >> 2) * 64 + ng * 4 + (c & 3);
        const float b1 = __ldg(p.b1 + col);
        float wa[4];
#pragma unroll
        for (int o = 0; o < 4; ++o) wa[o] = (o < p.A) ? __ldg(p.wa + (size_t)col * p.A + o) : 0.0f;
        const float wv = __ldg(p.wv + col);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float h = acc[i][c] + b1;
            h = h > 0.f ? h : 0.f;
#pragma unroll
            for (int o = 0; o < 4; ++o) part[i][o] = fmaf(h, wa[o], part[i][o]);
            part[i][4] = fmaf(h, wv, part[i][4]);
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int o = 0; o < 5; ++o) {
            float v = part[i][o];
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            part[i][o] = v;
        }
    if (ng == 0) {
        const float bv = __ldg(p.bv);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int m = mg * 8 + i;
            const int64_t pos = tile0 + m;
            if (pos >= n) continue;
            float l[4];
#pragma unroll
            for (int o = 0; o < 4; ++o) l[o] = (o < p.A) ? part[i][o] + __ldg(p.ba + o) : 0.0f;
            const int perm = perm_s[m];
            float out[4] = {l[0], l[1], l[2], l[3]};
            if (perm >= 0) {                                 // twist-out, nn/policy.rs:95-97
#pragma unroll
                for (int o = 0; o < 4; ++o) {
                    if (o < p.A) {
                        const int src = p.act_perms[perm * p.A + o];
                        out[o] = src == 0 ? l[0] : src == 1 ? l[1] : src == 2 ? l[2] : l[3];
                    }
                }
            }
            a.logits[pos] = make_float4(out[0], out[1], out[2], out[3]);
            a.values[pos] = part[i][4] + bv;
        }
    }
}

template <int H, int KC>
size_t smem_bytes(const PolicyDev& p, int n_obs) {
    const size_t rows = p.compact_n > 0 ? 4 * (size_t)p.compact_n : (size_t)p.obs_size;
    size_t b = sizeof(float) * (2 * rows * KC + 2 * (size_t)KC * H + (size_t)TM * KC);
    b += sizeof(uint16_t) * (size_t)TM * n_obs + TM;
    return (b + 15) & ~(size_t)15;
}

constexpr size_t SMEM_LIMIT = 227 * 1024;

template <int H, int KC>
void launch_kc(cudaStream_t st, const PolicyDev& p, const ForwardArgs& a, unsigned grid) {
    const size_t sm = smem_bytes<H, KC>(p, p.n_obs);
    auto kern = p.compact_n > 0 ? k_forward_fp32<H, KC, true> : k_forward_fp32<H, KC, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    kern<<<grid, NTHREADS, sm, st>>>(p, a);
}

// n_obs: the observation length the fit is sized for (the launch's own, p.n_obs, when not dry)
template <int H>
bool launch_h(cudaStream_t st, const PolicyDev& p, const ForwardArgs& a, int n_obs, bool dry) {
    const unsigned grid = (unsigned)((a.n + TM - 1) / TM);
    if (p.E % 32 == 0 && smem_bytes<H, 32>(p, n_obs) <= SMEM_LIMIT) {
        if (dry) return true;
        launch_kc<H, 32>(st, p, a, grid);
    } else if (p.E % 16 == 0 && smem_bytes<H, 16>(p, n_obs) <= SMEM_LIMIT) {
        if (dry) return true;
        launch_kc<H, 16>(st, p, a, grid);
    } else {
        return false;
    }
    g_twr_launches.fetch_add(1, std::memory_order_relaxed);
    return true;
}

bool dispatch(cudaStream_t st, const PolicyDev& p, const ForwardArgs& a, int n_obs, bool dry) {
    switch (p.H) {
        case 64: return launch_h<64>(st, p, a, n_obs, dry);
        case 128: return launch_h<128>(st, p, a, n_obs, dry);
        case 192: return launch_h<192>(st, p, a, n_obs, dry);
        case 256: return launch_h<256>(st, p, a, n_obs, dry);
        default: return false;
    }
}

}  // namespace

int forward_fp32_supported(const PolicyDev& p, int n_obs, const char** why) {
    static const char* msg_h = "common width must be 64, 128, 192 or 256";
    static const char* msg_e = "embedding size must be a multiple of 16 and the table slice must fit shared memory";
    static const char* msg_o = "obs_size must be < 65536 and obs per env <= 64";
    if (p.H != 64 && p.H != 128 && p.H != 192 && p.H != 256) { *why = msg_h; return 0; }
    if (p.obs_size >= 65536 || n_obs > TWR_MAX_OBS) { *why = msg_o; return 0; }
    ForwardArgs a{};
    a.n = 1;
    if (!dispatch(nullptr, p, a, n_obs, true)) { *why = msg_e; return 0; }
    return 1;
}

bool launch_forward_fp32(cudaStream_t st, const PolicyDev& p, const ForwardArgs& a) {
    if (a.n <= 0) return true;
    return dispatch(st, p, a, p.n_obs, false);
}
