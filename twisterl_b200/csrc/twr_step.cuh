// twr_step.cuh -- K3 + K4a + K1: one record of PPOCollector::single_collect's loop (collector/ppo.rs:69-80)
// for one env, shared by the stand-alone k_collect_step kernel and the fused epilogue of the
// tensor-core forward (twr_forward_tc2.cu).
#pragma once
#include "twr_kernels.cuh"

// Must be called by all 32 lanes of a warp (`active` false for padding lanes): reward(s_t), masked
// logits, value, Gumbel-max action and twist index go to record [t][env]; terminal states are recorded
// and retire (their action is not applied), the rest step and are appended to the next live list with
// one atomicAdd per warp (ballot + popc prefix).  F: the cell encodings the caller is compiled for (twr_common.cuh).
template <int F = TWR_CELLS_ANY>
__device__ __forceinline__ void collect_step_body(const StepArgs& a, const CollectBuffers& b, bool active, int e,
                                                  float4 raw, float value, int perm, int32_t* __restrict__ live_next) {
    bool survives = false;
    if (active) {
        EnvState s = env_load(b.cells, b.meta, e);
        const uint32_t gid = a.ids.gid((uint32_t)e);
        const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
        const uint32_t m = env_masks(a.env, s);
        float l[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) l[i] = (i < a.A) ? (((m >> i) & 1u) ? l[i] : -1e10f) : 0.0f;  // policy.rs:62

        uint32_t w[4];
        philox4x32_10(gid, (uint32_t)a.t, TWR_RNG_SAMPLE, a.cid, k0, k1, w);
        const float u[4] = {u32_to_unit_f32(w[0]), u32_to_unit_f32(w[1]), u32_to_unit_f32(w[2]), u32_to_unit_f32(w[3])};
        const int act = sample_from_logits4(l, u, a.A);
        const float rew = env_reward<F>(a.env, s);
        const bool fin = env_is_final<F>(a.env, s);

        const int64_t r = (int64_t)a.t * b.B + e;
        b.rec_state[r] = env_pack_cells(s);
        b.rec_logits[r] = make_float4(l[0], l[1], l[2], l[3]);
        b.rec_value[r] = value;
        b.rec_reward[r] = rew;
        b.rec_action[r] = (uint8_t)act;
        b.rec_perm[r] = (int8_t)perm;

        if (fin) {
            b.ep_len[e] = a.t + 1;
            if (env_success<F>(a.env, s)) atomicAdd(&b.stats[0], 1ull);
            atomicAdd(reinterpret_cast<double*>(&b.stats[2]), (double)rew);
        } else {
            env_step<F>(a.env, s, act);
            env_store(b.cells, b.meta, e, s);
            survives = true;
        }
    }
    if (!live_next) return;          // multi-step chunks re-compact the live list between launches instead
    const unsigned bal = __ballot_sync(0xffffffffu, survives);
    if (bal) {
        const int lane = threadIdx.x & 31;
        int base = 0;
        if (lane == 0) base = atomicAdd(&b.n_live[a.t + 1], __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (survives) live_next[base + __popc(bal & ((1u << lane) - 1u))] = e;
    }
}
