// twr_kernels.cu -- the HBM-bound kernels of the rollout engine (sm_100a):
//   K1  batched Env trait (reset / set_state / forced step / observe / masks / reward / is_final)
//   K3  mask + Gumbel-max sampling (Philox), fused in collect_step with
//   K4a trajectory write, env step and warp-ballot live-list compaction
//   K4b GAE reverse scan
//   K5  episode offsets (merge order) + transpose/compaction into concatenated episodes
// All are one-thread-per-env, 16-byte vector state loads, time-major [t][env] record stores
// (coalesced), grids sized from the env count.  Algorithmic bytes per record are listed in DESIGN.md.
#include "twr_kernels.cuh"
#include "twr_step.cuh"

#include <atomic>

std::atomic<long long> g_twr_launches{0};
#define TWR_COUNT_LAUNCH() g_twr_launches.fetch_add(1, std::memory_order_relaxed)

static inline unsigned grid_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }

// ------------------------------------------------------------------------- K1 ---
__global__ void __launch_bounds__(256) k_envs_reset(EnvParams p, uint4* __restrict__ cells, uint32_t* __restrict__ meta,
                                                    int64_t n, uint64_t seed, EnvIds ids, uint32_t cid,
                                                    int32_t* __restrict__ live, int32_t* __restrict__ n_live0) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e == 0 && n_live0) *n_live0 = (int32_t)n;
    if (e >= n) return;
    const EnvState s = env_reset(p, seed, ids.gid((uint32_t)e), cid);
    env_store(cells, meta, e, s);
    if (live) live[e] = (int32_t)e;
}

__global__ void __launch_bounds__(256) k_envs_fresh(EnvParams p, uint4* __restrict__ cells, uint32_t* __restrict__ meta, int64_t n) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    env_store(cells, meta, e, env_fresh(p));
}

// Env::set_state.  puzzle.rs:107-117 (depth = max_depth, blank = first zero) ; lib.rs:100-112
__global__ void __launch_bounds__(256) k_envs_set_state(EnvParams p, uint4* __restrict__ cells, uint32_t* __restrict__ meta,
                                                        int64_t n, const int64_t* __restrict__ states) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    EnvState s = env_load(cells, meta, e);
    const int64_t* st = states + e * p.N;
    if (p.kind == 0) {
        s.lo = TWR_IDENT_LO; s.hi = TWR_IDENT_HI;
        bool found = false;
        for (int i = 0; i < p.N; ++i) {
            const int64_t v = st[i];
            cell_set(s, i, (uint32_t)v);
            if (v == 0 && !found) { s.blank = (uint32_t)i; found = true; }
        }
        s.depth = (uint32_t)p.max_depth;
    } else {
        for (int i = 0; i < p.N; ++i) {
            const int64_t v = st[i];
            if (v == 1) cell_set(s, 0, (uint32_t)i);
            else if (v == 2) cell_set(s, 1, (uint32_t)i);
            else if (v == 3) cell_set(s, 2, (uint32_t)i);
        }
        s.depth = (uint32_t)p.max_depth;
    }
    env_store(cells, meta, e, s);
}

__global__ void __launch_bounds__(256) k_envs_step(EnvParams p, uint4* __restrict__ cells, uint32_t* __restrict__ meta,
                                                   int64_t n, const int32_t* __restrict__ actions) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    EnvState s = env_load(cells, meta, e);
    env_step(p, s, actions[e]);
    env_store(cells, meta, e, s);
}

__global__ void __launch_bounds__(256) k_envs_query(EnvParams p, const uint4* __restrict__ cells, const uint32_t* __restrict__ meta,
                                                    int64_t n, int64_t* __restrict__ states, int32_t* __restrict__ obs,
                                                    uint8_t* __restrict__ masks, float* __restrict__ reward,
                                                    uint8_t* __restrict__ fin, uint8_t* __restrict__ succ, int32_t* __restrict__ depth) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const EnvState s = env_load(cells, meta, e);
    if (states || obs) {
        for (int i = 0; i < p.N; ++i) {
            const uint32_t v = env_board(p, s, i);
            if (states) states[e * p.N + i] = (int64_t)v;
            if (obs) obs[e * p.N + i] = i * p.N + (int32_t)v;   // puzzle.rs:183-185
        }
    }
    if (masks) {
        const uint32_t m = env_masks(p, s);
        for (int a = 0; a < TWR_MAX_ACTIONS; ++a) masks[e * TWR_MAX_ACTIONS + a] = (m >> a) & 1u;
    }
    if (reward) reward[e] = env_reward(p, s);
    if (fin) fin[e] = env_is_final(p, s) ? 1 : 0;
    if (succ) succ[e] = env_success(p, s) ? 1 : 0;
    if (depth) depth[e] = (int32_t)s.depth;
}

// forward_with_perm's mask step (nn/policy.rs:62) for the parity API
__global__ void __launch_bounds__(256) k_mask_logits(EnvParams p, const uint4* __restrict__ cells, const uint32_t* __restrict__ meta,
                                                     int64_t n, int A, float4* __restrict__ logits) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const uint32_t m = env_masks(p, env_load(cells, meta, e));
    float4 l = logits[e];
    if (A > 0 && !(m & 1u)) l.x = -1e10f;
    if (A > 1 && !(m & 2u)) l.y = -1e10f;
    if (A > 2 && !(m & 4u)) l.z = -1e10f;
    if (A > 3 && !(m & 8u)) l.w = -1e10f;
    logits[e] = l;
}

void launch_envs_reset(cudaStream_t st, const EnvParams& p, uint4* cells, uint32_t* meta, int64_t n, uint64_t seed,
                       EnvIds ids, uint32_t cid, int32_t* live, int32_t* n_live0) {
    if (n <= 0) return;
    k_envs_reset<<<grid_for(n, 256), 256, 0, st>>>(p, cells, meta, n, seed, ids, cid, live, n_live0);
    TWR_COUNT_LAUNCH();
}
void launch_envs_fresh(cudaStream_t st, const EnvParams& p, uint4* cells, uint32_t* meta, int64_t n) {
    if (n <= 0) return;
    k_envs_fresh<<<grid_for(n, 256), 256, 0, st>>>(p, cells, meta, n);
    TWR_COUNT_LAUNCH();
}
void launch_envs_set_state(cudaStream_t st, const EnvParams& p, uint4* cells, uint32_t* meta, int64_t n, const int64_t* d_states) {
    if (n <= 0) return;
    k_envs_set_state<<<grid_for(n, 256), 256, 0, st>>>(p, cells, meta, n, d_states);
    TWR_COUNT_LAUNCH();
}
void launch_envs_step(cudaStream_t st, const EnvParams& p, uint4* cells, uint32_t* meta, int64_t n, const int32_t* d_actions) {
    if (n <= 0) return;
    k_envs_step<<<grid_for(n, 256), 256, 0, st>>>(p, cells, meta, n, d_actions);
    TWR_COUNT_LAUNCH();
}
void launch_envs_query(cudaStream_t st, const EnvParams& p, const uint4* cells, const uint32_t* meta, int64_t n,
                       int64_t* d_states, int32_t* d_obs, uint8_t* d_masks, float* d_reward, uint8_t* d_final,
                       uint8_t* d_success, int32_t* d_depth) {
    if (n <= 0) return;
    k_envs_query<<<grid_for(n, 256), 256, 0, st>>>(p, cells, meta, n, d_states, d_obs, d_masks, d_reward, d_final, d_success, d_depth);
    TWR_COUNT_LAUNCH();
}
void launch_mask_logits(cudaStream_t st, const EnvParams& p, const uint4* cells, const uint32_t* meta, int64_t n, int A, float4* logits) {
    if (n <= 0) return;
    k_mask_logits<<<grid_for(n, 256), 256, 0, st>>>(p, cells, meta, n, A, logits);
    TWR_COUNT_LAUNCH();
}

// ------------------------------------------------------------------------- K3 ---
__global__ void __launch_bounds__(256) k_sample(const float* __restrict__ logits, int64_t n, int A, uint64_t seed,
                                                uint32_t env_id_base, uint32_t step, uint32_t cid,
                                                int32_t* __restrict__ actions, float* __restrict__ uniforms) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[4];
    philox4x32_10(env_id_base + (uint32_t)i, step, TWR_RNG_SAMPLE, cid, (uint32_t)seed, (uint32_t)(seed >> 32), w);
    float l[4] = {0.f, 0.f, 0.f, 0.f}, u[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        u[a] = u32_to_unit_f32(w[a]);
        if (a < A) l[a] = logits[i * A + a];
        if (uniforms && a < A) uniforms[i * A + a] = u[a];
    }
    actions[i] = sample_from_logits4(l, u, A);
}

void launch_sample(cudaStream_t st, const float* d_logits, int64_t n, int A, uint64_t seed, uint32_t env_id_base,
                   uint32_t step, uint32_t cid, int32_t* d_actions, float* d_uniforms) {
    if (n <= 0) return;
    k_sample<<<grid_for(n, 256), 256, 0, st>>>(d_logits, n, A, seed, env_id_base, step, cid, d_actions, d_uniforms);
    TWR_COUNT_LAUNCH();
}

// ---------------------------------------------------- K3 + K4a + K1: collect step ---
// One record of PPOCollector::single_collect's loop (collector/ppo.rs:69-80) for every live env:
// reward(s_t), masked logits, value, Gumbel-max action, twist index -> record [t][env];
// terminal states are recorded and retire (their action is not applied), the rest step and are
// appended to the next live list with one atomicAdd per warp (ballot + popc prefix).
__global__ void __launch_bounds__(256) k_collect_step(StepArgs a, CollectBuffers b, const int32_t* __restrict__ live_cur,
                                                      int32_t* __restrict__ live_next) {
    const int nl = b.n_live[a.t];
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = pos < nl;
    int e = 0, perm = -1;
    float4 raw = make_float4(0.f, 0.f, 0.f, 0.f);
    float value = 0.f;
    if (active) {
        e = live_cur[pos];
        raw = b.logits[pos];
        value = b.values[pos];
        if (a.n_perms > 0) {                                  // get_perm_id, nn/policy.rs:67-77
            uint32_t w[4];
            philox4x32_10(a.ids.gid((uint32_t)e), (uint32_t)a.t, TWR_RNG_PERM, a.cid, (uint32_t)a.seed,
                          (uint32_t)(a.seed >> 32), w);
            perm = (int)mulhi_u32(w[0], (uint32_t)a.n_perms);
        }
    }
    collect_step_body(a, b, active, e, raw, value, perm, live_next);
}

__global__ void __launch_bounds__(256) k_compact_live(const int32_t* __restrict__ live_cur, const int32_t* __restrict__ n_cur,
                                                      const int32_t* __restrict__ ep_len, int32_t* __restrict__ live_next,
                                                      int32_t* __restrict__ n_next) {
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    int e = 0;
    bool survives = false;
    if (pos < *n_cur) { e = live_cur[pos]; survives = ep_len[e] == 0; }
    const unsigned bal = __ballot_sync(0xffffffffu, survives);
    if (bal) {
        const int lane = threadIdx.x & 31;
        int base = 0;
        if (lane == 0) base = atomicAdd(n_next, __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (survives) live_next[base + __popc(bal & ((1u << lane) - 1u))] = e;
    }
}

void launch_compact_live(cudaStream_t st, const int32_t* live_cur, const int32_t* n_cur, const int32_t* ep_len, int64_t max_n,
                         int32_t* live_next, int32_t* n_next) {
    k_compact_live<<<grid_for(max_n, 256), 256, 0, st>>>(live_cur, n_cur, ep_len, live_next, n_next);
    TWR_COUNT_LAUNCH();
}

void launch_collect_step(cudaStream_t st, const StepArgs& a, const CollectBuffers& b, const int32_t* live_cur, int32_t* live_next) {
    k_collect_step<<<grid_for(b.B, 256), 256, 0, st>>>(a, b, live_cur, live_next);
    TWR_COUNT_LAUNCH();
}

// ------------------------------------------------------------------------ K4b ---
// GAE, collector/ppo.rs:82-92, evaluation order as written: ret = r + gamma*(v' + lambda*adv').
// __fmul_rn/__fadd_rn keep nvcc from contracting into FMAs so the result is bit-identical to the
// reference's unfused f32 arithmetic.
__device__ __forceinline__ void gae_step(float r, float v, float v_next, float adv_next, float gamma, float lambda,
                                         float& adv, float& ret) {
    ret = __fadd_rn(r, __fmul_rn(gamma, __fadd_rn(v_next, __fmul_rn(lambda, adv_next))));
    adv = __fsub_rn(ret, v);
}

__global__ void __launch_bounds__(256) k_gae_concat(const float* __restrict__ rw, const float* __restrict__ vl,
                                                    const int64_t* __restrict__ off, int64_t n_ep, float gamma, float lambda,
                                                    float* __restrict__ advs, float* __restrict__ rets) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_ep) return;
    const int64_t lo = off[e], hi = off[e + 1];
    if (hi <= lo) return;
    float adv = __fsub_rn(rw[hi - 1], vl[hi - 1]), ret = rw[hi - 1], v_next = vl[hi - 1];
    advs[hi - 1] = adv; rets[hi - 1] = ret;
    for (int64_t i = hi - 2; i >= lo; --i) {
        const float v = vl[i];
        gae_step(rw[i], v, v_next, adv, gamma, lambda, adv, ret);
        advs[i] = adv; rets[i] = ret;
        v_next = v;
    }
}

void launch_gae_concat(cudaStream_t st, const float* r, const float* v, const int64_t* off, int64_t n_ep, float gamma,
                       float lambda, float* adv, float* ret) {
    if (n_ep <= 0) return;
    k_gae_concat<<<grid_for(n_ep, 256), 256, 0, st>>>(r, v, off, n_ep, gamma, lambda, adv, ret);
    TWR_COUNT_LAUNCH();
}

// ------------------------------------------------------------------------- K5 ---
// Exclusive scan of episode lengths in local order (the env-id rotation of EnvIds already puts the
// LAST episode id at local 0, i.e. local order == the reference's merge order, collector.rs:40-46).
// One CTA of 32 warps; warp w owns a contiguous segment that it walks 32 lengths at a time with coalesced loads
// and a shuffle scan (pass 1: segment totals, pass 2: offsets).  Also scatters ep_len by episode id.
__global__ void __launch_bounds__(1024) k_episode_offsets(CollectBuffers b, EnvIds ids) {
    __shared__ long long seg_total[32];
    const int64_t B = b.B;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t per = ((B + 1023) / 1024) * 32;               // lengths per warp, a multiple of 32
    const int64_t s0 = (int64_t)warp * per, s1 = min(B, s0 + per);
    long long sum = 0;
    for (int64_t s = s0 + lane; s < s1; s += 32) sum += b.ep_len[s];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
    if (lane == 0) seg_total[warp] = sum;
    __syncthreads();
    long long run = 0;
    for (int w = 0; w < warp; ++w) run += seg_total[w];
    for (int64_t c = s0; c < s1; c += 32) {
        const int64_t s = c + lane;
        const int len = s < s1 ? b.ep_len[s] : 0;
        long long inc = len;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long v = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += v;
        }
        if (s < s1) {
            b.ep_off[s] = run + inc - len;
            if (b.ep_len_id) b.ep_len_id[ids.gid((uint32_t)s) - ids.base] = len;
        }
        run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (threadIdx.x == 1023) {
        long long total = 0;
        for (int w = 0; w < 32; ++w) total += seg_total[w];
        b.stats[1] = (unsigned long long)total;
    }
}

void launch_episode_offsets(cudaStream_t st, const CollectBuffers& b, const EnvIds& ids) {
    k_episode_offsets<<<1, 1024, 0, st>>>(b, ids);
    TWR_COUNT_LAUNCH();
}

// Transpose/compaction: tile of 32 episodes x 32 timesteps.  Loads are coalesced along the env
// axis of the time-major records, stores are coalesced along time inside each episode's
// contiguous output range.  The 16-byte state is expanded to the sparse one-hot indices the
// reference returns from Env::observe (obs[i] = i*N + board[i]).
// One block transposes a 32-episode x 32-step tile of EVERY field: all loads of the tile (4 floats, 2 bytes and 2
// 16-byte words per record, 50 B) are issued before the single barrier, so a block keeps ~50 KB in flight instead of
// 4 KB per field phase; then each episode's run of records is written out contiguously.
struct CompactTiles {
    float f[4][32][33];
    uint8_t b[2][32][33];
    uint4 q[2][32][33];
};
// FUSE_GAE (the PPO collect): the block walks its 32 episodes' tiles from the LAST time tile to the first and computes
// advantages and returns on the way (K4b's reverse recursion, one lane of warp 0 per episode, carried across tiles in
// registers) -- the records are read once, and the time-major adv / ret arrays are neither written nor read: 42 B R + 66 B W
// per record instead of 16 + 16 (GAE) + 50 + 66.  Same f32 operations (gae_step) in the same order as k_gae_concat, the
// stand-alone GAE of twr_gae.
template <bool FUSE_GAE>
__global__ void __launch_bounds__(256) k_compact(EnvParams p, CollectBuffers b, int A, float gamma, float lambda) {
    extern __shared__ __align__(16) unsigned char compact_smem[];
    CompactTiles& tl = *reinterpret_cast<CompactTiles*>(compact_smem);
    __shared__ int lens[32];
    __shared__ long long offs[32];
    const int64_t e0 = (int64_t)blockIdx.x * 32;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    if (tid < 32) {
        const int64_t e = e0 + tid;
        lens[tid] = e < b.B ? b.ep_len[e] : 0;
        offs[tid] = e < b.B ? b.ep_off[e] : 0;
    }
    __syncthreads();
    int maxlen = 0;
    for (int i = 0; i < 32; ++i) maxlen = max(maxlen, lens[i]);
    if (maxlen == 0 || (!FUSE_GAE && (int)blockIdx.y * 32 >= maxlen)) return;
    float g_adv = 0.f, g_vnext = 0.f;          // GAE state of episode threadIdx.x (warp 0), carried from tile to tile
    for (int t0 = FUSE_GAE ? ((maxlen - 1) / 32) * 32 : (int)blockIdx.y * 32; t0 >= 0; t0 -= 32) {

    // ---- load phase: row t of the time-major records, 32 consecutive envs per warp (coalesced)
    {
        const int64_t e = e0 + threadIdx.x;
        const int len = lens[threadIdx.x];
        float vf[4][4];
        uint8_t vb[4][2];
        uint4 vq[4][2];
        bool ok[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            const int t = t0 + threadIdx.y + 8 * it;
            ok[it] = e < b.B && t < len;
            if (ok[it]) {
                const int64_t r = (int64_t)t * b.B + e;
                vf[it][0] = b.rec_value[r]; vf[it][1] = b.rec_reward[r];
                if (!FUSE_GAE) { vf[it][2] = b.rec_adv[r]; vf[it][3] = b.rec_ret[r]; }
                vb[it][0] = b.rec_action[r]; vb[it][1] = (uint8_t)b.rec_perm[r];
                vq[it][0] = reinterpret_cast<const uint4*>(b.rec_logits)[r]; vq[it][1] = b.rec_state[r];
            }
        }
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            if (ok[it]) {
                const int ty = threadIdx.y + 8 * it;
#pragma unroll
                for (int k = 0; k < (FUSE_GAE ? 2 : 4); ++k) tl.f[k][ty][threadIdx.x] = vf[it][k];
                tl.b[0][ty][threadIdx.x] = vb[it][0]; tl.b[1][ty][threadIdx.x] = vb[it][1];
                tl.q[0][ty][threadIdx.x] = vq[it][0]; tl.q[1][ty][threadIdx.x] = vq[it][1];
            }
        }
    }
    __syncthreads();
    if (FUSE_GAE) {
        if (threadIdx.y == 0) {                  // collector/ppo.rs:82-92, steps t0+nt-1 .. t0 of episode threadIdx.x
            const int ey = threadIdx.x, len = lens[ey];
            for (int x = min(32, len - t0) - 1; x >= 0; --x) {
                const float v = tl.f[0][x][ey], r = tl.f[1][x][ey];
                float ret;
                if (t0 + x == len - 1) { g_adv = __fsub_rn(r, v); ret = r; }
                else gae_step(r, v, g_vnext, g_adv, gamma, lambda, g_adv, ret);
                tl.f[2][x][ey] = g_adv; tl.f[3][x][ey] = ret;
                g_vnext = v;
            }
        }
        __syncthreads();
    }

    // ---- store phase: warp `ey` walks episodes ey, ey+8, ..; lane = step inside the tile
    for (int ey = threadIdx.y; ey < 32; ey += blockDim.y) {
        const int nt = min(32, lens[ey] - t0);                 // records of this episode in the tile
        if (e0 + ey >= b.B || nt <= 0) continue;
        const long long r0 = offs[ey] + t0;
        const int x = threadIdx.x;
        if (x < nt) {
            b.out_values[r0 + x] = tl.f[0][x][ey]; b.out_rets[r0 + x] = tl.f[3][x][ey];
            if (b.pack_misc) {
                const float rw = tl.f[1][x][ey];
                const uint32_t rcode = rw == 1.0f ? 2u : rw == -0.5f ? 1u : 0u;
                b.out_actions[r0 + x] = (uint8_t)((uint32_t)tl.b[0][x][ey] | (rcode << 2) | ((uint32_t)((int8_t)tl.b[1][x][ey] + 1) << 4));
            } else {
                b.out_rewards[r0 + x] = tl.f[1][x][ey]; b.out_advs[r0 + x] = tl.f[2][x][ey];
                b.out_actions[r0 + x] = tl.b[0][x][ey]; b.out_perms[r0 + x] = (int8_t)tl.b[1][x][ey];
            }
        }
        // logits: float4 per record -> [record][A] floats
        if (A == 4) {
            if (x < nt) reinterpret_cast<uint4*>(b.out_logits)[r0 + x] = tl.q[0][x][ey];
        } else {
            float* dst = b.out_logits + r0 * A;
            for (int j = x; j < nt * A; j += 32) {
                const uint4 q = tl.q[0][j / A][ey];
                const int c = j % A;
                const uint32_t w = c == 0 ? q.x : c == 1 ? q.y : c == 2 ? q.z : q.w;
                dst[j] = __uint_as_float(w);
            }
        }
        // obs: 16-byte state -> N one-hot indices per record (u16, or u8 for twr_host_buffers.obs_u8)
        uint16_t* dst = b.out_obs + r0 * p.N;
        uint8_t* dst8 = reinterpret_cast<uint8_t*>(b.out_obs) + r0 * p.N;
        if (p.kind == 0 && p.N == 16) {
            // 16-cell puzzle: one thread per record, the 16 indices leave as one (u8) or two (u16) 16-byte stores
            if (x < nt) {
                const uint4 q = tl.q[1][x][ey];
                const uint32_t w[4] = {q.x, q.y, q.z, q.w};
                if (b.obs_u8) {
                    uint32_t o[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k)            // cell i = 4k+j holds tile byte j of word k; index = i*16 + tile
                        o[k] = w[k] + (uint32_t)(k * 64) * 0x01010101u + 0x30201000u;
                    reinterpret_cast<uint4*>(dst8)[x] = make_uint4(o[0], o[1], o[2], o[3]);
                } else {
                    uint32_t o[8];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t i0 = (uint32_t)(4 * k) * 16u;
                        o[2 * k] = ((w[k] & 0xFFu) + i0) | ((((w[k] >> 8) & 0xFFu) + i0 + 16u) << 16);
                        o[2 * k + 1] = (((w[k] >> 16) & 0xFFu) + i0 + 32u) | ((((w[k] >> 24) & 0xFFu) + i0 + 48u) << 16);
                    }
                    uint4* d4 = reinterpret_cast<uint4*>(dst) + 2 * x;
                    d4[0] = make_uint4(o[0], o[1], o[2], o[3]);
                    d4[1] = make_uint4(o[4], o[5], o[6], o[7]);
                }
            }
            continue;
        }
        for (int j = x; j < nt * p.N; j += 32) {
            const uint4 q = tl.q[1][j / p.N][ey];
            EnvState s;
            s.lo = (uint64_t)q.x | ((uint64_t)q.y << 32);
            s.hi = (uint64_t)q.z | ((uint64_t)q.w << 32);
            s.blank = 0; s.depth = 0;
            const int i = j % p.N;
            const int idx = i * p.N + (int)env_board(p, s, i);
            if (b.obs_u8) dst8[j] = (uint8_t)idx; else dst[j] = (uint16_t)idx;
        }
    }
    if (!FUSE_GAE) break;
    __syncthreads();                             // the next (earlier) tile's loads overwrite the tiles
    }
}

__global__ void k_publish_stats(const unsigned long long* __restrict__ stats, unsigned long long* __restrict__ mapped_host) {
    if (threadIdx.x < 4) mapped_host[threadIdx.x] = stats[threadIdx.x];
    __threadfence_system();
}
void launch_publish_stats(cudaStream_t st, const unsigned long long* stats, unsigned long long* mapped_host) {
    k_publish_stats<<<1, 32, 0, st>>>(stats, mapped_host);
    TWR_COUNT_LAUNCH();
}

void launch_compact(cudaStream_t st, const EnvParams& p, const CollectBuffers& b, int A) {
    dim3 grid(grid_for(b.B, 32), (unsigned)((b.Tmax + 31) / 32));
    cudaFuncSetAttribute(k_compact<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CompactTiles));   // per device: set on every launch
    k_compact<false><<<grid, dim3(32, 8), sizeof(CompactTiles), st>>>(p, b, A, 0.f, 0.f);
    TWR_COUNT_LAUNCH();
}
// K4b + K5 in one pass (see k_compact<true>)
void launch_compact_gae(cudaStream_t st, const EnvParams& p, const CollectBuffers& b, int A, float gamma, float lambda) {
    cudaFuncSetAttribute(k_compact<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CompactTiles));
    k_compact<true><<<dim3(grid_for(b.B, 32)), dim3(32, 8), sizeof(CompactTiles), st>>>(p, b, A, gamma, lambda);
    TWR_COUNT_LAUNCH();
}

// ------------------------------------------------------------------------- f1 ---
// One iteration of single_solve's loop (rl/solve.rs:30-60) per live env: a final state adds its reward and
// retires; otherwise total += reward(s), probs = masked exp / (sum + 1e-6) (Policy::predict,
// nn/policy.rs:43-47), action = argmax (deterministic) or a draw proportional to probs (nn/policy.rs:153-167),
// then Env::step.
__global__ void __launch_bounds__(256) k_solve_step(SolveArgs a, const int32_t* __restrict__ live_cur, int32_t* __restrict__ live_next) {
    const int nl = a.n_live[a.t];
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    bool survives = false;
    int e = 0;
    if (pos < nl) {
        e = live_cur[pos];
        EnvState s = env_load(a.cells, a.meta, e);
        const float rew = env_reward(a.env, s);
        const float tot = a.total[e] + rew;
        a.total[e] = tot;
        if (env_is_final(a.env, s)) {
            a.success[e] = env_success(a.env, s) ? 1 : 0;
            a.n_steps[e] = a.t;
        } else {
            float pr[4];
            if (a.mcts_probs) {                     // solve.rs:37-48: probs come from predict_probs_mcts on a clone
#pragma unroll
                for (int i = 0; i < 4; ++i) pr[i] = i < a.A ? a.mcts_probs[(int64_t)e * a.A + i] : 0.0f;
            } else {
                const uint32_t m = env_masks(a.env, s);
                const float4 raw = a.logits[pos];
                const float l[4] = {raw.x, raw.y, raw.z, raw.w};
                float sum = 0.0f;
#pragma unroll
                for (int i = 0; i < 4; ++i) { pr[i] = (i < a.A && ((m >> i) & 1u)) ? expf(l[i]) : 0.0f; sum += pr[i]; }
#pragma unroll
                for (int i = 0; i < 4; ++i) pr[i] = pr[i] / (sum + 0.000001f);
            }
            int act = 0;
            if (a.deterministic) {
                float bv = pr[0];
#pragma unroll
                for (int i = 1; i < 4; ++i) if (i < a.A && pr[i] > bv) { bv = pr[i]; act = i; }
            } else {
                float tw = 0.0f;
#pragma unroll
                for (int i = 0; i < 4; ++i) if (i < a.A) tw += pr[i];
                if (tw > 0.0f) {                       // WeightedIndex: first i whose cumulative weight exceeds the draw
                    uint32_t w[4];
                    philox4x32_10(a.ids.gid((uint32_t)e), (uint32_t)a.t, TWR_RNG_SOLVE, a.cid, (uint32_t)a.seed, (uint32_t)(a.seed >> 32), w);
                    const float chosen = u32_to_unit_f32(w[0]) * tw;
                    float cum = 0.0f;
                    int last = 0;
                    bool found = false;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (i < a.A && pr[i] > 0.0f) {
                            cum += pr[i];
                            last = i;
                            if (!found && cum > chosen) { act = i; found = true; }
                        }
                    }
                    if (!found) act = last;
                }
            }
            if (a.act_rec) a.act_rec[(int64_t)a.t * a.B + e] = (uint8_t)act;
            env_step(a.env, s, act);
            env_store(a.cells, a.meta, e, s);
            survives = true;
        }
    }
    const unsigned bal = __ballot_sync(0xffffffffu, survives);
    if (bal) {
        const int lane = threadIdx.x & 31;
        int base = 0;
        if (lane == 0) base = atomicAdd(&a.n_live[a.t + 1], __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (survives) live_next[base + __popc(bal & ((1u << lane) - 1u))] = e;
    }
}

void launch_solve_step(cudaStream_t st, const SolveArgs& a, const int32_t* live_cur, int32_t* live_next) {
    k_solve_step<<<grid_for(a.B, 256), 256, 0, st>>>(a, live_cur, live_next);
    TWR_COUNT_LAUNCH();
}

__global__ void __launch_bounds__(256) k_envs_broadcast(const uint4* __restrict__ sc, const uint32_t* __restrict__ sm,
                                                        uint4* __restrict__ cells, uint32_t* __restrict__ meta, int64_t n) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    cells[e] = sc[0];
    meta[e] = sm[0];
}

void launch_envs_broadcast(cudaStream_t st, const uint4* sc, const uint32_t* sm, uint4* cells, uint32_t* meta, int64_t n) {
    if (n <= 0) return;
    k_envs_broadcast<<<grid_for(n, 256), 256, 0, st>>>(sc, sm, cells, meta, n);
    TWR_COUNT_LAUNCH();
}
