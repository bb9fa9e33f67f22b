// twr_mcts.cu -- K6: batched Monte-Carlo tree search for the AlphaZero collector
// (rust/src/rl/search.rs:20-189, rust/src/rl/tree.rs, rust/src/collector/az.rs:51-109).
//
// One tree per env in a pre-sized node pool (node (e, i) at index e*P + i, root at i = 0;
// P = 1 + A*(n_sims*max(1,max_expand_depth) + 1) nodes is the reference's worst case).  A node stores what the
// reference's MCTSNode stores -- the cloned+stepped env (16-byte cells + meta) and ONE 16-byte record
// {visit_count, value_sum, prior, first_child | n_children | action_taken} -- plus a parent link.  The children of a
// node are contiguous, so the UCB descent reads one 64-byte line per tree level (statistics AND the links of the
// child it moves to), and the descent records its path so that the backup is a set of independent updates instead
// of a parent-pointer walk.  All envs advance in lockstep, one simulation at a time:
//   k_mcts_select : UCB descent to a leaf (search.rs:134-137, ucb :29-39, next :77-91); terminal leaves back up
//                   their reward at once, the others are compacted (warp ballot) into the leaf batch
//   forward       : the SAME policy forward kernel as the PPO path evaluates the whole leaf batch (K2); a twisted policy
//                   takes one forward per twist, each into its own slice of the outputs
//   k_mcts_expand : Policy::full_predict's average of the twist slices (nn/policy.rs:102-126; one slice and no average
//                   without twists), Policy::predict epilogue (masked exp / (sum+1e-6)), expand (search.rs:56-75), child draw
//                   proportional to the priors (next_sample :94-100), backup (search.rs:45-53)
// k_az_finish turns root visit counts into the MCTS policy (search.rs:166-188), draws the action
// (az.rs:72), writes the record and steps the env; k_az_remaining computes az.rs:93's reward-to-go.
// These kernels are latency / L2 bound (pointer chasing, one thread per env); the flop live in K2.
#include "twr_kernels.cuh"

#include <atomic>
#include <cstdio>
#include <cstdlib>
extern std::atomic<long long> g_twr_launches;
#define TWR_COUNT_LAUNCH() g_twr_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

inline unsigned grid_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }

__device__ __forceinline__ EnvState node_state(const MctsPool& m, int64_t g) {
    return env_load(m.cells, m.meta, g);
}

// node record: x = visit_count, y = value_sum (f32 bits), z = prior (f32 bits), w = first_child | n_children << 20 | action << 24
__device__ __forceinline__ uint32_t link_pack(int first, int nch, int action) {
    return ((uint32_t)first & 0xFFFFFu) | ((uint32_t)nch << 20) | (((uint32_t)action & 0xFFu) << 24);
}
__device__ __forceinline__ int link_first(uint32_t w) { return (int)(w & 0xFFFFFu); }
__device__ __forceinline__ int link_nch(uint32_t w) { return (int)((w >> 20) & 0xFu); }
__device__ __forceinline__ int link_action(uint32_t w) { return (int)(w >> 24); }

// one node of MCTSTree::backpropagate (search.rs:45-53): value_sum += v, visit_count += 1
__device__ __forceinline__ void bump(const MctsPool& m, int64_t g, float v) {
    uint2* q = reinterpret_cast<uint2*>(m.node + g);
    uint2 r = *q;
    r.x += 1u;
    r.y = __float_as_uint(__uint_as_float(r.y) + v);
    *q = r;
}
// MCTSTree::backpropagate over the recorded path (root .. node); falls back to the parent walk when the path
// outgrew its buffer
__device__ __forceinline__ void backprop(const MctsPool& m, int e, int64_t base, int node, int len, float v) {
    if (len < 0) {
        for (int b = node; b >= 0; b = m.parent[base + b]) bump(m, base + b, v);
        return;
    }
    // the nodes of a path are distinct: all loads of a block of 8 are issued before the first store
    for (int k0 = 0; k0 < len; k0 += 8) {
        int idx[8];
        uint2 r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) idx[j] = k0 + j < len ? m.path[(int64_t)(k0 + j) * m.B + e] : -1;
#pragma unroll
        for (int j = 0; j < 8; ++j) if (idx[j] >= 0) r[j] = *reinterpret_cast<const uint2*>(m.node + base + idx[j]);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (idx[j] >= 0) {
                r[j].x += 1u;
                r[j].y = __float_as_uint(__uint_as_float(r[j].y) + v);
                *reinterpret_cast<uint2*>(m.node + base + idx[j]) = r[j];
            }
        }
    }
}

// the same with the lanes of a warp taking one path node each (the nodes of a path are distinct); every lane of the warp
// calls it with the same arguments
__device__ __forceinline__ void backprop_warp(const MctsPool& m, int e, int64_t base, int node, int len, float v, int lane) {
    if (len < 0) {
        if (lane == 0) for (int b = node; b >= 0; b = m.parent[base + b]) bump(m, base + b, v);
        return;
    }
    for (int k = lane; k < len; k += 32) bump(m, base + m.path[(int64_t)k * m.B + e], v);
}

// Policy::predict's epilogue (nn/policy.rs:43-47) on raw logits
__device__ __forceinline__ void masked_probs(const float4 raw, uint32_t mask, int A, float pr[4]) {
    const float l[4] = {raw.x, raw.y, raw.z, raw.w};
    float sum = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; ++i) { pr[i] = (i < A && ((mask >> i) & 1u)) ? expf(l[i]) : 0.0f; sum += pr[i]; }
#pragma unroll
    for (int i = 0; i < 4; ++i) pr[i] = pr[i] / (sum + 0.000001f);
}

// one term of Policy::full_predict's average (nn/policy.rs:109-115): acc += raw / n_perms per logit and for the value,
// each term divided before it is added; called for twists 0, 1, .. in that order
__device__ __forceinline__ void twist_accumulate(float4& acc, float& vacc, const float4 raw, float v, float np) {
    acc.x = __fadd_rn(acc.x, __fdiv_rn(raw.x, np)); acc.y = __fadd_rn(acc.y, __fdiv_rn(raw.y, np));
    acc.z = __fadd_rn(acc.z, __fdiv_rn(raw.z, np)); acc.w = __fadd_rn(acc.w, __fdiv_rn(raw.w, np));
    vacc = __fadd_rn(vacc, __fdiv_rn(v, np));
}

// raw logits and value of the leaf at forward-batch position pos: Policy::predict's without twists, full_predict's
// average over the a.n_perms forward slices with them
__device__ __forceinline__ float4 leaf_eval(const MctsArgs& a, int64_t pos, float& v) {
    if (a.n_perms == 0) { v = a.values[pos]; return a.logits[pos]; }
    const float np = (float)a.n_perms;
    float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    v = 0.0f;
    for (int pi = 0; pi < a.n_perms; ++pi) twist_accumulate(acc, v, a.logits[pi * a.twist_stride + pos], a.values[pi * a.twist_stride + pos], np);
    return acc;
}

// MCTSTree::expand (search.rs:56-75): one child per action with prior > 0, in action order.  Returns the first
// child index and fills cp[] with the children's priors (cnt entries).
__device__ __forceinline__ int expand(const MctsPool& m, const EnvParams& env, int e, int64_t base, int node, const float pr[4],
                                      float cp[4], int& cnt) {
    const EnvState s = node_state(m, base + node);
    int n = m.n_nodes[e];
    const int first = n;
    cnt = 0;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        cp[a] = 0.0f;
        if (a < m.A && pr[a] > 0.0f && n < m.P) {
            EnvState c = s;
            env_step(env, c, a);
            env_store(m.cells, m.meta, base + n, c);
            m.parent[base + n] = node;
            m.node[base + n] = make_uint4(0u, __float_as_uint(0.0f), __float_as_uint(pr[a]), link_pack(0, 0, a));
            // cp[] is indexed by child order; cnt <= a, so this never overwrites an entry still to be read
            if (cnt == 0) cp[0] = pr[a]; else if (cnt == 1) cp[1] = pr[a]; else if (cnt == 2) cp[2] = pr[a]; else cp[3] = pr[a];
            ++n; ++cnt;
        }
    }
    uint32_t* link = &m.node[base + node].w;
    *link = link_pack(first, cnt, link_action(*link));
    m.n_nodes[e] = n;
    return first;
}

// rand's WeightedIndex as used by nn/policy.rs:153-167
__device__ __forceinline__ int weighted_index(const float* w, int n, float u) {
    float tw = 0.0f;
    for (int i = 0; i < n; ++i) tw += w[i];
    if (!(tw > 0.0f)) return 0;
    const float chosen = u * tw;
    float cum = 0.0f;
    int last = 0;
    for (int i = 0; i < n; ++i) {
        if (w[i] > 0.0f) {
            cum += w[i]; last = i;
            if (cum > chosen) return i;
        }
    }
    return last;
}

// warp-aggregated append of (global node index, env) to the leaf batch
__device__ __forceinline__ void push_leaf(const MctsArgs& a, bool want, int64_t gnode, int e, int32_t* counter) {
    const unsigned bal = __ballot_sync(0xffffffffu, want);
    if (!bal) return;
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(counter, __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (want) {
        const int slot = base + __popc(bal & ((1u << lane) - 1u));
        a.fwd_list[slot] = (int32_t)gnode;
        a.fwd_env[slot] = e;
        a.leaf_pos[e] = slot;
    }
}

__global__ void __launch_bounds__(128) k_mcts_begin(MctsArgs a, const int32_t* __restrict__ live, const int32_t* __restrict__ n_live) {
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    const int nl = *n_live;
    if (pos == 0) { a.fwd_count[0] = nl; a.fwd_count[1] = 0; }
    if (pos >= nl) return;
    const int e = live[pos];
    const MctsPool& m = a.pool;
    const int64_t base = (int64_t)e * m.P;
    m.cells[base] = a.env_cells[e]; m.meta[base] = a.env_meta[e];
    m.parent[base] = -1;
    m.node[base] = make_uint4(1u, __float_as_uint(0.0f), __float_as_uint(0.0f), link_pack(0, 0, 0xFF));   // search.rs:119-125: root visit_count = 1
    m.n_nodes[e] = 1;
    m.path[e] = 0; m.path_len[e] = 1;                                          // path[0][e] = root
    a.fwd_list[pos] = (int32_t)base;
    a.fwd_env[pos] = e;
}

// mode 0: root expansion (search.rs:112-128); mode 1: simulation expansion round d (search.rs:142-160)
__device__ __forceinline__ void expand_body(const MctsArgs& a, int e, int pos, int mode, int sim, int d) {
    const MctsPool& m = a.pool;
    const int64_t base = (int64_t)e * m.P;
    const int node = mode == 0 ? 0 : a.cur_node[e];
    const EnvState s = node_state(m, base + node);
    float pr[4], v;
    masked_probs(leaf_eval(a, pos, v), env_masks(a.env, s), m.A, pr);
    float cp[4];
    int nch;
    const int first = expand(m, a.env, e, base, node, pr, cp, nch);
    if (mode == 0) return;
    // next_sample (search.rs:94-100): child drawn proportionally to the priors
    uint32_t w[4];
    const int med = a.max_expand_depth > 1 ? a.max_expand_depth : 1;
    philox4x32_10(a.ids.gid((uint32_t)e), (uint32_t)((a.t * (a.n_sims + 1) + sim) * med + d), TWR_RNG_MCTS, a.cid,
                  (uint32_t)a.seed, (uint32_t)(a.seed >> 32), w);
    const int child = nch > 0 ? first + weighted_index(cp, nch, u32_to_unit_f32(w[0])) : node;
    if (a.trace) a.trace[((int64_t)sim * m.B + e) * 2 + 1] = child;
    int len = m.path_len[e];
    if (child != node && len >= 0) {                     // the drawn child joins the recorded path
        if (len < TWR_MCTS_PATH) { m.path[(int64_t)len * m.B + e] = child; ++len; } else len = -1;
        m.path_len[e] = len;
    }
    if (d + 1 >= a.max_expand_depth) {
        backprop(m, e, base, child, len, v);
        a.active[e] = 0;
    } else {
        a.cur_node[e] = child;
        a.cur_value[e] = v;
    }
}
__global__ void __launch_bounds__(128) k_mcts_expand(MctsArgs a, int mode, int sim, int d, int which) {
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= a.fwd_count[which]) return;
    expand_body(a, a.fwd_env[pos], pos, mode, sim, d);
}

// descent + first rollout round (search.rs:132-146) of one env; returns whether its leaf needs a policy evaluation
__device__ __forceinline__ bool select_body(const MctsArgs& a, int e, int64_t& gnode, int sim) {
    bool want = false;
    {
        const MctsPool& m = a.pool;
        const int64_t base = (int64_t)e * m.P;
        int node = 0, len = 1;
        uint4 cur = m.node[base];                                              // root record (its path entry is permanent)
        while (link_nch(cur.w) > 0) {                                          // next(): argmax UCB, strict '>'
            const int first = link_first(cur.w), nch = link_nch(cur.w);
            const float sq = sqrtf((float)cur.x);
            uint4 ch[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) if (k < nch) ch[k] = m.node[base + first + k];   // one 64-byte line
            int best = -1;
            float best_ucb = -INFINITY;
            uint4 best_rec = cur;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (k < nch) {
                    const uint32_t n = ch[k].x;
                    const float q = n == 0u ? 0.0f : __fdiv_rn(__uint_as_float(ch[k].y), (float)n);
                    const float ucb = __fadd_rn(q, __fmul_rn(__fmul_rn(a.C, __fdiv_rn(sq, __fadd_rn((float)n, 1.0f))), __uint_as_float(ch[k].z)));
                    if (ucb > best_ucb) { best = first + k; best_ucb = ucb; best_rec = ch[k]; }
                }
            }
            if (best < 0) break;
            node = best; cur = best_rec;
            if (len >= 0) {
                if (len < TWR_MCTS_PATH) { m.path[(int64_t)len * m.B + e] = node; ++len; } else len = -1;
            }
        }
        m.path_len[e] = len;
        a.cur_node[e] = node;
        if (a.trace && sim < a.n_sims) { a.trace[((int64_t)sim * m.B + e) * 2] = node; a.trace[((int64_t)sim * m.B + e) * 2 + 1] = node; }
        if (a.max_expand_depth <= 0) {
            backprop(m, e, base, node, len, 0.0f);                             // the rollout loop never runs: value stays 0
            a.active[e] = 0;
        } else {
            const EnvState s = node_state(m, base + node);
            if (env_is_final(a.env, s) || m.n_nodes[e] + m.A > m.P) {
                backprop(m, e, base, node, len, env_reward(a.env, s));
                a.active[e] = 0;
            } else {
                a.active[e] = 1;
                want = true;
                gnode = base + node;
            }
        }
    }
    return want;
}
__global__ void __launch_bounds__(128) k_mcts_select(MctsArgs a, const int32_t* __restrict__ live, const int32_t* __restrict__ n_live,
                                                     int sim, int which) {
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos == 0) a.fwd_count[which ^ 1] = 0;          // the other counter is idle until the next round
    const bool valid = pos < *n_live;
    bool want = false;
    int e = 0;
    int64_t gnode = 0;
    if (valid) {
        e = live[pos];
        want = select_body(a, e, gnode, sim);
    }
    push_leaf(a, want, gnode, e, a.fwd_count + which);
}
// max_expand_depth == 1: expansion + backup of simulation `sim` and the descent of simulation sim+1 in one launch
// (one thread per live env; the leaf batch of sim was compacted into counter `which`, the next goes into which^1)
__global__ void __launch_bounds__(128) k_mcts_expand_select(MctsArgs a, const int32_t* __restrict__ live,
                                                            const int32_t* __restrict__ n_live, int sim, int which) {
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos == 0) a.fwd_count[which] = 0;              // consumed by the forward before this launch; the next launch fills it
    const bool valid = pos < *n_live;
    bool want = false;
    int e = 0;
    int64_t gnode = 0;
    if (valid) {
        e = live[pos];
        if (a.active[e]) expand_body(a, e, a.leaf_pos[e], 1, sim, 0);
        want = select_body(a, e, gnode, sim + 1);
    }
    push_leaf(a, want, gnode, e, a.fwd_count + (which ^ 1));
}

// rollout rounds d > 0 (search.rs:142-146 for the child sampled in the previous round)
__global__ void __launch_bounds__(128) k_mcts_pre(MctsArgs a, const int32_t* __restrict__ live, const int32_t* __restrict__ n_live, int which) {
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos == 0) a.fwd_count[which ^ 1] = 0;
    const bool valid = pos < *n_live;
    bool want = false;
    int e = 0;
    int64_t gnode = 0;
    if (valid) {
        e = live[pos];
        if (a.active[e]) {
            const MctsPool& m = a.pool;
            const int64_t base = (int64_t)e * m.P;
            const int node = a.cur_node[e];
            const EnvState s = node_state(m, base + node);
            if (env_is_final(a.env, s) || m.n_nodes[e] + m.A > m.P) {
                backprop(m, e, base, node, m.path_len[e], env_reward(a.env, s));
                a.active[e] = 0;
            } else {
                want = true;
                gnode = base + node;
            }
        }
    }
    push_leaf(a, want, gnode, e, a.fwd_count + which);
}

// root visit counts -> MCTS policy (search.rs:166-188); used by the debug entry point
__device__ __forceinline__ void root_probs(const MctsPool& m, int64_t base, float pr[4], int32_t vis[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { pr[i] = 0.0f; vis[i] = 0; }
    const uint32_t link = m.node[base].w;
    const int first = link_first(link), nch = link_nch(link);
    for (int k = 0; k < nch; ++k) {
        const uint4 rec = m.node[base + first + k];
        const int act = link_action(rec.w);
        const uint32_t n = rec.x;
        const float f = (float)n;
        if (act == 0) { pr[0] = f; vis[0] = (int32_t)n; } else if (act == 1) { pr[1] = f; vis[1] = (int32_t)n; }
        else if (act == 2) { pr[2] = f; vis[2] = (int32_t)n; } else { pr[3] = f; vis[3] = (int32_t)n; }
    }
    float sum = 0.0f;
    for (int i = 0; i < m.A; ++i) sum += pr[i];
    if (sum > 0.0f) { for (int i = 0; i < 4; ++i) pr[i] = i < m.A ? __fdiv_rn(pr[i], sum) : 0.0f; }
    else { for (int i = 0; i < 4; ++i) pr[i] = i < m.A ? __fdiv_rn(1.0f, (float)m.A) : 0.0f; }
}

__global__ void __launch_bounds__(128) k_mcts_read(MctsArgs a, int64_t n, float* __restrict__ probs, int32_t* __restrict__ visits) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float pr[4]; int32_t vis[4];
    root_probs(a.pool, e * a.pool.P, pr, vis);
    for (int i = 0; i < a.pool.A; ++i) { probs[e * a.pool.A + i] = pr[i]; visits[e * a.pool.A + i] = vis[i]; }
}

// Policy::full_predict (nn/policy.rs:102-126) of env e from the forward slices at position e: what expand_body
// computes for a leaf (parity API)
__global__ void __launch_bounds__(128) k_full_predict(MctsArgs a, const uint4* __restrict__ cells, const uint32_t* __restrict__ meta,
                                                      int64_t n, float* __restrict__ probs, float* __restrict__ values) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float pr[4], v;
    masked_probs(leaf_eval(a, e, v), env_masks(a.env, env_load(cells, meta, e)), a.pool.A, pr);
    for (int i = 0; i < a.pool.A; ++i) probs[e * a.pool.A + i] = pr[i];
    values[e] = v;
}

// one AZCollector loop iteration (az.rs:66-88) for every live env
__global__ void __launch_bounds__(128) k_az_finish(MctsArgs a, CollectBuffers b, const int32_t* __restrict__ live,
                                                   int32_t* __restrict__ live_next) {
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    const int nl = b.n_live[a.t];
    bool survives = false;
    int e = 0;
    if (pos < nl) {
        e = live[pos];
        float pr[4]; int32_t vis[4];
        root_probs(a.pool, (int64_t)e * a.pool.P, pr, vis);
        uint32_t w[4];
        philox4x32_10(a.ids.gid((uint32_t)e), (uint32_t)a.t, TWR_RNG_AZ_ACT, a.cid, (uint32_t)a.seed, (uint32_t)(a.seed >> 32), w);
        const int act = weighted_index(pr, a.pool.A, u32_to_unit_f32(w[0]));       // sample(&mcts_probs), az.rs:72
        EnvState s = env_load(b.cells, b.meta, e);
        const float rew = env_reward(a.env, s);
        const int64_t r = (int64_t)a.t * b.B + e;
        b.rec_state[r] = env_pack_cells(s);
        b.rec_logits[r] = make_float4(pr[0], pr[1], pr[2], pr[3]);               // CollectedData.logits holds the MCTS probs
        b.rec_reward[r] = rew;
        b.rec_action[r] = (uint8_t)act;
        b.rec_perm[r] = (int8_t)-1;
        b.rec_value[r] = 0.0f; b.rec_adv[r] = 0.0f;
        if (env_is_final(a.env, s)) {
            b.ep_len[e] = a.t + 1;
            if (env_success(a.env, s)) atomicAdd(&b.stats[0], 1ull);
            atomicAdd(reinterpret_cast<double*>(&b.stats[2]), (double)rew);
        } else {
            env_step(a.env, s, act);
            env_store(b.cells, b.meta, e, s);
            survives = true;
        }
    }
    const unsigned bal = __ballot_sync(0xffffffffu, survives);
    if (bal) {
        const int lane = threadIdx.x & 31;
        int base = 0;
        if (lane == 0) base = atomicAdd(&b.n_live[a.t + 1], __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (survives) live_next[base + __popc(bal & ((1u << lane) - 1u))] = e;
    }
}

// remaining_values[t] = total - sum_{k<t} r_k, f32 in the reference's order (az.rs:74-76,93)
__global__ void __launch_bounds__(256) k_az_remaining(CollectBuffers b) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.B) return;
    const int n = b.ep_len[e];
    float total = 0.0f;
    for (int t = 0; t < n; ++t) total = __fadd_rn(total, b.rec_reward[(int64_t)t * b.B + e]);
    float prefix = 0.0f;
    for (int t = 0; t < n; ++t) {
        const int64_t r = (int64_t)t * b.B + e;
        b.rec_ret[r] = __fsub_rn(total, prefix);
        prefix = __fadd_rn(prefix, b.rec_reward[r]);
    }
}


// ------------------------------------------------------------------------------------------------------------------
// Persistent whole-search kernel for SMALL batches (the reference's AlphaZero default is 512 episodes x 1000 simulations,
// src/twisterl/defaults.py:82-90).  The lockstep path above costs two dependent launches per simulation, and its forward
// keeps 2-4 SMs busy on a 512-leaf batch: ~30 us per simulation, below the host.  Here ONE launch runs all simulations of
// a search: a cluster of PM_CS CTAs owns up to PM_TPC trees and holds the policy STATIONARY in shared memory (fp32, the
// reference's arithmetic), split along the embedding features: CTA r keeps features [r*EC, (r+1)*EC) of the embedding table
// and the matching ROWS of the common Linear.  A simulation is four short phases separated by cluster barriers, with no
// launch, no global operand traffic and no inter-cluster dependency:
//   A  owner WARP of each tree (tree j -> warp j / PM_CS of CTA j % PM_CS): UCB descent, one lane per child (the
//      divisions of the UCB expression cost as much as the L2 round trip of a level when one thread does all four);
//      the leaf's 16-byte state goes to every CTA (DSMEM)
//   B  every CTA: its EC features of h1 = relu(bias + sum of table rows) for every leaf (local), then its K-slice of
//      W1.h1 for ALL H columns (the weights of a column cached in registers), sent to the CTA that OWNS the leaf's tree
//      (distributed shared memory moves 17-21 B/clk: the partial sums are half the bytes an all-gather of h1 would be)
//   C  owner CTA, local: h2 = relu(sum of the PM_CS partial sums + b1) and the five head dot products of its trees
//   D  owner warp: Policy::predict's epilogue, expand, child draw (lane 0) and the backup, one lane per path node,
//      exactly as expand_body does
// -- two cluster barriers per simulation (after A and after B).
// Trees stay in the global node pool (L2-resident: 512 trees x 160 KB), touched by one thread each.
constexpr int PM_CS = 8;
constexpr int PM_THREADS = 256;
constexpr int PM_TPC = 40;
constexpr int PM_MAX_EC = 64;        // E <= 512

struct PmLayout { int E, H, EC, obs; size_t w1s, tab, h1s, b1s, embb, headw, part2, hbuf, red, cells, flag, total; };
__host__ __device__ inline PmLayout pm_layout(int E, int H, int obs) {
    PmLayout l;
    l.E = E; l.H = H; l.obs = obs; l.EC = E / PM_CS;
    size_t o = 0;
    l.w1s = o; o += sizeof(float) * (size_t)l.EC * H;                    // W1 rows [r*EC, (r+1)*EC) x all H columns
    l.tab = o; o += sizeof(float) * (size_t)obs * l.EC;                  // table features [r*EC, (r+1)*EC)
    l.h1s = o; o += sizeof(float) * (size_t)PM_TPC * l.EC;               // this CTA's h1 slice of every leaf
    l.b1s = o; o += sizeof(float) * (size_t)H;
    l.embb = o; o += sizeof(float) * (size_t)l.EC;
    l.headw = o; o += sizeof(float) * (size_t)5 * (H + 8);                   // [output][column], rows padded by 8 floats
    l.part2 = o; o += sizeof(float) * (size_t)(PM_TPC / PM_CS) * PM_CS * H;   // partial h2 of MY trees (all H columns) from every rank
    l.hbuf = o; o += sizeof(float) * (size_t)(PM_TPC / PM_CS) * H;            // h2 of my trees
    l.red = o; o += sizeof(float) * (size_t)(PM_TPC / PM_CS) * 8;             // logits / value of my trees
    l.cells = o; o += sizeof(uint4) * (size_t)PM_TPC;
    l.flag = o; o += sizeof(int) * (size_t)PM_TPC;
    l.total = (o + 15) & ~(size_t)15;
    return l;
}

__device__ __forceinline__ uint32_t pm_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t pm_cluster_id() { uint32_t r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t pm_nclusters() { uint32_t r; asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ void pm_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// generic address of `p` (a shared-memory address of this CTA) inside CTA `rank` of the cluster
template <typename T>
__device__ __forceinline__ T* pm_remote(T* p, uint32_t rank) {
    uint64_t out;
    asm volatile("mapa.u64 %0, %1, %2;" : "=l"(out) : "l"(reinterpret_cast<uint64_t>(p)), "r"(rank));
    return reinterpret_cast<T*>(out);
}

// TW: a twisted policy (Policy::full_predict at every leaf).  A leaf slot is then a (tree, twist) pair: the PM_TPC slots hold
// PM_CS * (PM_TPC / PM_CS / T) trees of T slots each.  Slot g belongs to owner CTA g % PM_CS and is that CTA's local slot
// l = g / PM_CS; local slots l = w*T .. w*T + T-1 are the twists of the tree owned by warp w, so the T evaluations of a tree
// meet in its owner CTA (phase C) and are averaged by its owner warp (phase D).  Phase A stays per tree.  The twist tables
// are read through the read-only data path: GridWorld 5x5's table already fills shared memory (pm_layout).
template <bool TW>
__global__ void __launch_bounds__(PM_THREADS, 1)
k_mcts_persistent(MctsArgs a, PolicyDev p, const int32_t* __restrict__ live, const int32_t* __restrict__ n_live, int pos0, int cap) {
    extern __shared__ __align__(16) unsigned char pm_smem[];
    const PmLayout L = pm_layout(p.E, p.H, p.obs_size);
    float* w1s = reinterpret_cast<float*>(pm_smem + L.w1s);
    float* tab = reinterpret_cast<float*>(pm_smem + L.tab);
    float* h1s = reinterpret_cast<float*>(pm_smem + L.h1s);
    float* b1s = reinterpret_cast<float*>(pm_smem + L.b1s);
    float* embb = reinterpret_cast<float*>(pm_smem + L.embb);
    float* headw = reinterpret_cast<float*>(pm_smem + L.headw);
    float* part2 = reinterpret_cast<float*>(pm_smem + L.part2);
    float* red = reinterpret_cast<float*>(pm_smem + L.red);
    float* hbuf = reinterpret_cast<float*>(pm_smem + L.hbuf);
    uint4* leaf_cells = reinterpret_cast<uint4*>(pm_smem + L.cells);
    int* leaf_flag = reinterpret_cast<int*>(pm_smem + L.flag);
    const int tid = threadIdx.x;
    const uint32_t rank = pm_rank();
    const int E = L.E, H = L.H, EC = L.EC;
    const MctsPool& m = a.pool;

    // ---- stationary operands (fp32): this CTA's feature slice of the table and the matching rows of W1
    for (int i = tid; i < EC * H; i += PM_THREADS) w1s[i] = p.w1[(size_t)rank * EC * H + i];
    for (int i = tid; i < p.obs_size * EC; i += PM_THREADS) { const int r = i / EC, f = i % EC; tab[i] = p.emb[(size_t)r * E + rank * EC + f]; }
    for (int i = tid; i < H; i += PM_THREADS) {
        b1s[i] = p.b1[i];
        for (int o = 0; o < 4; ++o) headw[o * (H + 8) + i] = o < p.A ? p.wa[(size_t)i * p.A + o] : 0.0f;
        headw[4 * (H + 8) + i] = p.wv[i];
    }
    for (int i = tid; i < EC; i += PM_THREADS) embb[i] = p.emb_b[rank * EC + i];
    __syncthreads();
    // the W1 column of this thread, its EC rows cached in registers for the whole search (phase B)
    const int col = tid % H, lg = tid / H, nlg = PM_THREADS / H;          // H = 256: one leaf group; H = 128: two
    float wreg[PM_MAX_EC];
#pragma unroll
    for (int k = 0; k < PM_MAX_EC; ++k) wreg[k] = k < EC ? w1s[k * H + col] : 0.0f;

    // ---- trees of this launch: live positions [pos0, pos0 + cap) (a batch larger than the resident clusters can hold is cut
    // into several launches; trees are independent); tree j of the cluster is owned by thread j / PM_CS of CTA j % PM_CS
    const int n = max(0, min(*n_live - pos0, cap));
    const int ncl = (int)pm_nclusters();
    const int per = (n + ncl - 1) / ncl;
    const int first = pos0 + (int)pm_cluster_id() * per;
    const int nt = max(0, min(per, pos0 + n - first));     // host guarantees per <= PM_CS * (PM_TPC / PM_CS / T)
    const int T = TW ? p.n_perms : 1;                      // leaf slots per tree
    // leaf slots in use: g < ns (untwisted: slot g is tree g)
    const int ns = TW ? PM_CS * ((nt + PM_CS - 1) / PM_CS) * T : nt;
    auto slot_tree = [&](int g, int& pi) -> int {          // the tree of slot g (-1: none) and its twist
        if (!TW) { pi = -1; return g; }
        const int l = g / PM_CS, j = (l / T) * PM_CS + g % PM_CS;
        pi = l % T;
        return j < nt ? j : -1;
    };
    const int warp = tid >> 5, lane = tid & 31;
    const int j_own = warp * PM_CS + (int)rank;            // the tree this WARP owns (local slots warp*T .. warp*T + T-1 of this CTA)
    const bool owner = warp < PM_TPC / PM_CS / T && j_own < nt;    // warp-uniform
    int e = 0, node = 0, len = 1;
    int64_t base = 0;
    bool need = false;
    if (owner) { e = live[first + j_own]; base = (int64_t)e * m.P; }
    const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
    pm_cluster_sync();

    const bool prof = a.dbg != nullptr && blockIdx.x == 0 && tid == 0;   // warp 0 / lane 0: an owner warp's view of every phase
    long long tA = 0, tS1 = 0, tB = 0, tS2 = 0, tC = 0, tD = 0, t0 = 0;
    for (int sim = -1; sim < a.n_sims; ++sim) {
        if (prof) t0 = clock64();
        // ================= A: descent (owner warps; lane k evaluates child k) =================
        if (owner) {
            need = false;
            if (sim < 0) {                                  // k_mcts_begin: the root (search.rs:112-128), always evaluated
                if (lane == 0) {
                    m.cells[base] = a.env_cells[e]; m.meta[base] = a.env_meta[e];
                    m.parent[base] = -1;
                    m.node[base] = make_uint4(1u, __float_as_uint(0.0f), __float_as_uint(0.0f), link_pack(0, 0, 0xFF));
                    m.n_nodes[e] = 1;
                    m.path[e] = 0; m.path_len[e] = 1;
                }
                node = 0; len = 1; need = true;
            } else {                                        // select_body: next() = argmax UCB, strict '>', first child wins a tie
                node = 0; len = 1;
                uint4 cur = m.node[base];                   // every lane reads the root record (one broadcast load)
                while (link_nch(cur.w) > 0) {
                    const int fc = link_first(cur.w), nch = link_nch(cur.w);
                    const float sq = sqrtf((float)cur.x);
                    uint4 ch = cur;
                    float ucb = -INFINITY;
                    if (lane < nch) {
                        ch = m.node[base + fc + lane];
                        const uint32_t nv = ch.x;
                        const float q = nv == 0u ? 0.0f : __fdiv_rn(__uint_as_float(ch.y), (float)nv);
                        ucb = __fadd_rn(q, __fmul_rn(__fmul_rn(a.C, __fdiv_rn(sq, __fadd_rn((float)nv, 1.0f))), __uint_as_float(ch.z)));
                        if (!(ucb > -INFINITY)) ucb = -INFINITY;           // NaN / -inf never wins (search.rs:85: `>` is false)
                    }
                    int bk = lane < nch ? lane : 99;
                    float bu = ucb;
#pragma unroll
                    for (int d = 1; d < 4; d <<= 1) {       // max over lanes 0..3, smallest index on equal values
                        const float ou = __shfl_xor_sync(0xffffffffu, bu, d);
                        const int ok = __shfl_xor_sync(0xffffffffu, bk, d);
                        if (ou > bu || (ou == bu && ok < bk)) { bu = ou; bk = ok; }
                    }
                    bk = __shfl_sync(0xffffffffu, bk, 0);
                    bu = __shfl_sync(0xffffffffu, bu, 0);
                    if (bk >= nch || !(bu > -INFINITY)) break;             // no child with a comparable UCB: stay (search.rs:89)
                    cur.x = __shfl_sync(0xffffffffu, ch.x, bk); cur.y = __shfl_sync(0xffffffffu, ch.y, bk);
                    cur.z = __shfl_sync(0xffffffffu, ch.z, bk); cur.w = __shfl_sync(0xffffffffu, ch.w, bk);
                    node = fc + bk;
                    if (len >= 0) {
                        if (len < TWR_MCTS_PATH) { if (lane == 0) m.path[(int64_t)len * m.B + e] = node; ++len; } else len = -1;
                    }
                }
                if (a.trace && lane == 0) { a.trace[((int64_t)sim * m.B + e) * 2] = node; a.trace[((int64_t)sim * m.B + e) * 2 + 1] = node; }
                const EnvState s = node_state(m, base + node);
                __syncwarp();                               // lane 0's path stores are read by the other lanes in the backup
                if (env_is_final(a.env, s) || m.n_nodes[e] + m.A > m.P) backprop_warp(m, e, base, node, len, env_reward(a.env, s), lane);
                else need = true;
            }
            if (lane < PM_CS) {                             // the leaf's state to every CTA of the cluster: lane r -> CTA r
                const uint4 cells = need ? m.cells[base + node] : make_uint4(0, 0, 0, 0);
                *pm_remote(leaf_cells + j_own, (uint32_t)lane) = cells;
                *pm_remote(leaf_flag + j_own, (uint32_t)lane) = need ? 1 : 0;
            }
        }
        if (prof) { const long long t = clock64(); tA += t - t0; t0 = t; }
        pm_cluster_sync();
        if (prof) { const long long t = clock64(); tS1 += t - t0; t0 = t; }
        // ================= B: embedding slice (local), then this K-slice of W1.h1 for every column =================
        for (int idx = tid; idx < ns * (EC / 4); idx += PM_THREADS) {
            const int g = idx / (EC / 4), f4 = (idx % (EC / 4)) * 4;
            int pi;
            const int j = slot_tree(g, pi);
            if ((TW && j < 0) || !leaf_flag[j]) continue;
            const uint4 c = leaf_cells[j];
            EnvState s; s.blank = 0; s.depth = 0;
            s.lo = (uint64_t)c.x | ((uint64_t)c.y << 32); s.hi = (uint64_t)c.z | ((uint64_t)c.w << 32);
            float4 acc = *reinterpret_cast<const float4*>(embb + f4);                       // bias first, then the rows in
            for (int i = 0; i < a.env.N; ++i) {                                              // observation order (layers.rs:58-62)
                int r = i * a.env.N + (int)env_board(a.env, s, i);
                if (TW) r = __ldg(p.obs_perms + (size_t)pi * p.obs_size + r);               // twist-in, policy.rs:81-83
                const float4 t4 = *reinterpret_cast<const float4*>(tab + (size_t)r * EC + f4);
                acc.x = __fadd_rn(acc.x, t4.x); acc.y = __fadd_rn(acc.y, t4.y); acc.z = __fadd_rn(acc.z, t4.z); acc.w = __fadd_rn(acc.w, t4.w);
            }
            acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f);
            *reinterpret_cast<float4*>(h1s + (size_t)g * EC + f4) = acc;
        }
        __syncthreads();
        for (int i = lg; i < ns; i += nlg) {
            // leaf order rotated by the CTA rank: at any moment the PM_CS senders address PM_CS different owner CTAs
            // (all of them sending leaf j at once would queue on one shared-memory port: measured 2x on the whole search)
            const int g = (i + (int)rank) % ns;
            int pi;
            const int j = slot_tree(g, pi);
            if ((TW && j < 0) || !leaf_flag[j]) continue;
            const float4* x = reinterpret_cast<const float4*>(h1s + (size_t)g * EC);
            float acc = 0.0f;
#pragma unroll
            for (int k4 = 0; k4 < PM_MAX_EC / 4; ++k4) {
                if (4 * k4 < EC) {
                    const float4 v = x[k4];
                    acc = fmaf(wreg[4 * k4 + 0], v.x, acc); acc = fmaf(wreg[4 * k4 + 1], v.y, acc);
                    acc = fmaf(wreg[4 * k4 + 2], v.z, acc); acc = fmaf(wreg[4 * k4 + 3], v.w, acc);
                }
            }
            // to the tree's owner CTA: part2[local slot g / PM_CS][this rank][col]
            pm_remote(part2, (uint32_t)(g % PM_CS))[((size_t)(g / PM_CS) * PM_CS + rank) * H + col] = acc;
        }
        if (prof) { const long long t = clock64(); tB += t - t0; t0 = t; }
        pm_cluster_sync();
        if (prof) { const long long t = clock64(); tS2 += t - t0; t0 = t; }
        // ================= C: h2 and the heads of MY trees (local) =================
        {
            // local slots of the trees this CTA owns (slot jl <-> tree (jl / T)*PM_CS + rank, twist jl % T)
            const int my_slots = (nt - (int)rank + PM_CS - 1) / PM_CS * T;
            // C1: h2 of my trees, thread = column (independent loads per slot)
            for (int jl = lg; jl < my_slots; jl += nlg) {
                float h = 0.0f;
                if (leaf_flag[(TW ? jl / T : jl) * PM_CS + rank]) {
                    const float* q = part2 + (size_t)jl * PM_CS * H + col;
#pragma unroll
                    for (int r = 0; r < PM_CS; ++r) h += q[r * H];               // the K-slices in ascending order
                    h = fmaxf(h + b1s[col], 0.f);
                }
                hbuf[jl * H + col] = h;
            }
            __syncthreads();
            // C2: the 5 head dot products of every slot: 8 lanes per dot product, 3 shuffle steps
            {
                const int dsel = tid >> 3, part = tid & 7;                      // dot product (slot, output) and its eighth of the columns
                const int slot = dsel / 5, o = dsel % 5;
                float acc = 0.0f;
                if (slot < my_slots) {                                           // columns part, part + 8, ..: conflict-free rows of
                    const float* hb = hbuf + slot * H;                           // hbuf and of the padded, transposed head weights
                    const float* hw = headw + o * (H + 8);
                    for (int c = part; c < H; c += 8) acc = fmaf(hb[c], hw[c], acc);
                }
                acc += __shfl_xor_sync(0xffffffffu, acc, 4);
                acc += __shfl_xor_sync(0xffffffffu, acc, 2);
                acc += __shfl_xor_sync(0xffffffffu, acc, 1);
                if (part == 0 && slot < my_slots) red[slot * 8 + o] = acc;
            }
            __syncthreads();
            if (prof) { const long long t = clock64(); tC += t - t0; t0 = t; }
            // ================= D: predict epilogue, expand, child draw (lane 0), backup (owner warps) =================
            if (owner && need) {
                int child = node;
                float v = 0.0f;
                if (lane == 0) {
                    float4 raw;
                    if (!TW) {
                        float l[5];
#pragma unroll
                        for (int o = 0; o < 5; ++o) l[o] = red[warp * 8 + o];
                        raw = make_float4(l[0] + (p.A > 0 ? p.ba[0] : 0.f), l[1] + (p.A > 1 ? p.ba[1] : 0.f), l[2] + (p.A > 2 ? p.ba[2] : 0.f),
                                          l[3] + (p.A > 3 ? p.ba[3] : 0.f));
                        v = l[4] + p.bv[0];
                    } else {                                    // full_predict: every twist's heads, twisted out, then averaged
                        const float np = (float)T;
                        raw = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                        for (int pi = 0; pi < T; ++pi) {
                            const float* rs = red + (warp * T + pi) * 8;
                            float l[4], out[4];
#pragma unroll
                            for (int o = 0; o < 4; ++o) l[o] = rs[o] + (p.A > o ? p.ba[o] : 0.f);
#pragma unroll
                            for (int o = 0; o < 4; ++o) {                // twist-out, policy.rs:95-97 (bias included)
                                const int src = o < p.A ? __ldg(p.act_perms + pi * p.A + o) : o;
                                out[o] = src == 0 ? l[0] : src == 1 ? l[1] : src == 2 ? l[2] : l[3];
                            }
                            twist_accumulate(raw, v, make_float4(out[0], out[1], out[2], out[3]), rs[4] + p.bv[0], np);
                        }
                    }
                    const EnvState s = node_state(m, base + node);
                    float pr[4], cp[4];
                    masked_probs(raw, env_masks(a.env, s), m.A, pr);
                    int nch;
                    const int fc = expand(m, a.env, e, base, node, pr, cp, nch);
                    if (sim >= 0) {                             // next_sample (search.rs:94-100)
                        uint32_t w[4];
                        philox4x32_10(a.ids.gid((uint32_t)e), (uint32_t)(a.t * (a.n_sims + 1) + sim), TWR_RNG_MCTS, a.cid, k0, k1, w);
                        child = nch > 0 ? fc + weighted_index(cp, nch, u32_to_unit_f32(w[0])) : node;
                        if (a.trace) a.trace[((int64_t)sim * m.B + e) * 2 + 1] = child;
                        if (child != node && len >= 0 && len < TWR_MCTS_PATH) m.path[(int64_t)len * m.B + e] = child;
                    }
                }
                if (sim >= 0) {                                 // backup (search.rs:45-53), one lane per path node
                    child = __shfl_sync(0xffffffffu, child, 0);
                    v = __shfl_sync(0xffffffffu, v, 0);
                    if (child != node && len >= 0) { if (len < TWR_MCTS_PATH) ++len; else len = -1; }
                    __syncwarp();
                    backprop_warp(m, e, base, child, len, v, lane);
                }
                __syncwarp();                                   // lane 0's expansion and every lane's backup are read by the whole warp in the next A
            }
        }
        if (prof) { const long long t = clock64(); tD += t - t0; t0 = t; }
        // The owner's global writes of D are read by the same thread in the next A.  Shared-memory reuse needs no third
        // barrier: the next A overwrites (remotely) only the leaf slots of the WRITER's own trees, which no other CTA reads
        // after barrier 2 (C reads the flags of its own trees only); h1s / part2 are rewritten after the next barrier 1.
    }
    if (owner && lane == 0) m.path_len[e] = len;
    if (prof) { a.dbg[0] = tA; a.dbg[1] = tS1; a.dbg[2] = tB; a.dbg[3] = tS2; a.dbg[4] = tC; a.dbg[5] = tD; a.dbg[6] = nt; a.dbg[7] = a.n_sims + 1; }
    pm_cluster_sync();                                      // no CTA may exit while a peer can still write into its shared memory
}

}  // namespace

void launch_mcts_begin(cudaStream_t st, const MctsArgs& a, const int32_t* live, const int32_t* n_live, int64_t max_n) {
    k_mcts_begin<<<grid_for(max_n, 128), 128, 0, st>>>(a, live, n_live);
    TWR_COUNT_LAUNCH();
}
void launch_mcts_expand(cudaStream_t st, const MctsArgs& a, int mode, int sim, int d, int which, int64_t max_n) {
    k_mcts_expand<<<grid_for(max_n, 128), 128, 0, st>>>(a, mode, sim, d, which);
    TWR_COUNT_LAUNCH();
}
void launch_mcts_select(cudaStream_t st, const MctsArgs& a, const int32_t* live, const int32_t* n_live, int sim, int which, int64_t max_n) {
    k_mcts_select<<<grid_for(max_n, 128), 128, 0, st>>>(a, live, n_live, sim, which);
    TWR_COUNT_LAUNCH();
}
void launch_mcts_expand_select(cudaStream_t st, const MctsArgs& a, const int32_t* live, const int32_t* n_live, int sim, int which, int64_t max_n) {
    k_mcts_expand_select<<<grid_for(max_n, 128), 128, 0, st>>>(a, live, n_live, sim, which);
    TWR_COUNT_LAUNCH();
}
void launch_mcts_pre(cudaStream_t st, const MctsArgs& a, const int32_t* live, const int32_t* n_live, int which, int64_t max_n) {
    k_mcts_pre<<<grid_for(max_n, 128), 128, 0, st>>>(a, live, n_live, which);
    TWR_COUNT_LAUNCH();
}
void launch_mcts_read(cudaStream_t st, const MctsArgs& a, int64_t n, float* probs, int32_t* visits) {
    k_mcts_read<<<grid_for(n, 128), 128, 0, st>>>(a, n, probs, visits);
    TWR_COUNT_LAUNCH();
}
void launch_full_predict(cudaStream_t st, const MctsArgs& a, const uint4* cells, const uint32_t* meta, int64_t n, float* probs, float* values) {
    k_full_predict<<<grid_for(n, 128), 128, 0, st>>>(a, cells, meta, n, probs, values);
    TWR_COUNT_LAUNCH();
}
void launch_az_finish(cudaStream_t st, const MctsArgs& a, const CollectBuffers& b, const int32_t* live, int32_t* live_next) {
    k_az_finish<<<grid_for(b.B, 128), 128, 0, st>>>(a, b, live, live_next);
    TWR_COUNT_LAUNCH();
}
void launch_az_remaining(cudaStream_t st, const CollectBuffers& b) {
    k_az_remaining<<<grid_for(b.B, 256), 256, 0, st>>>(b);
    TWR_COUNT_LAUNCH();
}

// Whole-search persistent kernel (small batches, max_expand_depth == 1).  Returns false when it does not apply: the caller
// then runs the lockstep path.
bool launch_mcts_persistent(cudaStream_t st, const MctsArgs& a, const PolicyDev& p, const int32_t* live, const int32_t* n_live, int64_t max_n) {
    if (p.generic || a.max_expand_depth != 1 || max_n < 1) return false;
    if (p.E % (PM_CS * 4) || p.E > PM_CS * PM_MAX_EC || (p.H != 128 && p.H != 256) || p.A > 4) return false;
    // a twisted search takes T = n_perms leaf slots per tree: whole trees per CTA, at least one
    const int T = p.n_perms > 0 ? p.n_perms : 1;
    const int tpc = PM_CS * (PM_TPC / PM_CS / T);          // trees per cluster
    if (tpc < PM_CS) return false;
    void (*kern)(MctsArgs, PolicyDev, const int32_t*, const int32_t*, int, int) =
        p.n_perms > 0 ? k_mcts_persistent<true> : k_mcts_persistent<false>;
    const PmLayout L = pm_layout(p.E, p.H, p.obs_size);
    if (L.total > 227 * 1024) return false;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = PM_CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(PM_THREADS); cfg.dynamicSmemBytes = L.total; cfg.stream = st; cfg.attrs = at; cfg.numAttrs = 1;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total) != cudaSuccess) { cudaGetLastError(); return false; }
    int sms = 0, nc = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cfg.gridDim = dim3((unsigned)((sms / PM_CS) * PM_CS));
    // clusters of this size and shared-memory footprint the device holds at once (a host-side computation): all of a
    // launch's clusters are then resident, although nothing here waits on another cluster
    if (cudaOccupancyMaxActiveClusters(&nc, kern, &cfg) != cudaSuccess) { cudaGetLastError(); nc = 0; }
    if (nc > sms / PM_CS) nc = sms / PM_CS;
    if (nc < 1) return false;
    // Searches cost the same whether a cluster holds 1 or PM_TPC trees (latency bound), so the batch is cut into as few
    // launches as the resident clusters allow; beyond a few thousand trees the lockstep path's batched forward wins.
    const int64_t room = (int64_t)nc * tpc;
    const int n_launch = (int)((max_n + room - 1) / room);
    if (n_launch > 4) return false;
    const int slice = (int)((max_n + n_launch - 1) / n_launch);
    if (getenv("TWISTERL_B200_MCTS_DEBUG"))
        fprintf(stderr, "[mcts] persistent: %lld trees, %d twist(s), %d resident clusters of %d CTAs (%zu B shared memory), %d launch(es) of <= %d trees\n",
                (long long)max_n, p.n_perms, nc, PM_CS, L.total, n_launch, slice);
    MctsArgs args = a;
    static long long* d_dbg_dev[64] = {nullptr};           // debug counters, one buffer per device
    long long* d_dbg = nullptr;
    if (getenv("TWISTERL_B200_MCTS_DEBUG") && dev >= 0 && dev < 64) {
        if (!d_dbg_dev[dev]) cudaMalloc(reinterpret_cast<void**>(&d_dbg_dev[dev]), 8 * sizeof(long long));
        d_dbg = d_dbg_dev[dev];
        args.dbg = d_dbg;
    }
    for (int i = 0; i < n_launch; ++i) {
        const int pos0 = i * slice;
        const int ncl = slice < nc ? slice : nc;
        cfg.gridDim = dim3((unsigned)(ncl * PM_CS));
        if (cudaLaunchKernelEx(&cfg, kern, args, p, live, n_live, pos0, slice) != cudaSuccess) { cudaGetLastError(); return false; }
        TWR_COUNT_LAUNCH();
    }
    if (args.dbg) {
        long long h[8];
        cudaMemcpyAsync(h, d_dbg, sizeof(h), cudaMemcpyDeviceToHost, st);
        cudaStreamSynchronize(st);
        const double n = h[7] > 0 ? (double)h[7] : 1.0;
        fprintf(stderr, "[mcts] cycles per simulation (cluster 0, %lld trees): A descent %.0f | barrier %.0f | B embed+K-slice %.0f | barrier %.0f | C heads %.0f | D expand/backup %.0f\n",
                h[6], h[0] / n, h[1] / n, h[2] / n, h[3] / n, h[4] / n, h[5] / n);
    }
    return true;
}
