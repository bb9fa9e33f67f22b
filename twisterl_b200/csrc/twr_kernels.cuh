// twr_kernels.cuh -- launch wrappers of every kernel in the engine (defined in the .cu files).
#pragma once
#include "twr_common.cuh"

// Device-resident policy: fp32 master copy in the blob layout of include/twisterl_b200.h plus
// derived operand layouts for the tensor-core path.
struct PolicyDev {
    int obs_size, E, H, A, n_obs;  // n_obs = one-hot indices per observation (cells)
    int n_perms;
    const float* emb;     // [obs_size][E]
    const float* emb_b;   // [E]
    const float* w1;      // [E][H]   (k-major: W.T.flatten())
    const float* b1;      // [H]
    const float* wa;      // [H][A]
    const float* ba;      // [A]
    const float* wv;      // [H]
    const float* bv;      // [1]
    const int32_t* obs_perms;  // [n_perms][obs_size]
    const int32_t* act_perms;  // [n_perms][A]
    // operand image of the tensor-core kernel (fp16 hi/lo split and fp8 corrections, pre-swizzled K-major tiles in
    // streaming order), see k_tc2_pack in twr_forward_tc2.cu; NULL: the policy runs another kernel
    const void* tc_pack;
    // > 0: the forward runs on the COMPACT table of a GridWorld board of compact_n cells, only its 4 * compact_n reachable
    // rows (row (i, v) = i * compact_n + v, v in 0..3; examples/grid_world/src/lib.rs:74-81,161-163) at i * 4 + v.
    // With tc_pack: the pair kernel's GEMM1 image is built so at policy creation, and such a policy takes the tensor-core
    // path only for GridWorld envs of that size whose observation comes from the env state.  Without: set per forward by
    // the engine for GridWorld boards above 32 cells, k_forward_fp32 stages only those rows.
    int compact_n;
    // > 0: obs_size = tc_fold^2 and every twist maps each block of tc_fold consecutive rows onto another block, so an
    // observation that holds exactly ONE index per block (what Puzzle / GridWorld envs produce) selects exactly one row of
    // block 0 before and after a twist: the f16f8c operand image carries the embedding bias on the rows of block 0 and
    // the kernel's epilogue-1 skips the bias add (k_forward_tc2<.., .., FOLD>)
    int tc_fold;
    // General layer stacks (SURVEY 8f row f4): any policy that is not "embedding+ReLU -> one common Linear+ReLU ->
    // single-Linear heads" runs k_forward_generic (twr_forward_generic.cu) from this description instead.
    int generic;                              // 1: the fields above (w1..bv, H) are unused
    int emb_relu;
    int n_common, n_action, n_value;          // Linear counts; lin[] holds common..., action_net..., value_net... in order
    int max_width;                            // widest activation vector (embedding or any Linear output)
    struct Lin { const float* w; const float* b; int in, out, relu; } lin[12];
};
#define TWR_MAX_STACK 4                       // Linears per stack
size_t forward_generic_smem(const PolicyDev& p);
void   launch_forward_generic(cudaStream_t s, const PolicyDev& p, const struct ForwardArgs& a);

struct CollectBuffers {
    int64_t B;      // envs (episodes) in this collect
    int Tmax;       // horizon + 1 records at most
    // env state
    uint4* cells; uint32_t* meta;
    // live lists: position-indexed
    int32_t* live_a; int32_t* live_b; int32_t* n_live;  // n_live[Tmax+1]
    // forward outputs, position-indexed
    float4* logits; float* values;
    // time-major records [t][env]
    uint4* rec_state; float4* rec_logits; float* rec_value; float* rec_reward;
    float* rec_adv; float* rec_ret; uint8_t* rec_action; int8_t* rec_perm;
    int32_t* ep_len;      // [B]
    int64_t* ep_off;      // [B] record offset of local episode e (plain local order; the id rotation gives merge order)
    int32_t* ep_len_id;   // [total episodes] episode length by episode id (filled by k_episode_offsets)
    int64_t out_base;     // records of earlier sub-batches (pipelined host collect)
    int obs_u8;           // 1: compaction writes one byte per observation index (twr_host_buffers.obs_u8); 0: u16 indices
    int pack_misc;        // compaction writes ONE byte per record into out_actions -- action | reward code << 2 | (perm + 1) << 4 --
                          // and skips out_perms / out_rewards / out_advs: the pipelined host collect rebuilds those on the host
                          // (Puzzle rewards take three values, puzzle.rs:171-177; advs = rets - values, ppo.rs:87-91)
    unsigned long long* stats;  // [0] successes, [1] total records ; double at [2] = reward sum
    // compacted outputs
    uint16_t* out_obs; float* out_logits; float* out_values; float* out_rewards;
    float* out_advs; float* out_rets; uint8_t* out_actions; int8_t* out_perms;
};

struct StepArgs {
    EnvParams env;
    uint64_t seed; uint32_t cid; EnvIds ids;
    int n_perms; int A;
    int t;
};

// K1: batched Env-trait kernels (parity API + reset)
void launch_envs_reset(cudaStream_t s, const EnvParams& p, uint4* cells, uint32_t* meta, int64_t n,
                       uint64_t seed, EnvIds ids, uint32_t cid, int32_t* live, int32_t* n_live0);
void launch_envs_fresh(cudaStream_t s, const EnvParams& p, uint4* cells, uint32_t* meta, int64_t n);
void launch_envs_set_state(cudaStream_t s, const EnvParams& p, uint4* cells, uint32_t* meta, int64_t n,
                           const int64_t* d_states);
void launch_envs_step(cudaStream_t s, const EnvParams& p, uint4* cells, uint32_t* meta, int64_t n,
                      const int32_t* d_actions);
void launch_envs_query(cudaStream_t s, const EnvParams& p, const uint4* cells, const uint32_t* meta, int64_t n,
                       int64_t* d_states, int32_t* d_obs, uint8_t* d_masks, float* d_reward, uint8_t* d_final,
                       uint8_t* d_success, int32_t* d_depth);
void launch_mask_logits(cudaStream_t s, const EnvParams& p, const uint4* cells, const uint32_t* meta, int64_t n,
                        int A, float4* logits);
// K3 standalone
void launch_sample(cudaStream_t s, const float* d_logits, int64_t n, int A, uint64_t seed, uint32_t env_id_base,
                   uint32_t step, uint32_t cid, int32_t* d_actions, float* d_uniforms);
// K3+K4a+K1 fused collect step: mask, Gumbel-max sample, trajectory write, env step, live compaction
void launch_collect_step(cudaStream_t s, const StepArgs& a, const CollectBuffers& b, const int32_t* live_cur,
                         int32_t* live_next);
// survivors (ep_len == 0) of live_cur[0..*n_cur) -> live_next, count -> *n_next (must be zeroed)
void launch_compact_live(cudaStream_t s, const int32_t* live_cur, const int32_t* n_cur, const int32_t* ep_len, int64_t max_n,
                         int32_t* live_next, int32_t* n_next);
// K4b GAE, stand-alone over concatenated episodes (the PPO collect runs it inside launch_compact_gae)
void launch_gae_concat(cudaStream_t s, const float* r, const float* v, const int64_t* off, int64_t n_ep,
                       float gamma, float lambda, float* adv, float* ret);
// K5 episode offsets in merged order + transpose/compaction into concatenated episodes
void launch_episode_offsets(cudaStream_t s, const CollectBuffers& b, const EnvIds& ids);
void launch_compact(cudaStream_t s, const EnvParams& p, const CollectBuffers& b, int A);
void launch_compact_gae(cudaStream_t s, const EnvParams& p, const CollectBuffers& b, int A, float gamma, float lambda);   // GAE fused into the compaction
// the four statistics words of a collect -> mapped pinned host memory (no copy engine involved)
void launch_publish_stats(cudaStream_t s, const unsigned long long* stats, unsigned long long* mapped_host);

// K2 policy forward.  `live` may be NULL (identity); n_live_ptr may be NULL (use n).
struct ForwardArgs {
    EnvParams env;
    uint64_t seed; uint32_t cid; EnvIds ids; int t;  // twist pick stream
    const int32_t* perm_idx;  // explicit per-position twist (parity API) or NULL -> Philox pick
    const uint4* cells; const int32_t* live; const int32_t* n_live_ptr; int64_t n;
    const int32_t* obs_rows;  // optional [n][n_obs] sparse obs given directly (Policy.forward API); overrides cells
    int obs_blocks;           // obs_rows only: every row holds exactly one index per block of PolicyDev::tc_fold rows (checked on the host)
    float4* logits; float* values;
    // fused collect step (k_forward_tc2 only): when `fused` != 0 the epilogue does k_collect_step's work
    int fused; StepArgs step; CollectBuffers cb; int32_t* live_next;
    int t_count;      // steps t .. t+t_count-1 in this launch (fused pair kernel only; 0/1 = one step)
    // balanced item schedule of the persistent pair kernel: groups beyond a whole number per CTA pair are cut along
    // TIME into pieces handed from pair to pair; bal_flags[g] counts the finished steps of such a group (zeroed per launch)
    int32_t* bal_flags; int bal_delta;   // bal_delta: extra item slots granted to each hand-off (0 = balancing off)
    // split-operand terms of the tensor-core forward (k_forward_tc2): 0 = all (f16x2); otherwise 8 | bit 0 one-hot x table_lo
    // | bit 1 h1_lo x W_hi | bit 2 h1_hi x W_lo on top of the hi x hi products (TWR_PREC_F16X2_W16 = 8 | 1 | 2)
    int tc_terms;
    int dbg_flags;    // ablations (k_forward_tc2, timing only): 1 skip epilogue-1 TMEM traffic, 2 no operand TMA traffic, 4 skip GEMM2 MMAs, 8 skip GEMM1 MMAs
    long long* dbg;   // optional [gridDim][16] cycle counters written by k_forward_tc2 (debug/profiling), TWR_DBG_WORDS long
};
// ForwardArgs::dbg: 16 counters for each of up to TWR_DBG_CTAS CTAs (one per SM of a B200), then at TWR_DBG_TRACE the
// event trace of CTA 0 (8 items x 32 clock64 stamps)
#define TWR_DBG_CTAS 148
#define TWR_DBG_TRACE (TWR_DBG_CTAS * 16)
#define TWR_DBG_WORDS (TWR_DBG_TRACE + 256)
// does k_forward_fp32 take this policy (its table, or the compact one when compact_n > 0) for observations of up to
// n_obs indices?
int  forward_fp32_supported(const PolicyDev& p, int n_obs, const char** why);
bool launch_forward_fp32(cudaStream_t s, const PolicyDev& p, const ForwardArgs& a);   // false: shape does not fit shared memory
// Tensor-core (CTA-pair, tcgen05 cta_group::2) variant, twr_forward_tc2.cu; `pack` is its operand image (PolicyDev::tc_pack)
int    forward_tc2_supported(const PolicyDev& p);
// builds / refreshes the packed operand tiles from the fp32 blob
size_t forward_tc2_pack_bytes(const PolicyDev& p);
void   launch_forward_tc2_pack(cudaStream_t s, const PolicyDev& p, void* pack);
bool   launch_forward_tc2(cudaStream_t s, const PolicyDev& p, const ForwardArgs& a, const void* pack);  // false: forward_tc2_prepare missing / failed
// resolves, at policy creation, everything a later launch depends on (tensor map of the operand image, kernel attributes)
bool   forward_tc2_prepare(const PolicyDev& p, const void* pack);
void   forward_tc2_forget(const void* pack);    // before the operand image is freed

// f1: batched single_solve step (rust/src/rl/solve.rs:17-71) for every live env
struct SolveArgs {
    EnvParams env; uint64_t seed; uint32_t cid; EnvIds ids; int A; int t; int deterministic; int64_t B;
    uint4* cells; uint32_t* meta; const float4* logits; int32_t* n_live;   // n_live[t], n_live[t+1]
    float* total; uint8_t* success; uint8_t* act_rec;  // act_rec [T][B] or NULL
    int32_t* n_steps;   // [B] number of actions taken
    const float* mcts_probs;   // [B][A] root visit distribution of predict_probs_mcts, or NULL -> Policy::predict of `logits`
};
void launch_solve_step(cudaStream_t s, const SolveArgs& a, const int32_t* live_cur, int32_t* live_next);
void launch_envs_broadcast(cudaStream_t s, const uint4* src_cells, const uint32_t* src_meta, uint4* cells, uint32_t* meta, int64_t n);

// K6: batched MCTS (twr_mcts.cu)
#define TWR_MCTS_PATH 96                       // recorded descent path entries per env (deeper paths fall back to the parent walk)
struct MctsPool {
    int64_t B; int P; int A;                   // node (e, i) lives at e*P + i, root at i = 0
    uint4* cells; uint32_t* meta;              // the node's env (MCTSNode.state)
    int32_t* parent;
    uint4* node;                               // {visit_count, value_sum, prior, first_child | n_children << 20 | action << 24}
    int32_t* n_nodes;                          // [B]
    int32_t* path; int32_t* path_len;          // [TWR_MCTS_PATH][B] node indices of the current descent, [B] its length (-1: overflow)
};
struct MctsArgs {
    EnvParams env; uint64_t seed; uint32_t cid; EnvIds ids;
    int t; int n_sims; int max_expand_depth; float C;
    MctsPool pool;
    const uint4* env_cells; const uint32_t* env_meta;    // the envs being searched from
    int32_t* fwd_list; int32_t* fwd_env; int32_t* fwd_count;   // leaf batch: node indices, env ids, two counters
    int32_t* leaf_pos;                                          // [B] leaf-batch slot of env e in the current simulation
    const float4* logits; const float* values;           // forward outputs, indexed by leaf-batch position
    // twisted policies (Policy::full_predict): one forward per twist pi, its outputs at logits / values + pi * twist_stride
    int n_perms; int64_t twist_stride;
    int32_t* cur_node; float* cur_value; uint8_t* active; // per env, current simulation
    int32_t* trace;   // optional [n_sims][B][2] (parity API): leaf of the descent, node the value was backed up from
    long long* dbg;   // optional [8] cycle counters of cluster 0 / CTA 0 / thread 0 of k_mcts_persistent (TWISTERL_B200_MCTS_DEBUG)
};
void launch_mcts_begin(cudaStream_t s, const MctsArgs& a, const int32_t* live, const int32_t* n_live, int64_t max_n);
void launch_mcts_expand(cudaStream_t s, const MctsArgs& a, int mode, int sim, int d, int which, int64_t max_n);
void launch_mcts_select(cudaStream_t s, const MctsArgs& a, const int32_t* live, const int32_t* n_live, int sim, int which, int64_t max_n);
void launch_mcts_expand_select(cudaStream_t s, const MctsArgs& a, const int32_t* live, const int32_t* n_live, int sim, int which, int64_t max_n);
void launch_mcts_pre(cudaStream_t s, const MctsArgs& a, const int32_t* live, const int32_t* n_live, int which, int64_t max_n);
void launch_mcts_read(cudaStream_t s, const MctsArgs& a, int64_t n, float* probs, int32_t* visits);
bool launch_mcts_persistent(cudaStream_t s, const MctsArgs& a, const PolicyDev& p, const int32_t* live, const int32_t* n_live, int64_t max_n);
// Policy::full_predict of n envs from the forward outputs of every twist (a.logits / a.values, a.n_perms slices):
// probs [n][a.pool.A], values [n]; the leaf evaluation of the lockstep search
void launch_full_predict(cudaStream_t s, const MctsArgs& a, const uint4* cells, const uint32_t* meta, int64_t n, float* probs, float* values);
void launch_az_finish(cudaStream_t s, const MctsArgs& a, const CollectBuffers& b, const int32_t* live, int32_t* live_next);
void launch_az_remaining(cudaStream_t s, const CollectBuffers& b);
