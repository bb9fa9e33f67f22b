/*
 * twisterl_b200.h -- C ABI of the B200-native rollout engine for twisteRL.
 *
 * This is the drop-in boundary for the reference's Rust data-collection path.  Every entry
 * point names the reference interface it replaces (paths relative to the reference checkout).
 * A Rust shim (`extern "C"` block + `impl Collector for B200Collector`) binds it 1:1 -- see
 * INTEGRATION.md; in this repository the host side above it is Python (the twisterl_b200 package),
 * mirroring the PyO3 module `twisterl.twisterl.{env,nn,collector}`.
 *
 * Conventions
 *   - plain C, no torch / CUDA types in signatures; device pointers travel as `void*`/typed
 *     pointers documented "device"; everything else is a HOST pointer.
 *   - every function returns TWR_OK (0) or a negative twr_status; the message is in
 *     twr_last_error() (thread-local), which the host maps to RuntimeError exactly like
 *     rust/src/python_interface/error_mapping.rs:29-33.
 *   - one engine per CUDA device; an engine is used from one host thread at a time.
 *   - there is NO CPU fallback: without a CUDA device twr_engine_create fails.
 *
 * RNG contract (shared with oracle/twr_oracle.h): Philox4x32-10, key = 64-bit seed,
 * counter = (global_env_id, index, kind, collect_id); kinds: 0 reset, 1 twist pick, 2 action
 * sampling.  The reference itself is unseedable (rand::thread_rng, rl/evaluate.rs:29).
 */
#ifndef TWISTERL_B200_H
#define TWISTERL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TWR_ABI_VERSION 3

typedef enum {
    TWR_OK = 0,
    TWR_ERR_INVALID = -1,     /* bad argument */
    TWR_ERR_UNSUPPORTED = -2, /* env / policy shape the device path does not implement */
    TWR_ERR_CUDA = -3,        /* CUDA runtime failure (no device, launch error, OOM) */
    TWR_ERR_STATE = -4        /* call order (e.g. to_host before collect) */
} twr_status;

/* TWR_ENV_PUZZLE takes boards of up to 16 cells (one byte per cell in the env state); TWR_ENV_PUZZLE_WIDE is the same
 * env for boards of up to 25 cells (5x5, 4x6, ...: 5-bit cells in the same 16 bytes), and what a Puzzle above 16 cells
 * must be created as.  Both behave exactly as envs::Puzzle. */
typedef enum { TWR_ENV_PUZZLE = 0, TWR_ENV_GRIDWORLD = 1, TWR_ENV_PUZZLE_WIDE = 2 } twr_env_kind;

/* arithmetic of the policy forward (kernel K2) */
typedef enum {
    TWR_PREC_FP32 = 0,  /* SIMT fp32 FMA; parity bar 1e-5 */
    TWR_PREC_F16X2 = 1, /* tcgen05, every operand split into fp16 hi+lo (hi*hi + hi*lo + lo*hi), fp32 TMEM accumulate:
                         * fp32-grade results (1e-5 measured on the shipped trained weights; bar 1e-3).
                         * Policies whose shape does not fit the tensor-core kernel and multiset observations run the
                         * fp32 SIMT kernel on the same engine. */
    TWR_PREC_F16X2_W16 = 2, /* same kernel, the common Linear's weight held as ONE fp16 term (h1_hi*W + h1_lo*W; table and
                         * activations stay split): 2/3 of the GEMM2 work, 7e-4 worst case on the shipped trained
                         * weights -- the cheapest fp16 operand combination inside the 1e-3 bar (tests/test_gpu_precision.py
                         * holds the whole ladder; plain fp16 operands measure 4e-3 and miss it). */
    TWR_PREC_F16_F8C = 3 /* the terms of F16X2_W16 with the two CORRECTION products (one-hot * table_lo, h1_lo * W) issued as
                         * fp8 MMAs (K = 32 per instruction): a correction is ~2^-12 of its main term, so 2-3 mantissa bits
                         * of it keep the same 1e-3 grade at 3/4 of the tensor-core instructions.  Same bar, same tests. */
} twr_precision;

typedef struct twr_engine twr_engine;
typedef struct twr_policy twr_policy;
typedef struct twr_envs twr_envs;

int         twr_abi_version(void);
const char* twr_last_error(void);
/* number of CUDA devices visible (0 when none / no driver); never fails */
int         twr_device_count(void);

/* ------------------------------------------------------------------ engine --- */
typedef struct {
    int32_t  device;      /* CUDA ordinal */
    int32_t  precision;   /* twr_precision */
    uint64_t seed;        /* Philox key */
    int32_t  rank, world; /* env shard of this engine: global env id = rank*num_episodes + e */
    void*    stream;      /* cudaStream_t to launch on, NULL = engine-owned stream */
} twr_engine_cfg;

int  twr_engine_create(const twr_engine_cfg* cfg, twr_engine** out);
void twr_engine_destroy(twr_engine* e);
int  twr_engine_synchronize(twr_engine* e);
/* kernels launched by this engine since creation (bench.py reports the delta as gpu_launches) */
int64_t twr_engine_launch_count(const twr_engine* e);

/* --------------------------------------------------------------------- env --- */
/* Device-side equivalent of a `Box<dyn Env>` (rust/src/rl/env.rs:18-66): the constructor
 * arguments of envs::Puzzle (rust/src/envs/puzzle.rs:34-42, python_interface/env.rs:124-134)
 * or of grid_world::GridWorld (examples/grid_world/src/lib.rs:23-41) plus its difficulty.
 * Puzzle boards of up to 25 cells run on the device (above 16 cells as TWR_ENV_PUZZLE_WIDE); larger
 * ones are refused with TWR_ERR_UNSUPPORTED.  GridWorld takes 3..64 cells (up to 8x8) with the same encoding at
 * every size; larger boards are refused with TWR_ERR_UNSUPPORTED. */
typedef struct {
    int32_t kind;        /* twr_env_kind */
    int32_t width, height;
    int32_t difficulty;
    int32_t depth_slope; /* puzzle */
    int32_t max_depth;   /* puzzle: max_depth; grid_world: max_steps */
} twr_env_spec;

/* ------------------------------------------------------------------ policy --- */
/* One Linear as nn.Linear(weights_vector, bias_vector, apply_relu) receives it
 * (rust/src/python_interface/layers.rs:19-33): weights = W.T.flatten(), w[i*out + o] == W[o][i]. */
typedef struct {
    const float* weights; /* [in][out] */
    const float* bias;    /* [out] */
    int32_t in, out, apply_relu;
} twr_linear_desc;

/* nn.Policy(embeddings, common, action_net, value_net, obs_perms, act_perms)
 * (rust/src/python_interface/policy.rs:27-31, rust/src/nn/policy.rs:20-32), in the layouts
 * `BasicPolicy.to_rust()` produces (src/twisterl/nn/utils.py:17-59). */
typedef struct {
    const float* emb_vectors;  /* [obs_size][emb_size]  (EmbeddingBag vec_vectors) */
    const float* emb_bias;     /* [emb_size] */
    int32_t obs_size, emb_size, emb_apply_relu;
    /* EmbeddingBag obs_shape / conv_dim.  obs_shape_len == 2 is the Conv1dPolicy path (rust/src/nn/layers.rs:63-77,
     * src/twisterl/nn/utils.py:68-75): emb_vectors is [obs_size = obs_shape[conv_dim]][v] with
     * v = emb_size / obs_shape[1 - conv_dim], emb_bias stays [emb_size]; the observation indices then range over
     * obs_shape[0] * obs_shape[1]. */
    int32_t obs_shape[2], obs_shape_len, conv_dim;
    /* the three Sequentials (rust/src/nn/modules.rs:16-34): 0..4 common Linears, 1..4 per head; the shape
     * "one common Linear+ReLU, single-Linear heads" runs the tcgen05 / fp32 tile kernels, any other the generic fp32 kernel */
    const twr_linear_desc* common;     int32_t n_common;
    const twr_linear_desc* action_net; int32_t n_action;
    const twr_linear_desc* value_net;  int32_t n_value;
    const int32_t* obs_perms;  /* [n_perms][obs_size] or NULL */
    const int32_t* act_perms;  /* [n_perms][num_actions] or NULL */
    int32_t n_perms;
} twr_policy_desc;

/* Uploads the weights (H2D) and builds the device-side operand layouts.  The device path
 * implements the BasicPolicy family the three reference configs use: 1-D EmbeddingBag + ReLU,
 * exactly one common Linear+ReLU (width 64..256, multiple of 64), single-Linear action and
 * value heads, <= 4 actions.  Anything else returns TWR_ERR_UNSUPPORTED. */
int  twr_policy_create(twr_engine* e, const twr_policy_desc* desc, twr_policy** out);
/* In-place refresh with the same shapes (replaces rebuilding nn.Policy every iteration,
 * src/twisterl/rl/algorithm.py:91-93). */
int  twr_policy_update(twr_policy* p, const twr_policy_desc* desc);
/* Builds the policy straight from a safetensors checkpoint of the reference's BasicPolicy / Conv1dPolicy state dict
 * (src/twisterl/utils.py:131-190: tensors embeddings.weight/bias or conv_layer.weight, common.{0,2,..}, action.{..},
 * value.{..}; F32), putting the tensors into the layouts `to_rust()` produces (src/twisterl/nn/utils.py:17-75).
 * obs_shape / conv_dim are only read for a Conv1d checkpoint; obs_perms / act_perms as in twr_policy_desc. */
int  twr_policy_create_from_safetensors(twr_engine* e, const char* path, const int32_t* obs_shape, int32_t obs_shape_len,
                                        int32_t conv_dim, const int32_t* obs_perms, const int32_t* act_perms,
                                        int32_t n_perms, twr_policy** out);
/* Flat fp32 parameter blob: [emb_vectors][emb_bias][common w][common b][action w][action b]
 * [value w][value b], each in the layout above.  update_from_device takes a DEVICE pointer
 * (e.g. the buffer an NCCL broadcast just filled). */
int64_t twr_policy_blob_floats(const twr_policy* p);
int  twr_policy_update_from_device(twr_policy* p, const float* d_blob);
int  twr_policy_blob_device_ptr(twr_policy* p, float** d_blob);
void twr_policy_destroy(twr_policy* p);

/* ------------------------------------------------- batched env (parity API) --- */
/* n independent envs in structure-of-arrays form on the device; the methods are the Env trait
 * (rust/src/rl/env.rs:18-66) applied to all n at once. */
int  twr_envs_create(twr_engine* e, const twr_env_spec* spec, int64_t n, twr_envs** out);
void twr_envs_destroy(twr_envs* v);
int  twr_envs_set_difficulty(twr_envs* v, int32_t difficulty);
/* states: [n][width*height] boards (Env::set_state) */
int  twr_envs_set_state(twr_envs* v, const int64_t* states);
/* Puzzle::set_position (rust/src/envs/puzzle.rs:71-73, python_interface/env.rs:150-153): pokes ONE cell of env `env`;
 * blank location and depth are left alone, exactly like the reference. */
int  twr_envs_set_cell(twr_envs* v, int64_t env, int32_t cell, int32_t value);
/* Env::reset for all n, env i drawing from Philox stream (env_id_base + i, *, reset, collect_id) */
int  twr_envs_reset(twr_envs* v, uint32_t env_id_base, uint32_t collect_id);
/* Env::step with forced actions[n] */
int  twr_envs_step(twr_envs* v, const int32_t* actions);
int  twr_envs_get_state(twr_envs* v, int64_t* states /* [n][cells] */);
int  twr_envs_observe(twr_envs* v, int32_t* obs /* [n][cells] sparse one-hot indices */);
int  twr_envs_masks(twr_envs* v, uint8_t* masks /* [n][num_actions] */);
int  twr_envs_reward(twr_envs* v, float* rewards /* [n] */);
int  twr_envs_is_final(twr_envs* v, uint8_t* finals /* [n] */);
int  twr_envs_success(twr_envs* v, uint8_t* success /* [n] */);
int  twr_envs_depth(twr_envs* v, int32_t* depth /* [n] puzzle depth / grid_world steps_left */);

/* Policy::_raw_predict / forward_with_perm (rust/src/nn/policy.rs:56-100) for all n envs.
 * perm_idx: [n] twist index per env (-1 = none) or NULL.  apply_masks != 0 writes -1e10 on
 * masked actions like forward_with_perm.  logits [n][num_actions], values [n]. */
int  twr_policy_forward(twr_engine* e, const twr_policy* p, twr_envs* v, const int32_t* perm_idx,
                        int32_t apply_masks, float* logits, float* values);

/* Policy::_raw_predict for n sparse observations given directly: obs [n][n_obs] one-hot indices
 * (what Env::observe returns), as python_interface/policy.rs:33-44 receives them.  n_obs <= 64. */
int  twr_policy_forward_obs(twr_engine* e, const twr_policy* p, const int32_t* obs, int64_t n, int32_t n_obs,
                            const int32_t* perm_idx, float* logits, float* values);

/* Policy::full_predict (nn/policy.rs:102-126) for every env of `v`: the raw logits and value of each twist, each divided
 * by n_perms and added in twist order, then the masked exp / (sum + 1e-6) of Policy::predict.  probs [n][num_actions],
 * values [n].  Without twists it is Policy::predict.  This is the leaf evaluation of the MCTS searches, by the same
 * launches and the same averaging code. */
int  twr_policy_full_predict(twr_engine* e, const twr_policy* p, twr_envs* v, float* probs, float* values);

/* Debug: one forward over `v` with per-CTA cycle counters of the tensor-core kernel's pipeline waits
 * (16 int64 per CTA, max_ctas >= number of SMs; the counters are written at the end of k_forward_tc2 in
 * twr_forward_tc2.cu, and scripts/profile_tc.py names them). */
int  twr_debug_forward_profile(twr_engine* e, const twr_policy* p, twr_envs* v, int64_t* counters, int32_t max_ctas,
                               int32_t experiment_flags /* 0 = none; results are invalid when non-zero */);
/* Debug / precision ladder: which split-operand terms the tensor-core forward of this engine accumulates on top of the
 * hi*hi products: bit 0 one-hot * table_lo, bit 1 h1_lo * W_hi, bit 2 h1_hi * W_lo (7 = TWR_PREC_F16X2, 3 = .._W16,
 * 0 = plain fp16 operands; 16 | 3 = the two corrections of .._W16 as fp8 products = TWR_PREC_F16_F8C).
 * -1 restores the engine's precision. */
int  twr_debug_set_tc_terms(twr_engine* e, int32_t terms);

/* sample_from_logits (rust/src/nn/policy.rs:169-172) for n logit rows, row i using the uniforms
 * of Philox stream (env_id_base + i, step, sample, collect_id).  uniforms_out may be NULL. */
int  twr_sample(twr_engine* e, const float* logits, int64_t n, int32_t num_actions,
                uint32_t env_id_base, uint32_t step, uint32_t collect_id,
                int32_t* actions, float* uniforms_out /* [n][num_actions] */);

/* per-episode GAE (rust/src/collector/ppo.rs:82-92) over `num_episodes` concatenated episodes;
 * offsets has num_episodes+1 entries. */
int  twr_gae(twr_engine* e, const float* rewards, const float* values, const int64_t* offsets,
             int64_t num_episodes, float gamma, float lambda, float* advs, float* rets);

/* ----------------------------------------------------------------- collect --- */
typedef struct {
    int64_t n_records;      /* R = sum of episode lengths */
    int64_t num_episodes;
    int32_t n_cells, num_actions;
    int64_t successes;      /* episodes that ended with Env::success() */
    double  reward_sum;     /* sum over episodes of the terminal-state reward */
    /* DEVICE pointers, owned by the engine, valid until the next collect / destroy.
     * Episodes are concatenated in the reference's merge order [last, 0, 1, ..., n-2]
     * (rust/src/collector/collector.rs:40-46). */
    const uint16_t* obs;      /* [R][n_cells]  CollectedData.obs (sparse one-hot indices) */
    const float*    logits;   /* [R][num_actions]  masked logits, CollectedData.logits */
    const float*    values;   /* [R] */
    const float*    rewards;  /* [R] */
    const float*    advs;     /* [R]  additional_data["advs"] */
    const float*    rets;     /* [R]  additional_data["rets"] */
    const uint8_t*  actions;  /* [R] */
    const int8_t*   perms;    /* [R]  -1 == None */
    const int32_t*  ep_len;   /* [num_episodes] by episode id */
} twr_collected;

/* PPOCollector::collect (rust/src/collector/ppo.rs:108-126; PyBaseCollector.collect,
 * rust/src/python_interface/collector.rs:147-151).  Episode e of this call draws from Philox
 * env id rank*num_episodes + e and collect_id = number of collects this engine has run
 * (or the value set by twr_engine_set_collect_id). */
int  twr_ppo_collect(twr_engine* e, const twr_env_spec* spec, const twr_policy* p,
                     int64_t num_episodes, float gamma, float lambda, twr_collected* out);
int  twr_engine_set_collect_id(twr_engine* e, uint32_t collect_id);

/* Host mirror of twr_collected; the caller owns every buffer (capacity in records). */
typedef struct {
    int64_t   capacity;     /* records each buffer can hold */
    uint16_t* obs;          /* [capacity][n_cells] */
    float*    logits;       /* [capacity][num_actions] */
    float*    values;
    float*    rewards;
    float*    advs;
    float*    rets;
    uint8_t*  actions;
    int8_t*   perms;
    int32_t*  ep_len;       /* [num_episodes] or NULL */
    uint8_t*  obs_u8;       /* alternative to `obs` for envs with obs_size <= 256 (both puzzles): the same indices,
                             * one byte each -- halves the largest D2H stream of twr_ppo_collect_host.  Used when
                             * `obs` is NULL; the binding widens to usize either way (CollectedData.obs is Vec<Vec<usize>>) */
} twr_host_buffers;

/* D2H of the last collect into caller buffers (any field may be NULL to skip it) */
int  twr_collected_to_host(twr_engine* e, const twr_host_buffers* dst);
/* upper bound of records a collect of num_episodes can produce (episodes * (horizon+1)) */
int64_t twr_max_records(const twr_env_spec* spec, int64_t num_episodes);

/* End-to-end call with HOST buffers on both sides: uploads the weights in `desc` into `p`
 * (H2D), collects, and copies the result into `dst` (D2H).  This is what a Rust
 * `impl Collector` would call; bench.py times it as `e2e`. */
int  twr_ppo_collect_host(twr_engine* e, const twr_env_spec* spec, twr_policy* p,
                          const twr_policy_desc* desc, int64_t num_episodes, float gamma, float lambda,
                          const twr_host_buffers* dst, twr_collected* out);

/* collector.evaluate (rust/src/rl/evaluate.rs:22-89, python_interface/env.rs:194-207).  With num_mcts_searches > 0
 * every step's action distribution is predict_probs_mcts of the current state (rl/solve.rs:37-48) instead of Policy::predict:
 * num_episodes x [reset, best of num_searches rollouts of single_solve (rl/solve.rs:17-101)] run as one
 * device batch.  Returns (mean success, mean total reward) of the per-episode best (success, reward).  The search
 * evaluates its leaves with Policy::full_predict (rl/search.rs:113,150): a policy with twists averages every twist, as
 * twr_policy_full_predict does. */
int  twr_evaluate(twr_engine* e, const twr_env_spec* spec, const twr_policy* p, int64_t num_episodes,
                  int32_t deterministic, int32_t num_searches, int32_t num_mcts_searches, float C,
                  int32_t max_expand_depth, float* success_rate, float* mean_reward);
/* same, also returning every episode's best (success, reward) (what rl/evaluate.rs:41-46 sums): [num_episodes] each, or NULL */
int  twr_evaluate_episodes(twr_engine* e, const twr_env_spec* spec, const twr_policy* p, int64_t num_episodes,
                           int32_t deterministic, int32_t num_searches, int32_t num_mcts_searches, float C,
                           int32_t max_expand_depth, float* success_rate, float* mean_reward, float* best_success,
                           float* best_reward);
/* collector.solve (rl/solve.rs:73-101) from the state held by the one-env batch `start`: best of
 * num_searches rollouts; writes its action list (actions may be NULL to only query the score).  With
 * num_mcts_searches > 0 a policy with twists is searched with full_predict over all of them, as in twr_evaluate. */
int  twr_solve(twr_engine* e, twr_envs* start, const twr_policy* p, int32_t deterministic, int32_t num_searches,
               int32_t num_mcts_searches, float C, int32_t max_expand_depth,
               float* success, float* reward, int32_t* actions, int32_t max_actions, int32_t* n_actions);

/* AZCollector::collect (rust/src/collector/az.rs:112-130; python_interface/collector.rs:172-188): per record a
 * batched MCTS (predict_probs_mcts, rust/src/rl/search.rs:104-189) whose leaves are evaluated by the same
 * forward kernel as the PPO path.  In the result `logits` holds the MCTS visit distribution (what the reference
 * stores in CollectedData.logits), `rets` holds additional_data["remaining_values"] (az.rs:93), `rewards` and
 * `actions` the per-record reward / drawn action; `values`, `advs` are zero and `perms` is -1.  A policy with twists
 * is refused (TWR_ERR_UNSUPPORTED): the reference's AlphaZero trainer clears them (rl/az.py:24-26). */
int  twr_az_collect(twr_engine* e, const twr_env_spec* spec, const twr_policy* p, int64_t num_episodes,
                    int32_t num_mcts_searches, float C, int32_t max_expand_depth, twr_collected* out);
/* predict_probs_mcts for every env of `v` at once (parity API): probs / visit counts [n][num_actions].  Env i
 * draws from Philox stream env_id_base + i at record index t.  Leaves are evaluated with Policy::full_predict: a
 * policy with twists averages all of them (twr_policy_full_predict). */
int  twr_mcts_probs(twr_engine* e, const twr_policy* p, twr_envs* v, int32_t n_sims, float C, int32_t max_expand_depth,
                    uint32_t env_id_base, uint32_t collect_id, int32_t t, float* probs, int32_t* visits);

/* ------------------------------------------------------------ multi-GPU --- */
/* One engine per GPU (twr_engine_cfg.rank / world); envs shard by rank with no data-path collective (the reference maps
 * episodes over rayon threads, rust/src/collector/ppo.rs:119-123).  NCCL carries the two per-iteration exchanges:
 * the trainer rank's weights to every engine (replaces rebuilding nn.Policy on every worker,
 * src/twisterl/rl/algorithm.py:91-93,112) and the sum of the collect statistics the trainer logs (:124-141).
 * NCCL is bound at run time (libnccl.so.2 or $TWISTERL_B200_NCCL_LIB); without it these return TWR_ERR_UNSUPPORTED. */
#define TWR_COMM_ID_BYTES 128   /* sizeof(ncclUniqueId) */
#define TWR_COMM_MAX_STATS 16
typedef enum { TWR_REDUCE_SUM = 0, TWR_REDUCE_MAX = 1 } twr_reduce_op;
/* NCCL version code (e.g. 22809), 0 when NCCL cannot be loaded */
int  twr_comm_version(void);
/* rank 0: creates the id every rank passes to twr_comm_init (the host distributes the bytes: file, env, MPI, TCP store) */
int  twr_comm_unique_id(uint8_t* id /* [TWR_COMM_ID_BYTES] */);
/* collective over the `world` engines of the job (ncclCommInitRank with this engine's rank) */
int  twr_comm_init(twr_engine* e, const uint8_t* id);
void twr_comm_destroy(twr_engine* e);
/* ncclBroadcast of rank `root`'s fp32 parameter blob into policy `p` of every engine (same shapes everywhere), on the
 * engine stream, then the in-place operand refresh of twr_policy_update_from_device.  world == 1: refresh only. */
int  twr_broadcast_weights(twr_engine* e, twr_policy* p, int32_t root);
/* in-place all-reduce of n <= TWR_COMM_MAX_STATS host doubles (episodes, successes, reward sum, records, ...);
 * returns after the reduced values are in `stats`.  world == 1: no-op. */
int  twr_allreduce_stats(twr_engine* e, double* stats, int32_t n, int32_t op /* twr_reduce_op */);
/* Collective over the `world` engines: every rank has just finished a device-resident collect (twr_ppo_collect or
 * twr_az_collect) of the same shape; rank `root` receives all of them, merged in the order ONE collect of
 * world * num_episodes episodes lays out ([last, 0, 1, ..., n-2], collector/collector.rs:40-46).  On root `out` (and what
 * twr_collected_to_host / the next twr_collected query return) describes the merged result; on the other ranks `out` is
 * their own result, unchanged.  world == 1: returns the local result, needs no communicator.
 * Every rank first all-gathers a small header and reaches the same verdict before any record moves: TWR_ERR_STATE on every
 * rank when one holds no device-resident result (a failed or missing collect, a pipelined twr_ppo_collect_host of several
 * sub-batches, a root that already holds a gathered result), TWR_ERR_INVALID when the ranks' env specs, shapes,
 * num_episodes, seeds, precisions, collect ids or roots differ.  The merged buffers are engine-owned (grow-only) and stay
 * valid until the next gather or destroy; NCCL p2p sends / receives carry the records on the engine stream, and the call
 * returns once root's result is complete.  TWR_ERR_UNSUPPORTED when libnccl lacks ncclSend / ncclRecv / ncclAllGather.
 * A rank's local failure before the exchange travels in its header and is returned by every rank; a CUDA or NCCL failure
 * inside the collectives themselves can, as with any NCCL collective, leave the peers waiting. */
int  twr_gather_collected(twr_engine* e, int32_t root, twr_collected* out);

/* Parity API: twr_mcts_probs plus, per env and simulation, the leaf the UCB descent ended on and the node the value was
 * backed up from, as tree-local node indices in expansion order: trace [n_sims][n][2].  tests/ use it to find the first
 * simulation in which the device search and the oracle's part ways (and hold that one to a near-tie). */
int  twr_debug_mcts_trace(twr_engine* e, const twr_policy* p, twr_envs* v, int32_t n_sims, float C, int32_t max_expand_depth,
                          uint32_t env_id_base, uint32_t collect_id, int32_t t, float* probs, int32_t* visits, int32_t* trace);

/* pinned host memory helpers (cudaHostAlloc / cudaFreeHost) for the e2e path */
int  twr_host_alloc(void** ptr, int64_t bytes);
void twr_host_free(void* ptr);

/* device time in ms of the last collect's forward kernels / all its kernels (CUDA events on
 * the engine stream); used by bench.py for the roofline line */
int  twr_engine_set_timing(twr_engine* e, int32_t enabled);
int  twr_engine_last_timing(const twr_engine* e, float* forward_ms, float* total_ms, int64_t* forward_launches);

#ifdef __cplusplus
}
#endif
#endif /* TWISTERL_B200_H */
