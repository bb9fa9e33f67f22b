/*
 * twr_oracle.h -- CPU restatement of the twisteRL Rust data-collection path.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it.  The shipped engine
 * (twisterl_b200/) never links, imports or calls anything in this directory.
 *
 * Parity status: PINNED against the reference's own known-answer vectors (SURVEY.md
 * section 8c): Puzzle 2x2 unit tests, the 35- and 123-move notebook replays with every
 * intermediate board, the grid_world notebook replay, the Linear / EmbeddingBag / argmax /
 * merge-order unit tests, and logits/values of the reference's own torch BasicPolicy run
 * in the build container on the shipped ppo_puzzle15_v1.pt weights (tests/golden/).
 * RNG-dependent results (scrambles, twist picks, sampled actions) are "parity unpinned"
 * against the Rust binary by construction: the reference draws from an OS-seeded
 * thread_rng() that its API cannot seed.  They are pinned oracle<->GPU instead, through the
 * shared counter-based Philox4x32-10 stream declared below.
 *
 * Every function cites the reference file:line it restates (paths relative to the
 * reference checkout).
 */
#ifndef TWR_ORACLE_H
#define TWR_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORC_MAX_CELLS 64
#define ORC_MAX_LAYERS 8

enum { ORC_ENV_PUZZLE = 0, ORC_ENV_GRIDWORLD = 1 };

/* RNG stream kinds (counter word 2).  Shared, bit for bit, with the CUDA engine. */
enum { ORC_RNG_RESET = 0, ORC_RNG_PERM = 1, ORC_RNG_SAMPLE = 2, ORC_RNG_SOLVE = 3, ORC_RNG_MCTS = 4, ORC_RNG_AZ_ACT = 5 };

/* Philox4x32-10 (Salmon et al., SC'11).  counter = (env_id, index, kind, collect_id),
 * key = (seed_lo, seed_hi). */
void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* u32 -> f32 in [0,1) with 24 bits: what rand 0.8.5 `rng.gen::<f32>()` produces
 * (reference call site rust/src/nn/policy.rs:171). */
float orc_u32_to_unit_f32(uint32_t w);

typedef struct {
    int32_t kind;        /* ORC_ENV_* */
    int32_t width, height;
    int32_t difficulty;
    int32_t depth_slope; /* puzzle only */
    int32_t max_depth;   /* puzzle: max_depth ; grid_world: max_steps */
} orc_env_spec;

typedef struct {
    orc_env_spec spec;
    /* Puzzle (rust/src/envs/puzzle.rs:20-30) */
    int64_t cells[ORC_MAX_CELLS];
    int32_t zx, zy;
    int64_t depth;
    /* GridWorld (examples/grid_world/src/lib.rs:10-21) */
    int32_t ax, ay, gx, gy, tx, ty;
    int64_t steps_left;
} orc_env;

void    orc_env_init(orc_env* e, const orc_env_spec* spec);
int32_t orc_env_num_actions(const orc_env* e);
int32_t orc_env_num_cells(const orc_env* e);
void    orc_env_set_difficulty(orc_env* e, int32_t d);
int32_t orc_env_get_difficulty(const orc_env* e);
void    orc_env_set_state(orc_env* e, const int64_t* state, int32_t n);
/* reset with the shared Philox stream: draws come from (env_id, *, ORC_RNG_RESET, collect_id) */
void    orc_env_reset(orc_env* e, uint64_t seed, uint32_t env_id, uint32_t collect_id);
void    orc_env_step(orc_env* e, int32_t action);
void    orc_env_masks(const orc_env* e, uint8_t* masks /* [num_actions] */);
int32_t orc_env_is_final(const orc_env* e);
int32_t orc_env_success(const orc_env* e);
float   orc_env_reward(const orc_env* e);
void    orc_env_observe(const orc_env* e, int32_t* obs /* [num_cells] */);
void    orc_env_get_state(const orc_env* e, int64_t* board /* [num_cells] */);

/* ---- policy (rust/src/nn/layers.rs, modules.rs, policy.rs) ---- */
typedef struct orc_policy orc_policy;
enum { ORC_NET_COMMON = 0, ORC_NET_ACTION = 1, ORC_NET_VALUE = 2 };

orc_policy* orc_policy_new(void);
void        orc_policy_free(orc_policy* p);
/* vectors[obs_idx][emb] row-major (what embeddingbag_to_rust passes), bias[bias_len] */
int orc_policy_set_embedding(orc_policy* p, const float* vectors, int32_t n_vectors, int32_t vec_len,
                             const float* bias, int32_t bias_len, int32_t apply_relu,
                             const int32_t* obs_shape, int32_t obs_shape_len, int32_t conv_dim);
/* weights_vector = W.T.flatten(): data[i*out + o] == W[o][i] (column-major out x in, layers.rs:26) */
int orc_policy_add_linear(orc_policy* p, int32_t which, const float* weights_vector, int32_t n_weights,
                          const float* bias, int32_t out, int32_t apply_relu);
int orc_policy_set_perms(orc_policy* p, const int32_t* obs_perms, const int32_t* act_perms,
                         int32_t n_perms, int32_t obs_size, int32_t num_actions);
int32_t orc_policy_n_perms(const orc_policy* p);

/* perm < 0 == None.  logits has num_actions entries (size of the action head). */
int32_t orc_policy_raw_predict(const orc_policy* p, const int32_t* obs, int32_t n_obs, int32_t perm,
                               float* logits, float* value);
int32_t orc_policy_forward(const orc_policy* p, const int32_t* obs, int32_t n_obs, const uint8_t* masks,
                           int32_t perm, float* masked_logits, float* value);
int32_t orc_policy_predict(const orc_policy* p, const int32_t* obs, int32_t n_obs, const uint8_t* masks,
                           int32_t perm, float* probs, float* value);
int32_t orc_policy_full_predict(const orc_policy* p, const int32_t* obs, int32_t n_obs, const uint8_t* masks,
                                float* probs, float* value);

int32_t orc_argmax(const float* v, int32_t n);
/* Gumbel-max with caller-supplied uniforms in [0,1) (policy.rs:169-172) */
int32_t orc_sample_from_logits(const float* logits, int32_t n, const float* uniforms);
/* per-episode GAE (collector/ppo.rs:82-92) */
void orc_gae(const float* rewards, const float* values, int32_t n, float gamma, float lambda,
             float* advs, float* rets);
/* merge order of collector.rs:40-46: writes the episode index placed at each slot */
void orc_merge_order(int32_t num_episodes, int32_t* order);

typedef struct {
    int64_t  n_records;
    int32_t  num_episodes, n_cells, num_actions;
    int32_t* ep_len;   /* [num_episodes] by episode id (NOT merged order) */
    int32_t* obs;      /* [R][n_cells] sparse one-hot indices */
    float*   logits;   /* [R][num_actions] masked logits */
    float*   values;   /* [R] */
    float*   rewards;  /* [R] */
    float*   advs;     /* [R] */
    float*   rets;     /* [R] */
    int32_t* actions;  /* [R] */
    int32_t* perms;    /* [R], -1 == None */
} orc_collected;

/* PPOCollector::collect (collector/ppo.rs:108-126) with episode e using Philox env_id =
 * env_id_base + e.  Output is in the reference's merged order.  Returns 0 on success. */
int  orc_ppo_collect(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes,
                     float gamma, float lambda, uint64_t seed, uint32_t collect_id,
                     uint32_t env_id_base, int32_t num_threads, orc_collected* out);
void orc_collected_free(orc_collected* c);

/* ---- solve / evaluate (rust/src/rl/solve.rs, rust/src/rl/evaluate.rs), num_mcts_searches == 0 ---- */
/* single_solve (solve.rs:17-71) on `env` (modified in place) with Philox stream id `stream_id`:
 * twist pick (stream_id, t, PERM), weighted draw (stream_id, t, SOLVE).  actions may be NULL. */
void orc_single_solve(orc_env* env, const orc_policy* p, int32_t deterministic, uint64_t seed, uint32_t collect_id,
                      uint32_t stream_id, float* success, float* total, int32_t* actions, int32_t* n_actions);
/* solve (solve.rs:73-101): best of num_searches from a copy of `env`; search s uses stream id0 + s */
void orc_solve(const orc_env* env, const orc_policy* p, int32_t deterministic, int32_t num_searches, uint64_t seed,
               uint32_t collect_id, uint32_t id0, float* success, float* total, int32_t* actions, int32_t* n_actions);
/* evaluate (evaluate.rs:22-89): episode ep resets from stream (reset_base + ep) and searches with ids
 * search_base + ep*num_searches + s.  best_success/best_total: [num_episodes] or NULL. */
void orc_evaluate(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes, int32_t deterministic,
                  int32_t num_searches, uint64_t seed, uint32_t collect_id, uint32_t reset_base, uint32_t search_base,
                  float* success_rate, float* mean_reward, float* best_success, float* best_total);

/* the same three with num_mcts_searches > 0: the action distribution of every step is predict_probs_mcts of the
 * current state (solve.rs:40-47) on Philox stream (stream_id, t) */
void orc_single_solve_mcts(orc_env* env, const orc_policy* p, int32_t deterministic, int32_t n_mcts, float C,
                           int32_t max_expand_depth, uint64_t seed, uint32_t collect_id, uint32_t stream_id,
                           float* success, float* total, int32_t* actions, int32_t* n_actions);
void orc_solve_mcts(const orc_env* env, const orc_policy* p, int32_t deterministic, int32_t num_searches, int32_t n_mcts,
                    float C, int32_t max_expand_depth, uint64_t seed, uint32_t collect_id, uint32_t id0, float* success,
                    float* total, int32_t* actions, int32_t* n_actions);
void orc_evaluate_mcts(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes, int32_t deterministic,
                       int32_t num_searches, int32_t n_mcts, float C, int32_t max_expand_depth, uint64_t seed,
                       uint32_t collect_id, uint32_t reset_base, uint32_t search_base, float* success_rate,
                       float* mean_reward, float* best_success, float* best_total);

/* the same evaluation plus, per episode, the smallest decision margin met by any of its rollouts (argmax gap, weighted-draw
 * distance to a bin edge, UCB gap inside MCTS): an episode whose margin is tiny may legitimately differ between two
 * implementations whose logits differ in the last bits */
void orc_evaluate_margins(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes, int32_t deterministic,
                          int32_t num_searches, int32_t n_mcts, float C, int32_t max_expand_depth, uint64_t seed,
                          uint32_t collect_id, uint32_t reset_base, uint32_t search_base, float* best_success,
                          float* best_total, float* min_margin);

/* ---- AlphaZero path (rust/src/rl/search.rs, rust/src/rl/tree.rs, rust/src/collector/az.rs) ---- */
/* predict_probs_mcts (search.rs:104-189) from `env`; the child draw of simulation `sim`, expansion round d uses
 * Philox (stream_id, (t*(n_sims+1)+sim)*max(1,max_expand_depth)+d, MCTS, collect_id).  visits may be NULL. */
void orc_mcts_probs(const orc_env* env, const orc_policy* p, int32_t n_sims, float C, int32_t max_expand_depth,
                    uint64_t seed, uint32_t collect_id, uint32_t stream_id, int32_t t, float* probs, int32_t* visits);
/* same search with a per-simulation trace [n_sims]: the leaf the UCB descent ended on, the node the value was backed up
 * from, the simulation's smallest decision margin (UCB best - second best; child-draw distance to a bin edge) and the
 * length of its backup path (nodes from the root to the backed-up node, both included).  Any trace pointer may be NULL. */
void orc_mcts_trace(const orc_env* env, const orc_policy* p, int32_t n_sims, float C, int32_t max_expand_depth,
                    uint64_t seed, uint32_t collect_id, uint32_t stream_id, int32_t t, float* probs, int32_t* visits,
                    int32_t* trace_leaf, int32_t* trace_child, float* trace_margin, int32_t* trace_len);
typedef struct {
    int64_t n_records; int32_t num_episodes, n_cells, num_actions;
    int32_t* ep_len; int32_t* obs; float* probs; float* rewards; int32_t* actions; float* remaining_values;
} orc_az_collected;
/* AZCollector::collect (az.rs:112-130), merged order; the action draw of step t uses (id, t, AZ_ACT, cid) */
int  orc_az_collect(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes, int32_t n_sims, float C,
                    int32_t max_expand_depth, uint64_t seed, uint32_t collect_id, uint32_t env_id_base,
                    orc_az_collected* out);
void orc_az_collected_free(orc_az_collected* c);

#ifdef __cplusplus
}
#endif
#endif
