/*
 * twr_oracle.c -- CPU restatement of the twisteRL Rust data-collection path (see twr_oracle.h).
 *
 * TEST INFRASTRUCTURE ONLY: the product path never calls into this file.
 * Compile with -ffp-contract=off: the Rust reference does not fuse multiply-adds.
 *
 * All citations are `path:line` inside the reference checkout.
 */
#include "twr_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ RNG --- */

static inline void philox_round(uint32_t c[4], const uint32_t k[2]) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k[0];
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k[1];
    const uint32_t n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}

void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
    uint32_t k[2] = {key[0], key[1]};
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k);
        k[0] += 0x9E3779B9u;
        k[1] += 0xBB67AE85u;
    }
    memcpy(out, c, sizeof(c));
}

float orc_u32_to_unit_f32(uint32_t w) {
    /* rand 0.8.5 Standard for f32: 24 high bits * 2^-24, in [0,1) (called at nn/policy.rs:171) */
    return (float)(w >> 8) * (1.0f / 16777216.0f);
}

static inline uint32_t mulhi32(uint32_t a, uint32_t n) { return (uint32_t)(((uint64_t)a * n) >> 32); }

typedef struct {
    uint32_t key[2];
    uint32_t env_id, kind, collect_id;
    uint32_t next;  /* index of the next u32 in this stream */
    uint32_t buf[4];
    uint32_t buf_block;
    int have;
} rng_stream;

static void rng_open(rng_stream* s, uint64_t seed, uint32_t env_id, uint32_t kind, uint32_t collect_id) {
    s->key[0] = (uint32_t)seed; s->key[1] = (uint32_t)(seed >> 32);
    s->env_id = env_id; s->kind = kind; s->collect_id = collect_id;
    s->next = 0; s->have = 0; s->buf_block = 0;
}

static uint32_t rng_u32(rng_stream* s) {
    const uint32_t block = s->next >> 2;
    if (!s->have || block != s->buf_block) {
        const uint32_t ctr[4] = {s->env_id, block, s->kind, s->collect_id};
        orc_philox4x32_10(ctr, s->key, s->buf);
        s->buf_block = block; s->have = 1;
    }
    return s->buf[s->next++ & 3];
}

/* ------------------------------------------------------------------ envs --- */

void orc_env_init(orc_env* e, const orc_env_spec* spec) {
    memset(e, 0, sizeof(*e));
    e->spec = *spec;
    if (spec->kind == ORC_ENV_PUZZLE) {
        /* Puzzle::new, envs/puzzle.rs:34-42: identity board, blank (0,0), depth 1 */
        const int n = spec->width * spec->height;
        for (int i = 0; i < n; ++i) e->cells[i] = i;
        e->zx = 0; e->zy = 0; e->depth = 1;
    } else {
        /* GridWorld::new, examples/grid_world/src/lib.rs:23-41 */
        const int cap = spec->width + spec->height;
        e->spec.difficulty = spec->difficulty < cap ? spec->difficulty : cap;
        e->steps_left = spec->max_depth;
    }
}

int32_t orc_env_num_actions(const orc_env* e) { (void)e; return 4; } /* puzzle.rs:90-92, lib.rs:88 */
int32_t orc_env_num_cells(const orc_env* e) { return e->spec.width * e->spec.height; }

void orc_env_set_difficulty(orc_env* e, int32_t d) {
    if (e->spec.kind == ORC_ENV_PUZZLE) {
        e->spec.difficulty = d; /* puzzle.rs:99-101 */
    } else {
        const int cap = e->spec.width + e->spec.height; /* lib.rs:92-94 */
        e->spec.difficulty = d < cap ? d : cap;
    }
}
int32_t orc_env_get_difficulty(const orc_env* e) { return e->spec.difficulty; }

static int puzzle_solved(const orc_env* e) { /* puzzle.rs:44-50 */
    const int n = e->spec.width * e->spec.height;
    for (int i = 0; i < n; ++i) if (e->cells[i] != i) return 0;
    return 1;
}

void orc_env_set_state(orc_env* e, const int64_t* state, int32_t n) {
    const int W = e->spec.width;
    if (e->spec.kind == ORC_ENV_PUZZLE) {
        /* puzzle.rs:107-117 */
        for (int i = 0; i < n; ++i) e->cells[i] = state[i];
        e->depth = e->spec.max_depth;
        for (int i = 0; i < n; ++i) {
            if (state[i] == 0) { e->zx = i % W; e->zy = i / W; break; }
        }
    } else {
        /* lib.rs:100-112 */
        for (int i = 0; i < n; ++i) {
            if (state[i] == 1)      { e->ax = i % W; e->ay = i / W; }
            else if (state[i] == 2) { e->gx = i % W; e->gy = i / W; }
            else if (state[i] == 3) { e->tx = i % W; e->ty = i / W; }
        }
        e->steps_left = e->spec.max_depth;
    }
}

void orc_env_step(orc_env* e, int32_t action) {
    const int W = e->spec.width, H = e->spec.height;
    if (e->spec.kind == ORC_ENV_PUZZLE) {
        /* puzzle.rs:135-160: blank moves left/up/right/down; illegal = no-op; depth always -1 */
        int zx = e->zx, zy = e->zy, nx = zx, ny = zy, ok = 0;
        if (action == 0 && zx > 0)          { nx = zx - 1; ok = 1; }
        else if (action == 1 && zy > 0)     { ny = zy - 1; ok = 1; }
        else if (action == 2 && zx < W - 1) { nx = zx + 1; ok = 1; }
        else if (action == 3 && zy < H - 1) { ny = zy + 1; ok = 1; }
        if (ok) {
            e->cells[zy * W + zx] = e->cells[ny * W + nx];
            e->cells[ny * W + nx] = 0;
            e->zx = nx; e->zy = ny;
        }
        if (e->depth > 0) e->depth -= 1; /* saturating_sub, puzzle.rs:159 */
    } else {
        /* lib.rs:127-136: 0 up (y-1), 1 down (y+1), 2 left (x-1), 3 right (x+1) */
        if (action == 0 && e->ay > 0) e->ay -= 1;
        else if (action == 1 && e->ay + 1 < H) e->ay += 1;
        else if (action == 2 && e->ax > 0) e->ax -= 1;
        else if (action == 3 && e->ax + 1 < W) e->ax += 1;
        if (e->steps_left > 0) e->steps_left -= 1;
    }
}

void orc_env_reset(orc_env* e, uint64_t seed, uint32_t env_id, uint32_t collect_id) {
    const int W = e->spec.width, H = e->spec.height;
    rng_stream s;
    rng_open(&s, seed, env_id, ORC_RNG_RESET, collect_id);
    if (e->spec.kind == ORC_ENV_PUZZLE) {
        /* puzzle.rs:119-133.  The reference draws Uniform(0,4) `difficulty` times (illegal
         * draws are no-ops through step()).  Shared stream: draw j = 2-bit field (j%16) of
         * word (j%64)/16 of Philox block j/64. */
        const int n = W * H;
        for (int i = 0; i < n; ++i) e->cells[i] = i;
        e->zx = 0; e->zy = 0;
        uint32_t w = 0;
        for (int j = 0; j < e->spec.difficulty; ++j) {
            if ((j & 15) == 0) w = rng_u32(&s);
            orc_env_step(e, (int32_t)((w >> (2 * (j & 15))) & 3u));
        }
        e->depth = (int64_t)e->spec.depth_slope * e->spec.difficulty;
    } else {
        /* lib.rs:114-125, with random_pos :43-48 and random_pos_near :50-65 */
        const uint32_t n = (uint32_t)(W * H);
        uint32_t a = mulhi32(rng_u32(&s), n);
        e->ax = (int)(a % W); e->ay = (int)(a / W);
        int cx[ORC_MAX_CELLS], cy[ORC_MAX_CELLS], nc = 0;
        for (int x = 0; x < W; ++x)
            for (int y = 0; y < H; ++y) {
                const int d = abs(x - e->ax) + abs(y - e->ay);
                if (d <= e->spec.difficulty) { cx[nc] = x; cy[nc] = y; ++nc; }
            }
        if (nc < 2) abort(); /* difficulty 0 would spin forever in the reference; reject */
        for (;;) {
            const uint32_t k = mulhi32(rng_u32(&s), (uint32_t)nc);
            if (cx[k] != e->ax || cy[k] != e->ay) { e->gx = cx[k]; e->gy = cy[k]; break; }
        }
        for (;;) {
            const uint32_t t = mulhi32(rng_u32(&s), n);
            const int tx = (int)(t % W), ty = (int)(t / W);
            if ((tx != e->ax || ty != e->ay) && (tx != e->gx || ty != e->gy)) { e->tx = tx; e->ty = ty; break; }
        }
        e->steps_left = e->spec.max_depth;
    }
}

static int gw_at_goal(const orc_env* e) { return e->ax == e->gx && e->ay == e->gy; }
static int gw_at_trap(const orc_env* e) { return e->ax == e->tx && e->ay == e->ty; }

void orc_env_masks(const orc_env* e, uint8_t* m) {
    const int W = e->spec.width, H = e->spec.height;
    if (e->spec.kind == ORC_ENV_PUZZLE) { /* puzzle.rs:162-165 */
        m[0] = e->zx > 0; m[1] = e->zy > 0; m[2] = e->zx < W - 1; m[3] = e->zy < H - 1;
    } else { /* lib.rs:138-145 */
        m[0] = e->ay > 0; m[1] = e->ay + 1 < H; m[2] = e->ax > 0; m[3] = e->ax + 1 < W;
    }
}

int32_t orc_env_is_final(const orc_env* e) {
    if (e->spec.kind == ORC_ENV_PUZZLE) return e->depth == 0 || puzzle_solved(e); /* puzzle.rs:167-169 */
    return e->steps_left == 0 || gw_at_goal(e) || gw_at_trap(e);                   /* lib.rs:147-149 */
}

int32_t orc_env_success(const orc_env* e) {
    return e->spec.kind == ORC_ENV_PUZZLE ? puzzle_solved(e) : gw_at_goal(e);
}

float orc_env_reward(const orc_env* e) {
    if (e->spec.kind == ORC_ENV_PUZZLE) { /* puzzle.rs:171-177 */
        if (puzzle_solved(e)) return 1.0f;
        if (e->depth == 0) return -0.5f;
        return -0.5f / (float)e->spec.max_depth;
    }
    /* lib.rs:151-155 */
    if (gw_at_goal(e)) return 1.0f;
    if (gw_at_trap(e)) return -0.5f;
    if (e->steps_left == 0) return -0.5f;
    return -0.5f / (float)e->steps_left;
}

void orc_env_get_state(const orc_env* e, int64_t* board) {
    const int W = e->spec.width, n = e->spec.width * e->spec.height;
    if (e->spec.kind == ORC_ENV_PUZZLE) {
        for (int i = 0; i < n; ++i) board[i] = e->cells[i];
    } else { /* lib.rs:74-81: goal, then trap, then agent (agent overwrites) */
        for (int i = 0; i < n; ++i) board[i] = 0;
        board[e->gy * W + e->gx] = 2;
        board[e->ty * W + e->tx] = 3;
        board[e->ay * W + e->ax] = 1;
    }
}

void orc_env_observe(const orc_env* e, int32_t* obs) {
    /* puzzle.rs:183-185 / lib.rs:161-163: obs[i] = i*(H*W) + board[i] */
    int64_t board[ORC_MAX_CELLS];
    const int n = e->spec.width * e->spec.height;
    orc_env_get_state(e, board);
    for (int i = 0; i < n; ++i) obs[i] = (int32_t)(i * n + board[i]);
}

/* ---------------------------------------------------------------- policy --- */

typedef struct {
    int in, out, relu;
    float* w; /* data[i*out + o] == W[o][i]: nalgebra DMatrix::from_vec column-major, layers.rs:26 */
    float* b;
} lin_t;

struct orc_policy {
    int n_vectors, vec_len, bias_len, emb_relu;
    float* vectors; float* emb_bias;
    int obs_shape[2], obs_shape_len, conv_dim;
    int n_layers[3];
    lin_t layers[3][ORC_MAX_LAYERS];
    int n_perms, obs_size, num_actions;
    int32_t* obs_perms; int32_t* act_perms;
};

orc_policy* orc_policy_new(void) { return (orc_policy*)calloc(1, sizeof(orc_policy)); }

void orc_policy_free(orc_policy* p) {
    if (!p) return;
    free(p->vectors); free(p->emb_bias); free(p->obs_perms); free(p->act_perms);
    for (int n = 0; n < 3; ++n)
        for (int l = 0; l < p->n_layers[n]; ++l) { free(p->layers[n][l].w); free(p->layers[n][l].b); }
    free(p);
}

static float* dup_f32(const float* src, size_t n) {
    float* d = (float*)malloc((n ? n : 1) * sizeof(float));
    if (n) memcpy(d, src, n * sizeof(float));
    return d;
}

int orc_policy_set_embedding(orc_policy* p, const float* vectors, int32_t n_vectors, int32_t vec_len,
                             const float* bias, int32_t bias_len, int32_t apply_relu,
                             const int32_t* obs_shape, int32_t obs_shape_len, int32_t conv_dim) {
    if (obs_shape_len < 1 || obs_shape_len > 2) return -1;
    free(p->vectors); free(p->emb_bias);
    p->vectors = dup_f32(vectors, (size_t)n_vectors * vec_len);
    p->emb_bias = dup_f32(bias, (size_t)bias_len);
    p->n_vectors = n_vectors; p->vec_len = vec_len; p->bias_len = bias_len; p->emb_relu = apply_relu;
    p->obs_shape_len = obs_shape_len; p->conv_dim = conv_dim;
    for (int i = 0; i < obs_shape_len; ++i) p->obs_shape[i] = obs_shape[i];
    return 0;
}

int orc_policy_add_linear(orc_policy* p, int32_t which, const float* wv, int32_t n_weights,
                          const float* bias, int32_t out, int32_t apply_relu) {
    if (which < 0 || which > 2 || p->n_layers[which] >= ORC_MAX_LAYERS || out <= 0) return -1;
    lin_t* l = &p->layers[which][p->n_layers[which]++];
    l->out = out; l->in = n_weights / out; l->relu = apply_relu; /* layers.rs:26 */
    l->w = dup_f32(wv, (size_t)n_weights);
    l->b = dup_f32(bias, (size_t)out);
    return 0;
}

int orc_policy_set_perms(orc_policy* p, const int32_t* obs_perms, const int32_t* act_perms,
                         int32_t n_perms, int32_t obs_size, int32_t num_actions) {
    free(p->obs_perms); free(p->act_perms);
    p->obs_perms = NULL; p->act_perms = NULL;
    p->n_perms = n_perms; p->obs_size = obs_size; p->num_actions = num_actions;
    if (n_perms > 0) {
        p->obs_perms = (int32_t*)malloc(sizeof(int32_t) * (size_t)n_perms * obs_size);
        p->act_perms = (int32_t*)malloc(sizeof(int32_t) * (size_t)n_perms * num_actions);
        memcpy(p->obs_perms, obs_perms, sizeof(int32_t) * (size_t)n_perms * obs_size);
        memcpy(p->act_perms, act_perms, sizeof(int32_t) * (size_t)n_perms * num_actions);
    }
    return 0;
}

int32_t orc_policy_n_perms(const orc_policy* p) { return p->n_perms; }

static inline float relu_f(float x) { return x > 0.0f ? x : 0.0f; } /* layers.rs:89-91 */

/* Linear::forward, layers.rs:31-37: (W * x) + b, then optional ReLU.  nalgebra's gemv on a
 * column-major matrix accumulates one column (axpy) at a time: y = x0*col0; y += xj*colj. */
static void linear_forward(const lin_t* l, const float* x, float* y) {
    const int out = l->out;
    for (int o = 0; o < out; ++o) y[o] = 0.0f;
    for (int j = 0; j < l->in; ++j) {
        const float xj = x[j];
        const float* col = l->w + (size_t)j * out;
        for (int o = 0; o < out; ++o) y[o] += col[o] * xj;
    }
    for (int o = 0; o < out; ++o) y[o] += l->b[o];
    if (l->relu) for (int o = 0; o < out; ++o) y[o] = relu_f(y[o]);
}

/* EmbeddingBag::forward, layers.rs:56-86 */
static void embedding_forward(const orc_policy* p, const int32_t* obs, int n_obs, float* out) {
    memcpy(out, p->emb_bias, sizeof(float) * (size_t)p->bias_len);
    const int v = p->vec_len;
    if (p->obs_shape_len == 1) {
        for (int k = 0; k < n_obs; ++k) {
            const float* row = p->vectors + (size_t)obs[k] * v;
            for (int f = 0; f < v; ++f) out[f] += row[f];
        }
    } else {
        for (int k = 0; k < n_obs; ++k) {
            int row = obs[k] / p->obs_shape[1];
            int col = obs[k] % p->obs_shape[1];
            if (p->conv_dim == 1) { int t = row; row = col; col = t; }
            const float* r = p->vectors + (size_t)row * v;
            float* o = out + (size_t)col * v;
            for (int f = 0; f < v; ++f) o[f] += r[f];
        }
    }
    if (p->emb_relu) for (int f = 0; f < p->bias_len; ++f) out[f] = relu_f(out[f]);
}

#define ORC_MAX_WIDTH 8192

static int seq_forward(const lin_t* layers, int n, const float* x, int x_len, float* y /* out */, int* y_len) {
    /* Sequential::forward, modules.rs:28-34 */
    float a[ORC_MAX_WIDTH], b[ORC_MAX_WIDTH];
    const float* cur = x; int cur_len = x_len;
    float* bufs[2] = {a, b};
    for (int l = 0; l < n; ++l) {
        if (layers[l].in != cur_len || layers[l].out > ORC_MAX_WIDTH) return -1;
        linear_forward(&layers[l], cur, bufs[l & 1]);
        cur = bufs[l & 1]; cur_len = layers[l].out;
    }
    memcpy(y, cur, sizeof(float) * (size_t)cur_len);
    *y_len = cur_len;
    return 0;
}

int32_t orc_policy_raw_predict(const orc_policy* p, const int32_t* obs_in, int32_t n_obs, int32_t perm,
                               float* logits, float* value) {
    /* Policy::_raw_predict, nn/policy.rs:79-100 */
    int32_t obs[ORC_MAX_CELLS * 16];
    if (n_obs > (int)(sizeof(obs) / sizeof(obs[0])) || p->bias_len > ORC_MAX_WIDTH) return -1;
    for (int k = 0; k < n_obs; ++k)
        obs[k] = perm >= 0 ? p->obs_perms[(size_t)perm * p->obs_size + obs_in[k]] : obs_in[k];

    float emb[ORC_MAX_WIDTH], common[ORC_MAX_WIDTH], head[ORC_MAX_WIDTH];
    embedding_forward(p, obs, n_obs, emb);
    int clen = 0, hlen = 0;
    if (seq_forward(p->layers[ORC_NET_COMMON], p->n_layers[ORC_NET_COMMON], emb, p->bias_len, common, &clen)) return -1;

    if (seq_forward(p->layers[ORC_NET_VALUE], p->n_layers[ORC_NET_VALUE], common, clen, head, &hlen)) return -1;
    float v = 0.0f;
    for (int i = 0; i < hlen; ++i) v += head[i]; /* .sum(), policy.rs:89 */
    *value = v;

    if (seq_forward(p->layers[ORC_NET_ACTION], p->n_layers[ORC_NET_ACTION], common, clen, head, &hlen)) return -1;
    if (perm >= 0) {
        /* policy.rs:95-97: out[i] = logits[act_perms[pi][i]] */
        for (int i = 0; i < p->num_actions; ++i) logits[i] = head[p->act_perms[(size_t)perm * p->num_actions + i]];
        return p->num_actions;
    }
    memcpy(logits, head, sizeof(float) * (size_t)hlen);
    return hlen;
}

int32_t orc_policy_forward(const orc_policy* p, const int32_t* obs, int32_t n_obs, const uint8_t* masks,
                           int32_t perm, float* masked_logits, float* value) {
    /* Policy::forward_with_perm, nn/policy.rs:56-65 (perm chosen by the caller) */
    const int n = orc_policy_raw_predict(p, obs, n_obs, perm, masked_logits, value);
    for (int i = 0; i < n; ++i) if (!masks[i]) masked_logits[i] = -1e10f;
    return n;
}

static void masked_exp_normalise(float* l, int n, const uint8_t* masks) {
    /* nn/policy.rs:43-47 and :118-124: exp without max-subtraction, / (sum + 1e-6) */
    float s = 0.0f;
    for (int i = 0; i < n; ++i) { l[i] = masks[i] ? expf(l[i]) : 0.0f; s += l[i]; }
    for (int i = 0; i < n; ++i) l[i] = l[i] / (s + 0.000001f);
}

int32_t orc_policy_predict(const orc_policy* p, const int32_t* obs, int32_t n_obs, const uint8_t* masks,
                           int32_t perm, float* probs, float* value) {
    /* Policy::predict_with_perm, nn/policy.rs:39-49 */
    const int n = orc_policy_forward(p, obs, n_obs, masks, perm, probs, value);
    if (n < 0) return n;
    masked_exp_normalise(probs, n, masks);
    return n;
}

int32_t orc_policy_full_predict(const orc_policy* p, const int32_t* obs, int32_t n_obs, const uint8_t* masks,
                                float* probs, float* value) {
    /* Policy::full_predict, nn/policy.rs:102-126 */
    if (p->n_perms == 0) return orc_policy_predict(p, obs, n_obs, masks, -1, probs, value);
    const int n = p->num_actions;
    const float np = (float)p->n_perms;
    float v = 0.0f, tmp[256];
    for (int i = 0; i < n; ++i) probs[i] = 0.0f;
    for (int pi = 0; pi < p->n_perms; ++pi) {
        float vi;
        if (orc_policy_raw_predict(p, obs, n_obs, pi, tmp, &vi) < 0) return -1;
        v += vi / np;
        for (int i = 0; i < n; ++i) probs[i] += tmp[i] / np;
    }
    masked_exp_normalise(probs, n, masks);
    *value = v;
    return n;
}

int32_t orc_argmax(const float* v, int32_t n) {
    /* nn/policy.rs:130-151: strict '>', first max wins, a NaN never replaces the incumbent */
    if (n <= 0) return 0;
    int best = 0; float bv = v[0];
    for (int i = 1; i < n; ++i) if (v[i] > bv) { bv = v[i]; best = i; }
    return best;
}

int32_t orc_sample_from_logits(const float* logits, int32_t n, const float* u) {
    /* nn/policy.rs:169-172: argmax_i( l_i - ln(|ln(u_i)|) ) */
    float g[256];
    for (int i = 0; i < n; ++i) g[i] = logits[i] - logf(fabsf(logf(u[i])));
    return orc_argmax(g, n);
}

void orc_gae(const float* r, const float* v, int32_t n, float gamma, float lambda, float* adv, float* ret) {
    /* collector/ppo.rs:82-92, evaluation order as written */
    if (n <= 0) return;
    adv[n - 1] = r[n - 1] - v[n - 1];
    ret[n - 1] = r[n - 1];
    for (int t = n - 2; t >= 0; --t) {
        ret[t] = r[t] + gamma * (v[t + 1] + lambda * adv[t + 1]);
        adv[t] = ret[t] - v[t];
    }
}

void orc_merge_order(int32_t n, int32_t* order) {
    /* collector/collector.rs:40-46: pop() the last chunk, then append chunks 0..n-2 in order */
    if (n <= 0) return;
    order[0] = n - 1;
    for (int i = 0; i < n - 1; ++i) order[i + 1] = i;
}

/* ------------------------------------------------------------- collector --- */

typedef struct {
    int32_t n;
    int32_t* obs; float* logits; float* values; float* rewards; float* advs; float* rets;
    int32_t* actions; int32_t* perms;
} episode_t;

typedef struct {
    const orc_env_spec* spec; const orc_policy* p;
    int32_t num_episodes; float gamma, lambda; uint64_t seed; uint32_t collect_id, env_id_base;
    episode_t* eps;
    int next; pthread_mutex_t mu;
    int failed;
} job_t;

static int single_collect(const job_t* j, int ep, episode_t* out) {
    /* PPOCollector::single_collect, collector/ppo.rs:54-105 */
    orc_env env;
    orc_env_init(&env, j->spec);
    const uint32_t env_id = j->env_id_base + (uint32_t)ep;
    orc_env_reset(&env, j->seed, env_id, j->collect_id);
    const int nc = orc_env_num_cells(&env), na = orc_env_num_actions(&env);
    const uint32_t key[2] = {(uint32_t)j->seed, (uint32_t)(j->seed >> 32)};

    int cap = 64, n = 0;
    int32_t* obs = (int32_t*)malloc(sizeof(int32_t) * (size_t)cap * nc);
    float* logits = (float*)malloc(sizeof(float) * (size_t)cap * na);
    float* values = (float*)malloc(sizeof(float) * cap);
    float* rewards = (float*)malloc(sizeof(float) * cap);
    int32_t* actions = (int32_t*)malloc(sizeof(int32_t) * cap);
    int32_t* perms = (int32_t*)malloc(sizeof(int32_t) * cap);

    for (;;) {
        if (n == cap) {
            cap *= 2;
            obs = (int32_t*)realloc(obs, sizeof(int32_t) * (size_t)cap * nc);
            logits = (float*)realloc(logits, sizeof(float) * (size_t)cap * na);
            values = (float*)realloc(values, sizeof(float) * cap);
            rewards = (float*)realloc(rewards, sizeof(float) * cap);
            actions = (int32_t*)realloc(actions, sizeof(int32_t) * cap);
            perms = (int32_t*)realloc(perms, sizeof(int32_t) * cap);
        }
        /* get_step_data, collector/ppo.rs:41-52 */
        uint8_t masks[16];
        orc_env_observe(&env, obs + (size_t)n * nc);
        orc_env_masks(&env, masks);
        rewards[n] = orc_env_reward(&env);
        int perm = -1;
        if (j->p->n_perms > 0) { /* get_perm_id, nn/policy.rs:67-77 */
            const uint32_t ctr[4] = {env_id, (uint32_t)n, ORC_RNG_PERM, j->collect_id};
            uint32_t w[4];
            orc_philox4x32_10(ctr, key, w);
            perm = (int)mulhi32(w[0], (uint32_t)j->p->n_perms);
        }
        if (orc_policy_forward(j->p, obs + (size_t)n * nc, nc, masks, perm, logits + (size_t)n * na, &values[n]) != na) {
            free(obs); free(logits); free(values); free(rewards); free(actions); free(perms);
            return -1;
        }
        float u[16];
        for (int b = 0; b * 4 < na; ++b) {
            const uint32_t ctr[4] = {env_id, (uint32_t)n, ORC_RNG_SAMPLE + ((uint32_t)b << 8), j->collect_id};
            uint32_t w[4];
            orc_philox4x32_10(ctr, key, w);
            for (int i = 0; i < 4; ++i) u[b * 4 + i] = orc_u32_to_unit_f32(w[i]);
        }
        actions[n] = orc_sample_from_logits(logits + (size_t)n * na, na, u);
        perms[n] = perm;
        ++n;
        if (orc_env_is_final(&env)) break; /* ppo.rs:78: terminal state recorded, its action not applied */
        orc_env_step(&env, actions[n - 1]);
    }
    out->n = n; out->obs = obs; out->logits = logits; out->values = values; out->rewards = rewards;
    out->actions = actions; out->perms = perms;
    out->advs = (float*)malloc(sizeof(float) * n);
    out->rets = (float*)malloc(sizeof(float) * n);
    orc_gae(rewards, values, n, j->gamma, j->lambda, out->advs, out->rets);
    return 0;
}

static void* worker(void* arg) {
    job_t* j = (job_t*)arg;
    for (;;) {
        pthread_mutex_lock(&j->mu);
        const int ep = j->next < j->num_episodes ? j->next++ : -1;
        pthread_mutex_unlock(&j->mu);
        if (ep < 0) break;
        if (single_collect(j, ep, &j->eps[ep])) { j->failed = 1; break; }
    }
    return NULL;
}

int orc_ppo_collect(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes,
                    float gamma, float lambda, uint64_t seed, uint32_t collect_id,
                    uint32_t env_id_base, int32_t num_threads, orc_collected* out) {
    /* PPOCollector::collect, collector/ppo.rs:108-126; a fresh pool per call like ppo.rs:117 */
    memset(out, 0, sizeof(*out));
    if (num_episodes <= 0) return -1; /* merge() errors on zero chunks, collector.rs:41 */
    job_t j;
    memset(&j, 0, sizeof(j));
    j.spec = spec; j.p = p; j.num_episodes = num_episodes; j.gamma = gamma; j.lambda = lambda;
    j.seed = seed; j.collect_id = collect_id; j.env_id_base = env_id_base;
    j.eps = (episode_t*)calloc((size_t)num_episodes, sizeof(episode_t));
    pthread_mutex_init(&j.mu, NULL);
    if (num_threads <= 1) {
        worker(&j);
    } else {
        pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)num_threads);
        for (int t = 0; t < num_threads; ++t) pthread_create(&th[t], NULL, worker, &j);
        for (int t = 0; t < num_threads; ++t) pthread_join(th[t], NULL);
        free(th);
    }
    pthread_mutex_destroy(&j.mu);

    orc_env tmp; orc_env_init(&tmp, spec);
    const int nc = orc_env_num_cells(&tmp), na = orc_env_num_actions(&tmp);
    int64_t R = 0;
    for (int e = 0; e < num_episodes; ++e) R += j.eps[e].n;
    int rc = j.failed ? -1 : 0;
    if (!rc) {
        out->n_records = R; out->num_episodes = num_episodes; out->n_cells = nc; out->num_actions = na;
        out->ep_len = (int32_t*)malloc(sizeof(int32_t) * (size_t)num_episodes);
        out->obs = (int32_t*)malloc(sizeof(int32_t) * (size_t)R * nc);
        out->logits = (float*)malloc(sizeof(float) * (size_t)R * na);
        out->values = (float*)malloc(sizeof(float) * (size_t)R);
        out->rewards = (float*)malloc(sizeof(float) * (size_t)R);
        out->advs = (float*)malloc(sizeof(float) * (size_t)R);
        out->rets = (float*)malloc(sizeof(float) * (size_t)R);
        out->actions = (int32_t*)malloc(sizeof(int32_t) * (size_t)R);
        out->perms = (int32_t*)malloc(sizeof(int32_t) * (size_t)R);
        int32_t* order = (int32_t*)malloc(sizeof(int32_t) * (size_t)num_episodes);
        orc_merge_order(num_episodes, order);
        int64_t off = 0;
        for (int s = 0; s < num_episodes; ++s) {
            const episode_t* ep = &j.eps[order[s]];
            const size_t n = (size_t)ep->n;
            memcpy(out->obs + off * nc, ep->obs, sizeof(int32_t) * n * nc);
            memcpy(out->logits + off * na, ep->logits, sizeof(float) * n * na);
            memcpy(out->values + off, ep->values, sizeof(float) * n);
            memcpy(out->rewards + off, ep->rewards, sizeof(float) * n);
            memcpy(out->advs + off, ep->advs, sizeof(float) * n);
            memcpy(out->rets + off, ep->rets, sizeof(float) * n);
            memcpy(out->actions + off, ep->actions, sizeof(int32_t) * n);
            memcpy(out->perms + off, ep->perms, sizeof(int32_t) * n);
            off += ep->n;
        }
        for (int e = 0; e < num_episodes; ++e) out->ep_len[e] = j.eps[e].n;
        free(order);
    }
    for (int e = 0; e < num_episodes; ++e) {
        episode_t* ep = &j.eps[e];
        free(ep->obs); free(ep->logits); free(ep->values); free(ep->rewards);
        free(ep->advs); free(ep->rets); free(ep->actions); free(ep->perms);
    }
    free(j.eps);
    return rc;
}

void orc_collected_free(orc_collected* c) {
    free(c->ep_len); free(c->obs); free(c->logits); free(c->values); free(c->rewards);
    free(c->advs); free(c->rets); free(c->actions); free(c->perms);
    memset(c, 0, sizeof(*c));
}

/* ------------------------------------------------------- solve / evaluate --- */

/* Test infrastructure: while a sink is installed, every data-dependent decision of solve / evaluate / MCTS reports how
 * close it was to going the other way (argmax: best minus second best; weighted draw: distance to the nearest bin edge
 * as a fraction of the total weight; UCB descent: best minus second-best UCB).  The parity tests use the minimum over an
 * episode to tell a flipped near-tie from a real difference. */
static __thread float* g_margin_sink = NULL;
static void note_margin(float m) { if (g_margin_sink && m < *g_margin_sink) *g_margin_sink = m; }
static float weighted_margin(const float* w, int n, float u);

void orc_single_solve(orc_env* env, const orc_policy* p, int32_t deterministic, uint64_t seed, uint32_t collect_id,
                      uint32_t stream_id, float* success, float* total, int32_t* actions, int32_t* n_actions) {
    orc_single_solve_mcts(env, p, deterministic, 0, 0.0f, 0, seed, collect_id, stream_id, success, total, actions, n_actions);
}

void orc_single_solve_mcts(orc_env* env, const orc_policy* p, int32_t deterministic, int32_t n_mcts, float C,
                           int32_t max_expand_depth, uint64_t seed, uint32_t collect_id, uint32_t stream_id,
                           float* success, float* total, int32_t* actions, int32_t* n_actions) {
    /* rl/solve.rs:17-71 */
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    const int nc = orc_env_num_cells(env), na = orc_env_num_actions(env);
    float tot = 0.0f;
    int t = 0;
    while (!orc_env_is_final(env)) {
        int32_t obs[ORC_MAX_CELLS];
        uint8_t masks[16];
        float probs[16], value;
        tot += orc_env_reward(env);
        orc_env_observe(env, obs);
        orc_env_masks(env, masks);
        int perm = -1;
        if (p->n_perms > 0) {
            const uint32_t ctr[4] = {stream_id, (uint32_t)t, ORC_RNG_PERM, collect_id};
            uint32_t w[4];
            orc_philox4x32_10(ctr, key, w);
            perm = (int)mulhi32(w[0], (uint32_t)p->n_perms);
        }
        if (n_mcts > 0)   /* solve.rs:40-47: predict_probs_mcts on a clone of the env */
            orc_mcts_probs(env, p, n_mcts, C, max_expand_depth, seed, collect_id, stream_id, t, probs, NULL);
        else
            orc_policy_predict(p, obs, nc, masks, perm, probs, &value);
        int act = 0;
        if (deterministic) {
            act = orc_argmax(probs, na);
            if (g_margin_sink) {
                float second = -INFINITY;
                for (int i = 0; i < na; ++i) if (i != act && probs[i] > second) second = probs[i];
                if (na > 1) note_margin(probs[act] - second);
            }
        } else {
            /* nn/policy.rs:153-167: WeightedIndex -- first index whose cumulative weight exceeds the draw */
            float tw = 0.0f;
            for (int i = 0; i < na; ++i) tw += probs[i];
            if (tw > 0.0f) {
                const uint32_t ctr[4] = {stream_id, (uint32_t)t, ORC_RNG_SOLVE, collect_id};
                uint32_t w[4];
                orc_philox4x32_10(ctr, key, w);
                const float chosen = orc_u32_to_unit_f32(w[0]) * tw;
                if (g_margin_sink) note_margin(weighted_margin(probs, na, orc_u32_to_unit_f32(w[0])));
                float cum = 0.0f;
                int last = 0, found = 0;
                for (int i = 0; i < na; ++i) {
                    if (probs[i] > 0.0f) {
                        cum += probs[i];
                        last = i;
                        if (!found && cum > chosen) { act = i; found = 1; }
                    }
                }
                if (!found) act = last;
            }
        }
        orc_env_step(env, act);
        if (actions) actions[t] = act;
        ++t;
    }
    tot += orc_env_reward(env);
    *success = orc_env_success(env) ? 1.0f : 0.0f;
    *total = tot;
    if (n_actions) *n_actions = t;
}

void orc_solve(const orc_env* env, const orc_policy* p, int32_t deterministic, int32_t num_searches, uint64_t seed,
               uint32_t collect_id, uint32_t id0, float* success, float* total, int32_t* actions, int32_t* n_actions) {
    orc_solve_mcts(env, p, deterministic, num_searches, 0, 0.0f, 0, seed, collect_id, id0, success, total, actions, n_actions);
}

void orc_solve_mcts(const orc_env* env, const orc_policy* p, int32_t deterministic, int32_t num_searches, int32_t n_mcts,
                    float C, int32_t max_expand_depth, uint64_t seed, uint32_t collect_id, uint32_t id0, float* success,
                    float* total, int32_t* actions, int32_t* n_actions) {
    /* rl/solve.rs:73-101: best = ((0, -inf), []) ; strict tuple '>' keeps the first best */
    float bs = 0.0f, br = -INFINITY;
    int bn = 0;
    int32_t tmp[4096];
    for (int s = 0; s < num_searches; ++s) {
        orc_env e = *env;
        float s1, r1; int32_t n1 = 0;
        orc_single_solve_mcts(&e, p, deterministic, n_mcts, C, max_expand_depth, seed, collect_id, id0 + (uint32_t)s, &s1, &r1, tmp, &n1);
        if (s1 > bs || (s1 == bs && r1 > br)) {
            bs = s1; br = r1; bn = n1;
            if (actions) memcpy(actions, tmp, sizeof(int32_t) * (size_t)n1);
        }
    }
    *success = bs; *total = br;
    if (n_actions) *n_actions = bn;
}

void orc_evaluate(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes, int32_t deterministic,
                  int32_t num_searches, uint64_t seed, uint32_t collect_id, uint32_t reset_base, uint32_t search_base,
                  float* success_rate, float* mean_reward, float* best_success, float* best_total) {
    orc_evaluate_mcts(spec, p, num_episodes, deterministic, num_searches, 0, 0.0f, 0, seed, collect_id, reset_base, search_base,
                      success_rate, mean_reward, best_success, best_total);
}

void orc_evaluate_mcts(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes, int32_t deterministic,
                       int32_t num_searches, int32_t n_mcts, float C, int32_t max_expand_depth, uint64_t seed,
                       uint32_t collect_id, uint32_t reset_base, uint32_t search_base, float* success_rate,
                       float* mean_reward, float* best_success, float* best_total) {
    /* rl/evaluate.rs:22-48 (the serial branch; the rayon branch reduces the same per-episode values) */
    float succ = 0.0f, rew = 0.0f;
    for (int ep = 0; ep < num_episodes; ++ep) {
        orc_env env;
        orc_env_init(&env, spec);
        orc_env_reset(&env, seed, reset_base + (uint32_t)ep, collect_id);
        float s1, r1;
        orc_solve_mcts(&env, p, deterministic, num_searches, n_mcts, C, max_expand_depth, seed, collect_id,
                       search_base + (uint32_t)(ep * num_searches), &s1, &r1, NULL, NULL);
        succ += s1; rew += r1;
        if (best_success) best_success[ep] = s1;
        if (best_total) best_total[ep] = r1;
        if (g_margin_sink) ++g_margin_sink, *g_margin_sink = INFINITY;      /* next episode's slot (orc_evaluate_margins) */
    }
    *success_rate = succ / (float)num_episodes;
    *mean_reward = rew / (float)num_episodes;
}

void orc_evaluate_margins(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes, int32_t deterministic,
                          int32_t num_searches, int32_t n_mcts, float C, int32_t max_expand_depth, uint64_t seed,
                          uint32_t collect_id, uint32_t reset_base, uint32_t search_base, float* best_success,
                          float* best_total, float* min_margin) {
    /* orc_evaluate_mcts with the smallest decision margin of every episode (all its searches and steps) */
    float* sink = (float*)malloc(sizeof(float) * (size_t)(num_episodes + 1));
    float sr, mr;
    sink[0] = INFINITY;
    g_margin_sink = sink;
    orc_evaluate_mcts(spec, p, num_episodes, deterministic, num_searches, n_mcts, C, max_expand_depth, seed, collect_id,
                      reset_base, search_base, &sr, &mr, best_success, best_total);
    g_margin_sink = NULL;
    memcpy(min_margin, sink, sizeof(float) * (size_t)num_episodes);
    free(sink);
}

/* ---------------------------------------------------------------- AlphaZero --- */

typedef struct { orc_env state; int action, parent, first_child, n_children; float prior, value_sum; uint32_t visits; } mnode;
typedef struct { mnode* nodes; int n, cap; } mtree;

static int tree_add(mtree* t, const mnode* nd) {
    if (t->n == t->cap) { t->cap = t->cap ? t->cap * 2 : 256; t->nodes = (mnode*)realloc(t->nodes, sizeof(mnode) * (size_t)t->cap); }
    t->nodes[t->n] = *nd;
    return t->n++;
}

/* weighted draw like rand's WeightedIndex (nn/policy.rs:153-167): first index whose cumulative weight exceeds
 * u * total; 0 when every weight is zero (the reference prints an error and returns 0) */
static int weighted_index(const float* w, int n, float u) {
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

static void mcts_expand(mtree* t, int idx, const float* priors, int na) {
    /* search.rs:56-75: one child per action with prior > 0, in action order */
    t->nodes[idx].first_child = t->n;
    int cnt = 0;
    for (int a = 0; a < na; ++a) {
        if (priors[a] <= 0.0f) continue;
        mnode c;
        memset(&c, 0, sizeof(c));
        c.state = t->nodes[idx].state;
        orc_env_step(&c.state, a);
        c.action = a; c.parent = idx; c.prior = priors[a]; c.first_child = -1;
        tree_add(t, &c);
        ++cnt;
    }
    t->nodes[idx].n_children = cnt;
}

/* distance of a weighted draw from the nearest bin edge, as a fraction of the total weight: a device/host difference
 * of that size in the priors can move the draw into the neighbouring child */
static float weighted_margin(const float* w, int n, float u) {
    float tw = 0.0f, cum = 0.0f, m = INFINITY;
    for (int i = 0; i < n; ++i) tw += w[i];
    if (!(tw > 0.0f)) return INFINITY;
    const float chosen = u * tw;
    for (int i = 0; i + 1 < n; ++i) {                        /* the last edge (cum == tw) is never crossed: u < 1 */
        cum += w[i];
        const float d = fabsf(cum - chosen) / tw;
        if (d < m) m = d;
    }
    return m;
}

/* search.rs:104-189.  Optional per-simulation trace (test infrastructure): the leaf the UCB descent of simulation s
 * ended on, the node its value was backed up from (the sampled child, or the leaf itself when it was terminal), and the
 * smallest decision margin of that simulation -- best minus second-best UCB over the levels of the descent and the
 * bin-edge distance of the child draw -- and the number of nodes its backup updated (the root and the backed-up node
 * included).  Node indices count expansions in order, so two implementations that made the same decisions so far agree
 * on them. */
static void mcts_core(const orc_env* env, const orc_policy* p, int32_t n_sims, float C, int32_t max_expand_depth,
                      uint64_t seed, uint32_t collect_id, uint32_t stream_id, int32_t t_step, float* probs, int32_t* visits,
                      int32_t* trace_leaf, int32_t* trace_child, float* trace_margin, int32_t* trace_len) {
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    const int nc = orc_env_num_cells(env), na = orc_env_num_actions(env);
    const int med = max_expand_depth > 1 ? max_expand_depth : 1;
    mtree tr = {0, 0, 0};
    int32_t obs[ORC_MAX_CELLS];
    uint8_t masks[16];
    float pr[16], value;
    mnode root;
    memset(&root, 0, sizeof(root));
    root.state = *env; root.action = -1; root.parent = -1; root.visits = 1; root.first_child = -1;
    tree_add(&tr, &root);
    orc_env_observe(env, obs); orc_env_masks(env, masks);
    orc_policy_full_predict(p, obs, nc, masks, pr, &value);
    mcts_expand(&tr, 0, pr, na);
    for (int sim = 0; sim < n_sims; ++sim) {
        int node = 0;
        float margin = INFINITY;
        while (tr.nodes[node].n_children > 0) {                      /* next(): argmax UCB, strict '>' (search.rs:77-91) */
            const mnode* par = &tr.nodes[node];
            int best = -1; float best_ucb = -INFINITY, second = -INFINITY;
            for (int k = 0; k < par->n_children; ++k) {
                const mnode* ch = &tr.nodes[par->first_child + k];
                const float q = ch->visits == 0 ? 0.0f : ch->value_sum / (float)ch->visits;      /* search.rs:29-39 */
                const float ucb = q + C * (sqrtf((float)par->visits) / ((float)ch->visits + 1.0f)) * ch->prior;
                if (ucb > best_ucb) { second = best_ucb; best = par->first_child + k; best_ucb = ucb; }
                else if (ucb > second) second = ucb;
            }
            if (best < 0) break;
            if (par->n_children > 1 && best_ucb - second < margin) margin = best_ucb - second;
            node = best;
        }
        if (trace_leaf) trace_leaf[sim] = node;
        float v = 0.0f;
        for (int d = 0; d < max_expand_depth; ++d) {
            const orc_env* st = &tr.nodes[node].state;
            v = orc_env_reward(st);
            if (orc_env_is_final(st)) break;
            float nv;
            orc_env_observe(st, obs); orc_env_masks(st, masks);
            orc_policy_full_predict(p, obs, nc, masks, pr, &nv);
            mcts_expand(&tr, node, pr, na);
            const uint32_t ctr[4] = {stream_id, (uint32_t)((t_step * (n_sims + 1) + sim) * med + d), ORC_RNG_MCTS, collect_id};
            uint32_t w[4];
            orc_philox4x32_10(ctr, key, w);
            float cp[16];
            const mnode* par = &tr.nodes[node];
            for (int k = 0; k < par->n_children; ++k) cp[k] = tr.nodes[par->first_child + k].prior;
            const float u = orc_u32_to_unit_f32(w[0]);
            const float wm = weighted_margin(cp, par->n_children, u);
            if (wm < margin) margin = wm;
            node = par->first_child + weighted_index(cp, par->n_children, u);   /* next_sample */
            v = nv;
        }
        if (trace_child) trace_child[sim] = node;
        if (trace_margin) trace_margin[sim] = margin;
        note_margin(margin);
        int len = 0;
        for (int b = node; b >= 0; b = tr.nodes[b].parent) { tr.nodes[b].value_sum += v; tr.nodes[b].visits += 1; ++len; }
        if (trace_len) trace_len[sim] = len;
    }
    float sum = 0.0f;
    for (int a = 0; a < na; ++a) { probs[a] = 0.0f; if (visits) visits[a] = 0; }
    for (int k = 0; k < tr.nodes[0].n_children; ++k) {
        const mnode* ch = &tr.nodes[tr.nodes[0].first_child + k];
        probs[ch->action] = (float)ch->visits;
        if (visits) visits[ch->action] = (int32_t)ch->visits;
    }
    for (int a = 0; a < na; ++a) sum += probs[a];
    if (sum > 0.0f) { for (int a = 0; a < na; ++a) probs[a] /= sum; }
    else { for (int a = 0; a < na; ++a) probs[a] = 1.0f / (float)na; }
    free(tr.nodes);
}

void orc_mcts_probs(const orc_env* env, const orc_policy* p, int32_t n_sims, float C, int32_t max_expand_depth,
                    uint64_t seed, uint32_t collect_id, uint32_t stream_id, int32_t t_step, float* probs, int32_t* visits) {
    mcts_core(env, p, n_sims, C, max_expand_depth, seed, collect_id, stream_id, t_step, probs, visits, NULL, NULL, NULL, NULL);
}

void orc_mcts_trace(const orc_env* env, const orc_policy* p, int32_t n_sims, float C, int32_t max_expand_depth,
                    uint64_t seed, uint32_t collect_id, uint32_t stream_id, int32_t t_step, float* probs, int32_t* visits,
                    int32_t* trace_leaf, int32_t* trace_child, float* trace_margin, int32_t* trace_len) {
    mcts_core(env, p, n_sims, C, max_expand_depth, seed, collect_id, stream_id, t_step, probs, visits, trace_leaf, trace_child, trace_margin,
              trace_len);
}

int orc_az_collect(const orc_env_spec* spec, const orc_policy* p, int32_t num_episodes, int32_t n_sims, float C,
                   int32_t max_expand_depth, uint64_t seed, uint32_t collect_id, uint32_t env_id_base, orc_az_collected* out) {
    /* az.rs:51-130 */
    memset(out, 0, sizeof(*out));
    if (num_episodes <= 0) return -1;
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    orc_env tmp; orc_env_init(&tmp, spec);
    const int nc = orc_env_num_cells(&tmp), na = orc_env_num_actions(&tmp);
    typedef struct { int n; int32_t* obs; float* probs; float* rew; int32_t* act; float* rem; } ep_t;
    ep_t* eps = (ep_t*)calloc((size_t)num_episodes, sizeof(ep_t));
    int64_t R = 0;
    for (int ep = 0; ep < num_episodes; ++ep) {
        orc_env env; orc_env_init(&env, spec);
        const uint32_t id = env_id_base + (uint32_t)ep;
        orc_env_reset(&env, seed, id, collect_id);
        int cap = 64, n = 0;
        ep_t* E = &eps[ep];
        E->obs = (int32_t*)malloc(sizeof(int32_t) * (size_t)cap * nc); E->probs = (float*)malloc(sizeof(float) * (size_t)cap * na);
        E->rew = (float*)malloc(sizeof(float) * cap); E->act = (int32_t*)malloc(sizeof(int32_t) * cap);
        float total = 0.0f;
        float* totals = (float*)malloc(sizeof(float) * cap);
        for (;;) {
            if (n == cap) {
                cap *= 2;
                E->obs = (int32_t*)realloc(E->obs, sizeof(int32_t) * (size_t)cap * nc); E->probs = (float*)realloc(E->probs, sizeof(float) * (size_t)cap * na);
                E->rew = (float*)realloc(E->rew, sizeof(float) * cap); E->act = (int32_t*)realloc(E->act, sizeof(int32_t) * cap);
                totals = (float*)realloc(totals, sizeof(float) * cap);
            }
            orc_mcts_probs(&env, p, n_sims, C, max_expand_depth, seed, collect_id, id, n, E->probs + (size_t)n * na, NULL);
            const uint32_t ctr[4] = {id, (uint32_t)n, ORC_RNG_AZ_ACT, collect_id};
            uint32_t w[4];
            orc_philox4x32_10(ctr, key, w);
            const int action = weighted_index(E->probs + (size_t)n * na, na, orc_u32_to_unit_f32(w[0]));
            const float val = orc_env_reward(&env);
            totals[n] = total;
            total += val;
            orc_env_observe(&env, E->obs + (size_t)n * nc);
            E->rew[n] = val; E->act[n] = action;
            ++n;
            if (orc_env_is_final(&env)) break;
            orc_env_step(&env, action);
        }
        E->n = n;
        E->rem = (float*)malloc(sizeof(float) * n);
        for (int t = 0; t < n; ++t) E->rem[t] = total - totals[t];          /* az.rs:93 */
        free(totals);
        R += n;
    }
    out->n_records = R; out->num_episodes = num_episodes; out->n_cells = nc; out->num_actions = na;
    out->ep_len = (int32_t*)malloc(sizeof(int32_t) * (size_t)num_episodes);
    out->obs = (int32_t*)malloc(sizeof(int32_t) * (size_t)R * nc); out->probs = (float*)malloc(sizeof(float) * (size_t)R * na);
    out->rewards = (float*)malloc(sizeof(float) * (size_t)R); out->actions = (int32_t*)malloc(sizeof(int32_t) * (size_t)R);
    out->remaining_values = (float*)malloc(sizeof(float) * (size_t)R);
    int32_t* order = (int32_t*)malloc(sizeof(int32_t) * (size_t)num_episodes);
    orc_merge_order(num_episodes, order);
    int64_t off = 0;
    for (int s2 = 0; s2 < num_episodes; ++s2) {
        const ep_t* E = &eps[order[s2]];
        const size_t n = (size_t)E->n;
        memcpy(out->obs + off * nc, E->obs, sizeof(int32_t) * n * nc);
        memcpy(out->probs + off * na, E->probs, sizeof(float) * n * na);
        memcpy(out->rewards + off, E->rew, sizeof(float) * n);
        memcpy(out->actions + off, E->act, sizeof(int32_t) * n);
        memcpy(out->remaining_values + off, E->rem, sizeof(float) * n);
        off += E->n;
    }
    for (int ep = 0; ep < num_episodes; ++ep) {
        out->ep_len[ep] = eps[ep].n;
        free(eps[ep].obs); free(eps[ep].probs); free(eps[ep].rew); free(eps[ep].act); free(eps[ep].rem);
    }
    free(order); free(eps);
    return 0;
}

void orc_az_collected_free(orc_az_collected* c) {
    free(c->ep_len); free(c->obs); free(c->probs); free(c->rewards); free(c->actions); free(c->remaining_values);
    memset(c, 0, sizeof(*c));
}
