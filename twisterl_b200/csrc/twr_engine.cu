// twr_engine.cu -- host side of the C ABI declared in include/twisterl_b200.h: owns device memory,
// validates env specs / policy shapes, drives the per-step kernel sequence of a collect on one CUDA
// stream, and moves results to caller buffers.  No CPU compute path exists here: every Env / Policy /
// collector operation is a kernel launch (twr_kernels.cu, twr_forward_*.cu).
#include "../../include/twisterl_b200.h"
#include "twr_kernels.cuh"

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <functional>
#include <map>
#include <algorithm>
#include <string>
#include <thread>
#include <vector>

extern std::atomic<long long> g_twr_launches;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
}  // namespace
// No C++ exception may leave through the C boundary (std::bad_alloc of a host staging vector, std::system_error of a
// thread): the exported functions whose bodies can throw run inside this guard.
template <typename F>
static int twr_guard(F&& body) {
    try {
        return body();
    } catch (const std::exception& ex) {
        return fail(TWR_ERR_INVALID, std::string("host-side failure: ") + ex.what());
    } catch (...) {
        return fail(TWR_ERR_INVALID, "host-side failure");
    }
}
// error hook for the other translation units of the library (twr_safetensors.cpp)
extern "C" int twr_set_error(int code, const char* msg) { return fail(code, msg ? msg : ""); }
namespace {

#define CU_TRY(expr)                                                                              \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return fail(TWR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));        \
    } while (0)

template <typename T>
int dev_alloc(T** p, size_t count) {
    *p = nullptr;
    if (count == 0) count = 1;
    CU_TRY(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
    return TWR_OK;
}
template <typename T>
void dev_free(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}

int check_spec(const twr_env_spec* s, EnvParams* out) {
    if (!s) return fail(TWR_ERR_INVALID, "env spec is NULL");
    if (s->width < 1 || s->height < 1) return fail(TWR_ERR_INVALID, "env width/height must be >= 1");
    EnvParams p{};
    p.kind = s->kind; p.W = s->width; p.H = s->height; p.N = s->width * s->height;
    p.difficulty = s->difficulty; p.depth_slope = s->depth_slope; p.max_depth = s->max_depth;
    if (s->difficulty < 0 || s->max_depth < 0) return fail(TWR_ERR_INVALID, "difficulty/max_depth must be >= 0");
    if (s->kind == TWR_ENV_PUZZLE || s->kind == TWR_ENV_PUZZLE_WIDE) {
        // one env; the kernels see one Puzzle kind and pick the cell encoding from the board size (twr_common.cuh)
        p.kind = TWR_ENV_PUZZLE;
        if (s->kind == TWR_ENV_PUZZLE && p.N > TWR_MAX_CELLS_BYTES)
            return fail(TWR_ERR_UNSUPPORTED, "Puzzle boards above 16 cells are env kind TWR_ENV_PUZZLE_WIDE "
                                             "(5-bit cells, up to 25 cells)");
        if (p.N > TWR_MAX_CELLS_PUZZLE)
            return fail(TWR_ERR_UNSUPPORTED, "Puzzle boards above 25 cells are not implemented on the device path "
                                             "(the 128-bit env state holds at most 25 five-bit cells)");
        if (s->depth_slope < 0) return fail(TWR_ERR_INVALID, "depth_slope must be >= 0");
        if ((int64_t)s->depth_slope * s->difficulty >= (1 << 24)) return fail(TWR_ERR_INVALID, "depth budget too large");
    } else if (s->kind == TWR_ENV_GRIDWORLD) {
        // bytes 0..2 of the state hold any cell index; the bound is the forward's: above 64 cells the compact table
        // (4 rows per cell) leaves the pair kernel's 256-row operand and a record carries more than 64 indices
        if (p.N > TWR_MAX_OBS || p.N < 3)
            return fail(TWR_ERR_UNSUPPORTED, "GridWorld needs 3..64 cells on the device path");
        const int cap = s->width + s->height;                      // lib.rs:36,92-94
        p.difficulty = s->difficulty < cap ? s->difficulty : cap;
        if (s->max_depth >= (1 << 24)) return fail(TWR_ERR_INVALID, "max_steps too large");
    } else {
        return fail(TWR_ERR_UNSUPPORTED, "unknown env kind: only Puzzle and GridWorld run on the device "
                                         "(arbitrary Env implementations have no CPU fallback here)");
    }
    *out = p;
    return TWR_OK;
}

int horizon_of(const EnvParams& p) {   // max env steps of one episode
    return p.kind == TWR_ENV_PUZZLE ? p.depth_slope * p.difficulty : p.max_depth;
}

}  // namespace

#include "twr_private.cuh"

template <typename T>
struct Staging {
    T* d = nullptr;
    ~Staging() { if (d) cudaFree(d); }
    int alloc(size_t n) { return dev_alloc(&d, n); }
};


template <typename T>
static int query_field(twr_envs* v, T* host, size_t per_env, int which) {
    if (!v || !host) return fail(TWR_ERR_INVALID, "envs/out is NULL");
    if (v->n == 0) return TWR_OK;
    twr_engine* e = v->eng;
    CU_TRY(cudaSetDevice(e->device));
    Staging<T> st;
    int rc = st.alloc((size_t)v->n * per_env);
    if (rc) return rc;
    launch_envs_query(e->stream, v->p, v->cells, v->meta, v->n,
                      which == 0 ? reinterpret_cast<int64_t*>(st.d) : nullptr,
                      which == 1 ? reinterpret_cast<int32_t*>(st.d) : nullptr,
                      which == 2 ? reinterpret_cast<uint8_t*>(st.d) : nullptr,
                      which == 3 ? reinterpret_cast<float*>(st.d) : nullptr,
                      which == 4 ? reinterpret_cast<uint8_t*>(st.d) : nullptr,
                      which == 5 ? reinterpret_cast<uint8_t*>(st.d) : nullptr,
                      which == 6 ? reinterpret_cast<int32_t*>(st.d) : nullptr);
    CU_TRY(cudaMemcpyAsync(host, st.d, sizeof(T) * (size_t)v->n * per_env, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
}


// ---------------------------------------------------------------------------------------
extern "C" {

int twr_abi_version(void) { return TWR_ABI_VERSION; }
const char* twr_last_error(void) { return g_err.c_str(); }

int twr_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ForwardArgs::tc_terms of an engine precision (bit 3 marks "explicit", bit 4 = fp8 correction products)
static int terms_of_precision(int precision) {
    return precision == TWR_PREC_F16X2_W16 ? (8 | 1 | 2) : precision == TWR_PREC_F16_F8C ? (16 | 8 | 1 | 2) : 0;
}

int twr_engine_create(const twr_engine_cfg* cfg, twr_engine** out) {
    return twr_guard([&]() -> int {
    if (!cfg || !out) return fail(TWR_ERR_INVALID, "cfg/out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t ce = cudaGetDeviceCount(&n);
    if (ce != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(TWR_ERR_CUDA, "no CUDA device: the twisterl_b200 engine has no CPU fallback");
    }
    if (cfg->device < 0 || cfg->device >= n) return fail(TWR_ERR_INVALID, "device ordinal out of range");
    if (cfg->precision != TWR_PREC_FP32 && cfg->precision != TWR_PREC_F16X2 && cfg->precision != TWR_PREC_F16X2_W16 &&
        cfg->precision != TWR_PREC_F16_F8C)
        return fail(TWR_ERR_INVALID, "unknown precision");
    if (cfg->world < 1 || cfg->rank < 0 || cfg->rank >= cfg->world) return fail(TWR_ERR_INVALID, "bad rank/world");
    CU_TRY(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major < 10)
        return fail(TWR_ERR_UNSUPPORTED, std::string("device '") + prop.name + "' is not Blackwell (sm_100a kernels only)");
    twr_engine* e = new twr_engine();
    e->device = cfg->device; e->precision = cfg->precision; e->seed = cfg->seed;
    e->rank = cfg->rank; e->world = cfg->world;
    e->tc_terms = terms_of_precision(cfg->precision);
    if (const char* f = getenv("TWISTERL_B200_TC_FLAGS")) e->tc_flags = atoi(f);
    if (cfg->stream) {
        e->stream = reinterpret_cast<cudaStream_t>(cfg->stream);
    } else {
        cudaError_t se = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
        if (se != cudaSuccess) { delete e; return fail(TWR_ERR_CUDA, cudaGetErrorString(se)); }
        e->own_stream = true;
    }
    cudaError_t ce2 = cudaEventCreate(&e->ev_t0);
    if (ce2 == cudaSuccess) ce2 = cudaEventCreate(&e->ev_t1);
    if (ce2 == cudaSuccess) ce2 = cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking);
    if (ce2 == cudaSuccess) ce2 = cudaMalloc(reinterpret_cast<void**>(&e->bal_flags), 1024 * sizeof(int32_t));
    for (int i = 0; i < 2 && ce2 == cudaSuccess; ++i) ce2 = cudaEventCreateWithFlags(&e->ev_done[i], cudaEventDisableTiming);
    for (int i = 0; i < TWR_MAX_SUBBATCH && ce2 == cudaSuccess; ++i) {
        ce2 = cudaEventCreate(&e->ev_copied[i]);   // timing on: TWISTERL_B200_E2E_TRACE
        if (ce2 == cudaSuccess) ce2 = cudaEventCreateWithFlags(&e->ev_small[i], cudaEventDisableTiming);
    }
    // collect statistics come back through MAPPED pinned memory written by a one-thread kernel, not through a D2H copy:
    // a 32-byte cudaMemcpyAsync queues on the copy engine behind the bulk D2H of the previous sub-batch (measured: the
    // host learned a sub-batch's record count up to 2.3 ms late, and every later copy started that much later)
    if (ce2 == cudaSuccess) ce2 = cudaHostAlloc(reinterpret_cast<void**>(&e->h_stats), 8 * sizeof(unsigned long long), cudaHostAllocMapped);
    if (ce2 == cudaSuccess) ce2 = cudaHostGetDevicePointer(reinterpret_cast<void**>(&e->d_hstats), e->h_stats, 0);
    if (ce2 != cudaSuccess) {
        const std::string msg = std::string("twr_engine_create: ") + cudaGetErrorString(ce2);
        twr_engine_destroy(e);
        return fail(TWR_ERR_CUDA, msg);
    }
    e->launches0 = g_twr_launches.load();
    *out = e;
    return TWR_OK;
    });
}

static void mcts_release(twr_engine* e) {
    MctsCache& c = e->mcts;
    dev_free(c.cells); dev_free(c.node); dev_free(c.meta); dev_free(c.parent); dev_free(c.n_nodes); dev_free(c.fwd_list);
    dev_free(c.fwd_env); dev_free(c.fwd_count); dev_free(c.cur_node); dev_free(c.path); dev_free(c.path_len); dev_free(c.leaf_pos);
    dev_free(c.active); dev_free(c.cur_value);
    c.cap_nodes = 0; c.cap_B = 0;
}

static void free_outset(twr_engine::OutSet& o) {
    dev_free(o.obs); dev_free(o.logits); dev_free(o.values); dev_free(o.rewards);
    dev_free(o.advs); dev_free(o.rets); dev_free(o.actions); dev_free(o.perms);
}

static void free_collect_buffers(twr_engine* e) {
    CollectBuffers& b = e->buf;
    dev_free(b.cells); dev_free(b.meta); dev_free(b.live_a); dev_free(b.live_b); dev_free(b.n_live);
    dev_free(b.logits); dev_free(b.values);
    dev_free(b.rec_state); dev_free(b.rec_logits); dev_free(b.rec_value); dev_free(b.rec_reward);
    dev_free(b.rec_adv); dev_free(b.rec_ret); dev_free(b.rec_action); dev_free(b.rec_perm);
    dev_free(b.ep_len); dev_free(b.ep_off); dev_free(b.stats);
    for (auto& o : e->outs) free_outset(o);
    e->cap_B = 0; e->cap_T = 0; e->cap_R = 0; e->cap_cells = 0;
}

void twr_engine_destroy(twr_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    twr_comm_destroy(e);
    mcts_release(e);
    if (e->trace_buf) { cudaFree(e->trace_buf); e->trace_buf = nullptr; }
    free_collect_buffers(e);
    free_outset(e->merged);
    dev_free(e->merged_ep_len);
    for (auto ev : e->ev) cudaEventDestroy(ev);
    dev_free(e->ep_len_id);
    for (int i = 0; i < 2; ++i) if (e->ev_done[i]) cudaEventDestroy(e->ev_done[i]);
    for (int i = 0; i < TWR_MAX_SUBBATCH; ++i) {
        if (e->ev_copied[i]) cudaEventDestroy(e->ev_copied[i]);
        if (e->ev_small[i]) cudaEventDestroy(e->ev_small[i]);
    }
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->bal_flags) cudaFree(e->bal_flags);
    if (e->h_stats) cudaFreeHost(e->h_stats);
    if (e->ev_t0) cudaEventDestroy(e->ev_t0);
    if (e->ev_t1) cudaEventDestroy(e->ev_t1);
    if (e->own_stream) cudaStreamDestroy(e->stream);
    delete e;
}

int twr_engine_synchronize(twr_engine* e) {
    if (!e) return fail(TWR_ERR_INVALID, "engine is NULL");
    CU_TRY(cudaSetDevice(e->device));
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
}

int64_t twr_engine_launch_count(const twr_engine* e) {
    return e ? (int64_t)(g_twr_launches.load() - e->launches0) : 0;
}

int twr_engine_set_collect_id(twr_engine* e, uint32_t collect_id) {
    if (!e) return fail(TWR_ERR_INVALID, "engine is NULL");
    e->collect_id = collect_id;
    return TWR_OK;
}

int twr_engine_set_timing(twr_engine* e, int32_t enabled) {
    if (!e) return fail(TWR_ERR_INVALID, "engine is NULL");
    e->timing = enabled != 0;
    return TWR_OK;
}

int twr_engine_last_timing(const twr_engine* e, float* forward_ms, float* total_ms, int64_t* forward_launches) {
    if (!e) return fail(TWR_ERR_INVALID, "engine is NULL");
    if (forward_ms) *forward_ms = e->last_fwd_ms;
    if (total_ms) *total_ms = e->last_total_ms;
    if (forward_launches) *forward_launches = e->last_fwd_launches;
    return TWR_OK;
}

// ----------------------------------------------------------------------- policy ---
// every Linear of the three stacks, in blob order (common..., action_net..., value_net...)
static std::vector<const twr_linear_desc*> all_linears(const twr_policy_desc* d) {
    std::vector<const twr_linear_desc*> v;
    for (int i = 0; i < d->n_common; ++i) v.push_back(d->common + i);
    for (int i = 0; i < d->n_action; ++i) v.push_back(d->action_net + i);
    for (int i = 0; i < d->n_value; ++i) v.push_back(d->value_net + i);
    return v;
}
// the shape the tile kernels (tcgen05 / fp32) implement: embedding+ReLU -> one common Linear+ReLU -> single-Linear heads
static bool is_standard_shape(const twr_policy_desc* d) {
    return d->emb_apply_relu && d->n_common == 1 && d->n_action == 1 && d->n_value == 1 && d->common[0].apply_relu;
}

static int validate_desc(const twr_policy_desc* d) {
    if (!d || !d->emb_vectors || !d->emb_bias) return fail(TWR_ERR_INVALID, "policy desc / embedding is NULL");
    if (d->obs_shape_len != 1)
        return fail(TWR_ERR_UNSUPPORTED, "EmbeddingBag obs_shape must have 1 (BasicPolicy) or 2 (Conv1dPolicy) dimensions");
    if (d->n_common < 0 || d->n_common > TWR_MAX_STACK || d->n_action < 1 || d->n_action > TWR_MAX_STACK || d->n_value < 1 ||
        d->n_value > TWR_MAX_STACK)
        return fail(TWR_ERR_UNSUPPORTED, "layer stacks: 0..4 common Linears and 1..4 Linears per head are implemented");
    if ((d->n_common > 0 && !d->common) || !d->action_net || !d->value_net) return fail(TWR_ERR_INVALID, "layer array is NULL");
    if (d->emb_size < 1) return fail(TWR_ERR_INVALID, "empty embedding");
    int width = d->emb_size;                                     // Sequential::forward chains the layers (nn/modules.rs:28-34)
    for (int i = 0; i < d->n_common; ++i) {
        const twr_linear_desc& l = d->common[i];
        if (!l.weights || !l.bias || l.in != width || l.out < 1) return fail(TWR_ERR_INVALID, "common layer sizes do not chain");
        width = l.out;
    }
    const int trunk = width;
    for (int i = 0; i < d->n_action; ++i) {
        const twr_linear_desc& l = d->action_net[i];
        if (!l.weights || !l.bias || l.in != width || l.out < 1) return fail(TWR_ERR_INVALID, "action_net layer sizes do not chain");
        width = l.out;
    }
    const twr_linear_desc& a = d->action_net[d->n_action - 1];
    if (a.apply_relu || a.out > TWR_MAX_ACTIONS) return fail(TWR_ERR_UNSUPPORTED, "action head must end in a Linear without ReLU, at most 4 actions");
    width = trunk;
    for (int i = 0; i < d->n_value; ++i) {
        const twr_linear_desc& l = d->value_net[i];
        if (!l.weights || !l.bias || l.in != width || l.out < 1) return fail(TWR_ERR_INVALID, "value_net layer sizes do not chain");
        width = l.out;
    }
    const twr_linear_desc& v = d->value_net[d->n_value - 1];
    if (v.apply_relu || v.out != 1) return fail(TWR_ERR_UNSUPPORTED, "value head must end in a Linear(.., 1) without ReLU");
    if (d->n_perms < 0 || d->n_perms > 127) return fail(TWR_ERR_INVALID, "n_perms must be in 0..127");
    if (d->n_perms > 0 && (!d->obs_perms || !d->act_perms)) return fail(TWR_ERR_INVALID, "perm arrays are NULL");
    if (d->obs_size < 1 || d->obs_size >= 65536) return fail(TWR_ERR_UNSUPPORTED, "obs_size must be in 1..65535");
    if (d->n_perms > 0) {
        for (int64_t i = 0; i < (int64_t)d->n_perms * d->obs_size; ++i)
            if (d->obs_perms[i] < 0 || d->obs_perms[i] >= d->obs_size) return fail(TWR_ERR_INVALID, "obs_perms entry out of range");
        for (int64_t i = 0; i < (int64_t)d->n_perms * a.out; ++i)
            if (d->act_perms[i] < 0 || d->act_perms[i] >= a.out) return fail(TWR_ERR_INVALID, "act_perms entry out of range");
    }
    return TWR_OK;
}

// Conv1dPolicy (nn/layers.rs:63-77): observation index i adds vectors[row] into the output slice
// [col*v, (col+1)*v), (row, col) = (i / shape[1], i % shape[1]) swapped when conv_dim == 1.  That is the 1-D
// EmbeddingBag of a block-sparse table T[i][col*v + k] = vectors[row][k]; adding the table's exact zeros leaves
// every fp32 partial sum unchanged, so the device path runs the expanded table through the same kernels.
// Returns a desc whose embedding points into `store` (obs_shape_len == 1 descs pass through untouched).
static int expand_conv1d(const twr_policy_desc* d, twr_policy_desc* out, std::vector<float>* store) {
    *out = *d;
    if (!d || d->obs_shape_len != 2) return TWR_OK;
    if (!d->emb_vectors) return fail(TWR_ERR_INVALID, "policy desc / embedding is NULL");
    const int s0 = d->obs_shape[0], s1 = d->obs_shape[1];
    if (s0 < 1 || s1 < 1 || (d->conv_dim != 0 && d->conv_dim != 1)) return fail(TWR_ERR_INVALID, "bad obs_shape / conv_dim");
    const int n_vec = d->conv_dim == 0 ? s0 : s1, n_col = d->conv_dim == 0 ? s1 : s0;
    if (d->obs_size != n_vec) return fail(TWR_ERR_INVALID, "conv1d EmbeddingBag needs obs_shape[conv_dim] vectors");
    if (d->emb_size % n_col) return fail(TWR_ERR_INVALID, "conv1d EmbeddingBag: bias length must be vector length x obs_shape[1-conv_dim]");
    const int v = d->emb_size / n_col;
    const int64_t full = (int64_t)s0 * s1;
    if (full >= 65536) return fail(TWR_ERR_UNSUPPORTED, "obs_size must be in 1..65535");
    store->assign((size_t)full * d->emb_size, 0.0f);
    for (int64_t i = 0; i < full; ++i) {
        int row = (int)(i / s1), col = (int)(i % s1);
        if (d->conv_dim == 1) { const int t = row; row = col; col = t; }
        memcpy(store->data() + (size_t)i * d->emb_size + (size_t)col * v, d->emb_vectors + (size_t)row * v, sizeof(float) * (size_t)v);
    }
    out->emb_vectors = store->data();
    out->obs_size = (int32_t)full;
    out->obs_shape_len = 1; out->obs_shape[0] = (int32_t)full; out->obs_shape[1] = 0; out->conv_dim = 0;
    return TWR_OK;
}

// the largest N with N * N <= obs_size: the board side of a table whose rows are (cell, value) pairs of an N-cell board
static int board_side(int obs_size) {
    int N = 1;
    while ((N + 1) * (N + 1) <= obs_size) ++N;
    return N;
}

// PolicyDev::tc_fold: N when obs_size = N * N and every twist maps each block of N rows onto a block (all blocks hit once)
static int fold_block(const twr_policy_desc* d) {
    const int N = board_side(d->obs_size);
    if (N * N != d->obs_size || N > TWR_MAX_CELLS) return 0;
    for (int q = 0; q < d->n_perms; ++q) {
        const int32_t* pm = d->obs_perms + (size_t)q * d->obs_size;
        uint64_t seen = 0;
        for (int c = 0; c < N; ++c) {
            const int tb = pm[c * N] / N;
            for (int v = 1; v < N; ++v)
                if (pm[c * N + v] / N != tb) return 0;
            if (tb < 0 || tb >= N || ((seen >> tb) & 1ull)) return 0;
            seen |= 1ull << tb;
        }
    }
    return N;
}

static int upload_policy(twr_policy* p, const twr_policy_desc* d) {
    twr_engine* e = p->eng;
    p->dev.tc_fold = p->tc_pack && !p->dev.generic ? fold_block(d) : 0;
    const int E = d->emb_size, A = d->action_net[d->n_action - 1].out;
    const std::vector<const twr_linear_desc*> lins = all_linears(d);
    bool same = d->obs_size == p->dev.obs_size && E == p->dev.E && A == p->dev.A && d->n_perms == p->dev.n_perms &&
                d->n_common == p->dev.n_common && d->n_action == p->dev.n_action && d->n_value == p->dev.n_value &&
                (d->emb_apply_relu != 0) == (p->dev.emb_relu != 0) && is_standard_shape(d) == !p->dev.generic;
    for (size_t i = 0; same && i < lins.size(); ++i)
        same = lins[i]->in == p->dev.lin[i].in && lins[i]->out == p->dev.lin[i].out && (lins[i]->apply_relu != 0) == (p->dev.lin[i].relu != 0);
    if (!same) return fail(TWR_ERR_INVALID, "twr_policy_update: shapes differ from the ones the policy was created with");
    cudaStream_t st = e->stream;
    float* b = p->d_blob;
    CU_TRY(cudaMemcpyAsync(b, d->emb_vectors, sizeof(float) * (size_t)d->obs_size * E, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(b + p->off_emb_b, d->emb_bias, sizeof(float) * E, cudaMemcpyHostToDevice, st));
    for (size_t i = 0; i < lins.size(); ++i) {
        CU_TRY(cudaMemcpyAsync(b + p->off_w[i], lins[i]->weights, sizeof(float) * (size_t)lins[i]->in * lins[i]->out, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(b + p->off_b[i], lins[i]->bias, sizeof(float) * (size_t)lins[i]->out, cudaMemcpyHostToDevice, st));
    }
    if (d->n_perms > 0) {
        CU_TRY(cudaMemcpyAsync(p->d_obs_perms, d->obs_perms, sizeof(int32_t) * (size_t)d->n_perms * d->obs_size, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(p->d_act_perms, d->act_perms, sizeof(int32_t) * (size_t)d->n_perms * A, cudaMemcpyHostToDevice, st));
    }
    if (p->tc_pack) launch_forward_tc2_pack(st, p->dev, p->tc_pack);
    CU_TRY(cudaStreamSynchronize(st));   // host source buffers may be freed by the caller after return
    return TWR_OK;
}

int twr_policy_create(twr_engine* e, const twr_policy_desc* d_in, twr_policy** out) {
    return twr_guard([&]() -> int {
    if (!e || !out) return fail(TWR_ERR_INVALID, "engine/out is NULL");
    *out = nullptr;
    if (!d_in) return fail(TWR_ERR_INVALID, "policy desc / embedding is NULL");
    twr_policy_desc flat;
    std::vector<float> table;
    int rc = expand_conv1d(d_in, &flat, &table);
    if (rc) return rc;
    const twr_policy_desc* d = &flat;
    if ((rc = validate_desc(d))) return rc;
    CU_TRY(cudaSetDevice(e->device));
    const std::vector<const twr_linear_desc*> lins = all_linears(d);
    const bool standard = is_standard_shape(d);
    const int E = d->emb_size, A = d->action_net[d->n_action - 1].out;
    const int H = d->n_common > 0 ? d->common[d->n_common - 1].out : E;     // trunk width
    twr_policy* p = new twr_policy();
    p->eng = e;
    p->dev.obs_size = d->obs_size; p->dev.E = E; p->dev.H = H; p->dev.A = A; p->dev.n_perms = d->n_perms;
    p->dev.n_obs = 0;
    p->dev.generic = standard ? 0 : 1;
    p->dev.emb_relu = d->emb_apply_relu ? 1 : 0;
    p->dev.n_common = d->n_common; p->dev.n_action = d->n_action; p->dev.n_value = d->n_value;
    int64_t off = (int64_t)d->obs_size * E;
    p->off_emb_b = off; off += E;
    int max_width = E;
    for (const twr_linear_desc* l : lins) {
        p->off_w.push_back(off); off += (int64_t)l->in * l->out;
        p->off_b.push_back(off); off += l->out;
        if (l->out > max_width) max_width = l->out;
    }
    p->dev.max_width = max_width;
    p->blob_floats = off;
    bool use_tc = false;
    if (standard) {
        PolicyDev probe = p->dev;
        probe.n_obs = 1;
        const char* why = "";
        // TWR_PREC_F16X2 = tensor cores where the shape fits the tcgen05 kernel (obs_size <= 256, E % 128 == 0 and
        // E <= 1024, H in {128, 256}); other shapes (GridWorld's 625-row table) run the fp32 SIMT kernel -- still on the device.
        // GridWorld-shaped tables (obs_size = N*N > 256, only rows i*N + {0,1,2,3} reachable): the pair kernel runs on
        // the compact 4N-row table when the twists (if any) keep the reachable rows among themselves
        const int N = board_side(d->obs_size);
        const bool square = N * N == d->obs_size;
        if (d->obs_size > 256) {
            bool ok = square && 4 * N <= 256;
            for (int64_t i = 0; ok && i < (int64_t)d->n_perms * d->obs_size; ++i)
                if ((i % d->obs_size) % N < 4 && d->obs_perms[i] % N >= 4) ok = false;
            if (ok) p->grid_n = N;
            if (ok && e->precision != TWR_PREC_FP32) probe.compact_n = p->dev.compact_n = N;
        }
        use_tc = e->precision != TWR_PREC_FP32 && forward_tc2_supported(probe);
        // The fp32 kernel's fit holds for the longest observation the policy can meet: N indices for the table of a board
        // above 32 cells.  Such a table (up to 64 cells) is taken whether or not it fits whole: call_dev sends GridWorld
        // forwards to the compact table and any forward the fp32 kernel cannot hold to the generic one.
        const int max_obs = square && N > TWR_MAX_CELLS ? N : TWR_MAX_CELLS;
        const bool big_board = max_obs > TWR_MAX_CELLS && N <= TWR_MAX_OBS && max_width <= 1024;
        // a compact-table policy still meets non-GridWorld callers (twr_policy_forward_obs): those run the fp32 kernel
        PolicyDev full = probe;
        full.compact_n = 0;
        if ((!use_tc || p->dev.compact_n > 0) && !forward_fp32_supported(full, max_obs, &why) && !big_board) {
            if (!use_tc) {
                delete p;
                return fail(TWR_ERR_UNSUPPORTED, std::string("policy shape not supported on the device: ") + why);
            }
            use_tc = false;
        }
        if (!use_tc) p->dev.compact_n = 0;
    } else if (max_width > 1024) {
        delete p;
        return fail(TWR_ERR_UNSUPPORTED, "general layer stacks are implemented for layer widths up to 1024");
    }
    if ((rc = dev_alloc(&p->d_blob, (size_t)p->blob_floats))) { delete p; return rc; }
    if (d->n_perms > 0) {
        if ((rc = dev_alloc(&p->d_obs_perms, (size_t)d->n_perms * d->obs_size)) ||
            (rc = dev_alloc(&p->d_act_perms, (size_t)d->n_perms * A))) { twr_policy_destroy(p); return rc; }
    }
    p->dev.emb = p->d_blob; p->dev.emb_b = p->d_blob + p->off_emb_b;
    for (size_t i = 0; i < lins.size(); ++i)
        p->dev.lin[i] = PolicyDev::Lin{p->d_blob + p->off_w[i], p->d_blob + p->off_b[i], lins[i]->in, lins[i]->out, lins[i]->apply_relu ? 1 : 0};
    if (standard) {          // the tile kernels' named views of the same blob
        p->dev.w1 = p->dev.lin[0].w; p->dev.b1 = p->dev.lin[0].b;
        p->dev.wa = p->dev.lin[1].w; p->dev.ba = p->dev.lin[1].b;
        p->dev.wv = p->dev.lin[2].w; p->dev.bv = p->dev.lin[2].b;
    }
    p->dev.obs_perms = p->d_obs_perms; p->dev.act_perms = p->d_act_perms;
    if (use_tc) {
        const size_t bytes = forward_tc2_pack_bytes(p->dev);
        cudaError_t ce = cudaMalloc(&p->tc_pack, bytes);
        if (ce != cudaSuccess) { twr_policy_destroy(p); return fail(TWR_ERR_CUDA, cudaGetErrorString(ce)); }
        p->dev.tc_pack = p->tc_pack;
    }
    if ((rc = upload_policy(p, d))) { twr_policy_destroy(p); return rc; }
    if (use_tc && !forward_tc2_prepare(p->dev, p->tc_pack)) {
        twr_policy_destroy(p);
        return fail(TWR_ERR_CUDA, "tensor-core forward: cuTensorMapEncodeTiled / kernel attributes unavailable on this device or driver");
    }
    *out = p;
    return TWR_OK;
    });
}

int twr_policy_update(twr_policy* p, const twr_policy_desc* d_in) {
    return twr_guard([&]() -> int {
    if (!p) return fail(TWR_ERR_INVALID, "policy is NULL");
    if (!d_in) return fail(TWR_ERR_INVALID, "policy desc / embedding is NULL");
    twr_policy_desc flat;
    std::vector<float> table;
    int rc = expand_conv1d(d_in, &flat, &table);
    if (rc) return rc;
    const twr_policy_desc* d = &flat;
    if ((rc = validate_desc(d))) return rc;
    CU_TRY(cudaSetDevice(p->eng->device));
    return upload_policy(p, d);
    });
}

int64_t twr_policy_blob_floats(const twr_policy* p) { return p ? p->blob_floats : 0; }

int twr_policy_blob_device_ptr(twr_policy* p, float** d_blob) {
    if (!p || !d_blob) return fail(TWR_ERR_INVALID, "policy/out is NULL");
    *d_blob = p->d_blob;
    return TWR_OK;
}

int twr_policy_update_from_device(twr_policy* p, const float* d_src) {
    if (!p || !d_src) return fail(TWR_ERR_INVALID, "policy/blob is NULL");
    twr_engine* e = p->eng;
    CU_TRY(cudaSetDevice(e->device));
    if (d_src != p->d_blob)
        CU_TRY(cudaMemcpyAsync(p->d_blob, d_src, sizeof(float) * (size_t)p->blob_floats, cudaMemcpyDeviceToDevice, e->stream));
    if (p->tc_pack) launch_forward_tc2_pack(e->stream, p->dev, p->tc_pack);
    CU_TRY(cudaGetLastError());
    return TWR_OK;
}

void twr_policy_destroy(twr_policy* p) {
    if (!p) return;
    cudaSetDevice(p->eng->device);
    cudaStreamSynchronize(p->eng->stream);
    dev_free(p->d_blob); dev_free(p->d_obs_perms); dev_free(p->d_act_perms);
    if (p->tc_pack) { forward_tc2_forget(p->tc_pack); cudaFree(p->tc_pack); }
    delete p;
}

// ------------------------------------------------------------------ batched env ---
int twr_envs_create(twr_engine* e, const twr_env_spec* spec, int64_t n, twr_envs** out) {
    if (!e || !out) return fail(TWR_ERR_INVALID, "engine/out is NULL");
    *out = nullptr;
    if (n < 0) return fail(TWR_ERR_INVALID, "n must be >= 0");
    EnvParams p;
    int rc = check_spec(spec, &p);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(e->device));
    twr_envs* v = new twr_envs();
    v->eng = e; v->p = p; v->n = n;
    if ((rc = dev_alloc(&v->cells, (size_t)n)) || (rc = dev_alloc(&v->meta, (size_t)n))) { twr_envs_destroy(v); return rc; }
    launch_envs_fresh(e->stream, p, v->cells, v->meta, n);
    CU_TRY(cudaGetLastError());
    *out = v;
    return TWR_OK;
}

void twr_envs_destroy(twr_envs* v) {
    if (!v) return;
    cudaSetDevice(v->eng->device);
    cudaStreamSynchronize(v->eng->stream);
    dev_free(v->cells); dev_free(v->meta);
    delete v;
}

int twr_envs_set_difficulty(twr_envs* v, int32_t difficulty) {
    if (!v) return fail(TWR_ERR_INVALID, "envs is NULL");
    if (difficulty < 0) return fail(TWR_ERR_INVALID, "difficulty must be >= 0");
    if (v->p.kind == TWR_ENV_GRIDWORLD) {
        const int cap = v->p.W + v->p.H;
        v->p.difficulty = difficulty < cap ? difficulty : cap;
    } else {
        if ((int64_t)v->p.depth_slope * difficulty >= (1 << 24)) return fail(TWR_ERR_INVALID, "depth budget too large");
        v->p.difficulty = difficulty;
    }
    return TWR_OK;
}

int twr_envs_set_state(twr_envs* v, const int64_t* states) {
    return twr_guard([&]() -> int {
    if (!v || !states) return fail(TWR_ERR_INVALID, "envs/states is NULL");
    if (v->n == 0) return TWR_OK;
    const int N = v->p.N;
    // the reference indexes its tables with these values and panics on anything else (puzzle.rs:99-117, lib.rs:100-112);
    // here an out-of-range cell would index past the embedding table on the device, so it is rejected up front
    const int64_t vmax = v->p.kind == TWR_ENV_PUZZLE ? N - 1 : 3;
    for (int64_t i = 0; i < v->n * N; ++i)
        if (states[i] < 0 || states[i] > vmax)
            return fail(TWR_ERR_INVALID, v->p.kind == TWR_ENV_PUZZLE ? "set_state: Puzzle cell values must be tiles 0..cells-1"
                                                                     : "set_state: GridWorld cell values must be 0 (empty), 1 (agent), 2 (goal) or 3 (trap)");
    if (v->p.kind == TWR_ENV_PUZZLE) {
        for (int64_t e = 0; e < v->n; ++e) {
            bool zero = false;
            for (int i = 0; i < N; ++i) zero |= states[e * N + i] == 0;
            if (!zero) return fail(TWR_ERR_INVALID, "set_state: a Puzzle board needs a blank (0) cell");
        }
    }
    twr_engine* e = v->eng;
    CU_TRY(cudaSetDevice(e->device));
    Staging<int64_t> st;
    int rc = st.alloc((size_t)v->n * N);
    if (rc) return rc;
    CU_TRY(cudaMemcpyAsync(st.d, states, sizeof(int64_t) * (size_t)v->n * N, cudaMemcpyHostToDevice, e->stream));
    launch_envs_set_state(e->stream, v->p, v->cells, v->meta, v->n, st.d);
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
    });
}

int twr_envs_set_cell(twr_envs* v, int64_t env, int32_t cell, int32_t value) {
    if (!v) return fail(TWR_ERR_INVALID, "envs is NULL");
    if (v->p.kind != TWR_ENV_PUZZLE) return fail(TWR_ERR_UNSUPPORTED, "set_cell is Puzzle::set_position; GridWorld has no such method");
    if (env < 0 || env >= v->n || cell < 0 || cell >= v->p.N) return fail(TWR_ERR_INVALID, "set_cell: env / cell index out of range");
    if (value < 0 || value >= v->p.N) return fail(TWR_ERR_INVALID, "set_cell: Puzzle cell values must be tiles 0..cells-1");
    twr_engine* e = v->eng;
    CU_TRY(cudaSetDevice(e->device));
    // one cell of the env's board, rewritten in the board's encoding; blank index and depth stay as they are (puzzle.rs:71-73)
    uint4 c;
    CU_TRY(cudaMemcpyAsync(&c, v->cells + env, sizeof(c), cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    EnvState s = env_from_cells(c);
    cell_set(s, cell, (uint32_t)value, cells_wide(v->p));
    c = env_pack_cells(s);
    CU_TRY(cudaMemcpyAsync(v->cells + env, &c, sizeof(c), cudaMemcpyHostToDevice, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
}

int twr_envs_reset(twr_envs* v, uint32_t env_id_base, uint32_t collect_id) {
    if (!v) return fail(TWR_ERR_INVALID, "envs is NULL");
    if (v->p.kind == TWR_ENV_GRIDWORLD && v->p.difficulty < 1)
        return fail(TWR_ERR_INVALID, "GridWorld reset needs difficulty >= 1 (the reference loops forever at 0)");
    twr_engine* e = v->eng;
    CU_TRY(cudaSetDevice(e->device));
    launch_envs_reset(e->stream, v->p, v->cells, v->meta, v->n, e->seed, EnvIds{env_id_base, 0u, 0u}, collect_id, nullptr, nullptr);
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
}

int twr_envs_step(twr_envs* v, const int32_t* actions) {
    if (!v || !actions) return fail(TWR_ERR_INVALID, "envs/actions is NULL");
    if (v->n == 0) return TWR_OK;
    twr_engine* e = v->eng;
    CU_TRY(cudaSetDevice(e->device));
    Staging<int32_t> st;
    int rc = st.alloc((size_t)v->n);
    if (rc) return rc;
    CU_TRY(cudaMemcpyAsync(st.d, actions, sizeof(int32_t) * (size_t)v->n, cudaMemcpyHostToDevice, e->stream));
    launch_envs_step(e->stream, v->p, v->cells, v->meta, v->n, st.d);
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
}

int twr_envs_get_state(twr_envs* v, int64_t* states) { return query_field<int64_t>(v, states, v ? v->p.N : 0, 0); }
int twr_envs_observe(twr_envs* v, int32_t* obs) { return query_field<int32_t>(v, obs, v ? v->p.N : 0, 1); }
int twr_envs_masks(twr_envs* v, uint8_t* masks) { return query_field<uint8_t>(v, masks, TWR_MAX_ACTIONS, 2); }
int twr_envs_reward(twr_envs* v, float* r) { return query_field<float>(v, r, 1, 3); }
int twr_envs_is_final(twr_envs* v, uint8_t* f) { return query_field<uint8_t>(v, f, 1, 4); }
int twr_envs_success(twr_envs* v, uint8_t* s) { return query_field<uint8_t>(v, s, 1, 5); }
int twr_envs_depth(twr_envs* v, int32_t* d) { return query_field<int32_t>(v, d, 1, 6); }

// -------------------------------------------------------------------- forward ---
// The policy as one forward runs it, over envs `env` or (env NULL) the n rows of n_obs indices in `obs`: tc_pack cleared,
// so the fp32 kernel runs, for a compact-table policy outside GridWorld envs of its size, or a row that repeats an index
// (the one-hot GEMM operand cannot express one).  The fp32 kernel stages the compact table for GridWorld boards above
// 32 cells; a forward whose table or rows it cannot hold in shared memory runs the generic kernel, which reads the
// table from global memory.
static PolicyDev call_dev(const twr_policy* p, const EnvParams* env, const int32_t* obs, int64_t n, int n_obs) {
    const PolicyDev& pol = p->dev;
    PolicyDev dev = pol;
    dev.n_obs = env ? env->N : n_obs;
    const bool grid = env && env->kind == TWR_ENV_GRIDWORLD && env->N == p->grid_n;
    bool tc = pol.tc_pack && (pol.compact_n == 0 || grid);
    for (int64_t i = 0; tc && obs && i < n; ++i)
        for (int a = 0; tc && a < n_obs; ++a)
            for (int b = a + 1; tc && b < n_obs; ++b) tc = obs[i * n_obs + a] != obs[i * n_obs + b];
    if (!tc) {
        dev.tc_pack = nullptr;
        dev.compact_n = grid && env->N > TWR_MAX_CELLS ? env->N : 0;
        const char* why = "";
        if (!dev.generic && !forward_fp32_supported(dev, dev.n_obs, &why)) dev.generic = 1;
    }
    return dev;
}

static int check_policy_env(const twr_policy* p, const EnvParams& env, PolicyDev* dev) {
    if (p->dev.obs_size != env.N * env.N)
        return fail(TWR_ERR_INVALID, "policy obs_size does not match the env's obs_shape (cells*cells)");
    if (p->dev.A != 4) return fail(TWR_ERR_INVALID, "policy has " + std::to_string(p->dev.A) + " actions, env has 4");
    *dev = call_dev(p, &env, nullptr, 0, 0);
    return TWR_OK;
}

// what every forward sets: its envs, its twist-pick stream (t = -1 outside a rollout) and its outputs
static ForwardArgs forward_args(const twr_engine* e, const EnvParams& env, uint32_t cid, EnvIds ids, const uint4* cells,
                                int64_t n, float4* logits, float* values) {
    ForwardArgs a{};
    a.env = env; a.seed = e->seed; a.cid = cid; a.ids = ids; a.t = -1;
    a.cells = cells; a.n = n; a.logits = logits; a.values = values;
    return a;
}

static void launch_forward(twr_engine* e, const PolicyDev& dev, const ForwardArgs& a) {
    bool ok = true;
    if (dev.generic) launch_forward_generic(e->stream, dev, a);   // general layer stacks (f4)
    else if (dev.tc_pack) {                                       // policies whose shape fits the tensor-core kernel (f16x2 engines)
        ForwardArgs t = a;
        t.tc_terms = e->tc_terms;
        t.dbg_flags |= e->tc_flags;
        ok = launch_forward_tc2(e->stream, dev, t, dev.tc_pack);
    } else ok = launch_forward_fp32(e->stream, dev, a);
    if (!ok) e->launch_error = true;
}
// after the launches of a call: a launch error or an unlaunched forward must not look like success (no records, TWR_OK)
#define FWD_CHECK(e)                                                                                          \
    do {                                                                                                      \
        CU_TRY(cudaGetLastError());                                                                           \
        if ((e)->launch_error) {                                                                              \
            (e)->launch_error = false;                                                                        \
            return fail(TWR_ERR_CUDA, "policy forward kernel could not be launched (shape / shared memory / tensor map)"); \
        }                                                                                                     \
    } while (0)

// A forward whose results go back to the caller: outputs for `slices` x n rows (full_predict: one slice per twist) and
// the caller's perm_idx (NULL: Philox pick), range-checked before anything is allocated.
struct HostForward {
    Staging<float4> logits; Staging<float> values; Staging<int32_t> perm;
    int64_t n = 0;
    int stage(twr_engine* e, const PolicyDev& dev, const EnvParams& env, const uint4* cells, int64_t rows, size_t slices,
              const int32_t* perm_idx, ForwardArgs* a) {
        if (perm_idx)
            for (int64_t i = 0; i < rows; ++i)
                if (perm_idx[i] < -1 || perm_idx[i] >= dev.n_perms) return fail(TWR_ERR_INVALID, "perm_idx out of range");
        CU_TRY(cudaSetDevice(e->device));
        n = rows;
        int rc;
        if ((rc = logits.alloc(slices * (size_t)n)) || (rc = values.alloc(slices * (size_t)n))) return rc;
        if (perm_idx) {
            if ((rc = perm.alloc((size_t)n))) return rc;
            CU_TRY(cudaMemcpyAsync(perm.d, perm_idx, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, e->stream));
        }
        *a = forward_args(e, env, 0, EnvIds{}, cells, n, logits.d, values.d);
        a->perm_idx = perm.d;
        return TWR_OK;
    }
    // after FWD_CHECK: logits as [n][A] and values to the host
    int to_host(twr_engine* e, int A, float* h_logits, float* h_values) {
        std::vector<float4> h((size_t)n);
        CU_TRY(cudaMemcpyAsync(h.data(), logits.d, sizeof(float4) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
        CU_TRY(cudaMemcpyAsync(h_values, values.d, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
        CU_TRY(cudaStreamSynchronize(e->stream));
        for (int64_t i = 0; i < n; ++i) {
            const float l[4] = {h[i].x, h[i].y, h[i].z, h[i].w};
            for (int k = 0; k < A; ++k) h_logits[i * A + k] = l[k];
        }
        return TWR_OK;
    }
};

int twr_policy_forward(twr_engine* e, const twr_policy* p, twr_envs* v, const int32_t* perm_idx, int32_t apply_masks,
                       float* logits, float* values) {
    return twr_guard([&]() -> int {
    if (!e || !p || !v || !logits || !values) return fail(TWR_ERR_INVALID, "NULL argument");
    if (p->eng != e || v->eng != e) return fail(TWR_ERR_INVALID, "policy/envs belong to another engine");
    if (v->n == 0) return TWR_OK;
    PolicyDev dev;
    int rc = check_policy_env(p, v->p, &dev);
    if (rc) return rc;
    HostForward f;
    ForwardArgs a;
    if ((rc = f.stage(e, dev, v->p, v->cells, v->n, 1, perm_idx, &a))) return rc;
    launch_forward(e, dev, a);
    if (apply_masks) launch_mask_logits(e->stream, v->p, v->cells, v->meta, v->n, dev.A, a.logits);
    FWD_CHECK(e);
    return f.to_host(e, dev.A, logits, values);
    });
}

int twr_debug_forward_profile(twr_engine* e, const twr_policy* p, twr_envs* v, int64_t* counters, int32_t max_ctas, int32_t flags) {
    return twr_guard([&]() -> int {
    if (!e || !p || !v || !counters) return fail(TWR_ERR_INVALID, "NULL argument");
    PolicyDev dev;
    int rc = check_policy_env(p, v->p, &dev);
    if (rc) return rc;
    if (max_ctas < TWR_DBG_CTAS + 16)
        return fail(TWR_ERR_INVALID, "counters buffer must hold " + std::to_string(TWR_DBG_CTAS) + "*16 + 256 int64");
    HostForward f;
    ForwardArgs a;
    Staging<long long> d_dbg;
    if ((rc = f.stage(e, dev, v->p, v->cells, v->n, 1, nullptr, &a)) || (rc = d_dbg.alloc(TWR_DBG_WORDS))) return rc;
    CU_TRY(cudaMemsetAsync(d_dbg.d, 0, sizeof(long long) * TWR_DBG_WORDS, e->stream));
    a.dbg = d_dbg.d; a.dbg_flags = flags;
    launch_forward(e, dev, a);
    FWD_CHECK(e);
    CU_TRY(cudaMemcpyAsync(counters, d_dbg.d, sizeof(long long) * TWR_DBG_WORDS, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
    });
}

int twr_debug_set_tc_terms(twr_engine* e, int32_t terms) {
    if (!e) return fail(TWR_ERR_INVALID, "engine is NULL");
    if (terms < -1 || (terms > 7 && terms != (16 | 3))) return fail(TWR_ERR_INVALID, "terms must be -1, a 3-bit mask, or 16|3");
    e->tc_terms = terms < 0 ? terms_of_precision(e->precision) : (8 | terms);
    return TWR_OK;
}

int twr_policy_forward_obs(twr_engine* e, const twr_policy* p, const int32_t* obs, int64_t n, int32_t n_obs,
                           const int32_t* perm_idx, float* logits, float* values) {
    return twr_guard([&]() -> int {
    if (!e || !p || !obs || !logits || !values) return fail(TWR_ERR_INVALID, "NULL argument");
    if (p->eng != e) return fail(TWR_ERR_INVALID, "policy belongs to another engine");
    if (n_obs < 1 || n_obs > TWR_MAX_OBS) return fail(TWR_ERR_UNSUPPORTED, "n_obs must be in 1..64");
    if (n <= 0) return TWR_OK;
    for (int64_t i = 0; i < n * n_obs; ++i)
        if (obs[i] < 0 || obs[i] >= p->dev.obs_size) return fail(TWR_ERR_INVALID, "observation index out of range");
    // one index per block of tc_fold rows? (then the bias-folded f16f8c image applies to these observations too)
    bool blocks = p->dev.tc_fold > 0 && n_obs == p->dev.tc_fold;
    for (int64_t i = 0; blocks && i < n; ++i) {
        uint64_t seen = 0;
        for (int a2 = 0; a2 < n_obs; ++a2) seen |= 1ull << (obs[i * n_obs + a2] / p->dev.tc_fold);
        blocks = seen == (n_obs >= 64 ? ~0ull : (1ull << n_obs) - 1);
    }
    const PolicyDev dev = call_dev(p, nullptr, obs, n, n_obs);
    EnvParams obs_env{};                     // only the index count: the rows are given, not read from env state
    obs_env.N = n_obs;
    HostForward f;
    ForwardArgs a;
    Staging<int32_t> d_obs;
    int rc;
    if ((rc = f.stage(e, dev, obs_env, nullptr, n, 1, perm_idx, &a)) || (rc = d_obs.alloc((size_t)n * n_obs))) return rc;
    CU_TRY(cudaMemcpyAsync(d_obs.d, obs, sizeof(int32_t) * (size_t)n * n_obs, cudaMemcpyHostToDevice, e->stream));
    a.obs_rows = d_obs.d; a.obs_blocks = blocks ? 1 : 0;
    launch_forward(e, dev, a);
    FWD_CHECK(e);
    return f.to_host(e, dev.A, logits, values);
    });
}

int twr_sample(twr_engine* e, const float* logits, int64_t n, int32_t A, uint32_t env_id_base, uint32_t step,
               uint32_t collect_id, int32_t* actions, float* uniforms_out) {
    return twr_guard([&]() -> int {
    if (!e || !logits || !actions) return fail(TWR_ERR_INVALID, "NULL argument");
    if (A < 1 || A > TWR_MAX_ACTIONS) return fail(TWR_ERR_UNSUPPORTED, "num_actions must be 1..4");
    if (n <= 0) return TWR_OK;
    CU_TRY(cudaSetDevice(e->device));
    Staging<float> d_l, d_u; Staging<int32_t> d_a;
    int rc;
    if ((rc = d_l.alloc((size_t)n * A)) || (rc = d_a.alloc((size_t)n)) || (rc = d_u.alloc((size_t)n * A))) return rc;
    CU_TRY(cudaMemcpyAsync(d_l.d, logits, sizeof(float) * (size_t)n * A, cudaMemcpyHostToDevice, e->stream));
    launch_sample(e->stream, d_l.d, n, A, e->seed, env_id_base, step, collect_id, d_a.d, d_u.d);
    CU_TRY(cudaMemcpyAsync(actions, d_a.d, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    if (uniforms_out)
        CU_TRY(cudaMemcpyAsync(uniforms_out, d_u.d, sizeof(float) * (size_t)n * A, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
    });
}

int twr_gae(twr_engine* e, const float* rewards, const float* values, const int64_t* offsets, int64_t n_ep, float gamma,
            float lambda, float* advs, float* rets) {
    return twr_guard([&]() -> int {
    if (!e || !rewards || !values || !offsets || !advs || !rets) return fail(TWR_ERR_INVALID, "NULL argument");
    if (n_ep <= 0) return TWR_OK;
    const int64_t R = offsets[n_ep];
    for (int64_t i = 0; i < n_ep; ++i)
        if (offsets[i] > offsets[i + 1] || offsets[i] < 0) return fail(TWR_ERR_INVALID, "offsets must be non-decreasing");
    if (R == 0) return TWR_OK;
    CU_TRY(cudaSetDevice(e->device));
    Staging<float> d_r, d_v, d_a, d_t; Staging<int64_t> d_o;
    int rc;
    if ((rc = d_r.alloc((size_t)R)) || (rc = d_v.alloc((size_t)R)) || (rc = d_a.alloc((size_t)R)) ||
        (rc = d_t.alloc((size_t)R)) || (rc = d_o.alloc((size_t)n_ep + 1))) return rc;
    CU_TRY(cudaMemcpyAsync(d_r.d, rewards, sizeof(float) * (size_t)R, cudaMemcpyHostToDevice, e->stream));
    CU_TRY(cudaMemcpyAsync(d_v.d, values, sizeof(float) * (size_t)R, cudaMemcpyHostToDevice, e->stream));
    CU_TRY(cudaMemcpyAsync(d_o.d, offsets, sizeof(int64_t) * (size_t)(n_ep + 1), cudaMemcpyHostToDevice, e->stream));
    launch_gae_concat(e->stream, d_r.d, d_v.d, d_o.d, n_ep, gamma, lambda, d_a.d, d_t.d);
    CU_TRY(cudaMemcpyAsync(advs, d_a.d, sizeof(float) * (size_t)R, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaMemcpyAsync(rets, d_t.d, sizeof(float) * (size_t)R, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
    });
}

// -------------------------------------------------------------------- collect ---
int64_t twr_max_records(const twr_env_spec* spec, int64_t num_episodes) {
    EnvParams p;
    if (check_spec(spec, &p)) return -1;
    return num_episodes * (int64_t)(horizon_of(p) + 1);
}

static void select_outset(twr_engine* e, int which) {
    CollectBuffers& b = e->buf;
    const twr_engine::OutSet& o = e->outs[which];
    b.out_obs = o.obs; b.out_logits = o.logits; b.out_values = o.values; b.out_rewards = o.rewards;
    b.out_advs = o.advs; b.out_rets = o.rets; b.out_actions = o.actions; b.out_perms = o.perms;
}

static int alloc_outset(twr_engine::OutSet* o, size_t R, int cells) {
    int rc;
    if ((rc = dev_alloc(&o->obs, R * cells)) || (rc = dev_alloc(&o->logits, R * TWR_MAX_ACTIONS)) ||
        (rc = dev_alloc(&o->values, R)) || (rc = dev_alloc(&o->rewards, R)) || (rc = dev_alloc(&o->advs, R)) ||
        (rc = dev_alloc(&o->rets, R)) || (rc = dev_alloc(&o->actions, R)) || (rc = dev_alloc(&o->perms, R))) return rc;
    return TWR_OK;
}

static int ensure_collect_buffers(twr_engine* e, int64_t B, int T, int cells, int64_t total_episodes) {
    if (total_episodes > e->cap_E) {
        CU_TRY(cudaStreamSynchronize(e->stream));
        dev_free(e->ep_len_id);
        int rc = dev_alloc(&e->ep_len_id, (size_t)total_episodes);
        if (rc) return rc;
        e->cap_E = total_episodes;
    }
    e->buf.ep_len_id = e->ep_len_id;
    if (B <= e->cap_B && T <= e->cap_T && cells <= e->cap_cells && B * T <= e->cap_R) {
        e->buf.B = B; e->buf.Tmax = T;
        return TWR_OK;
    }
    CU_TRY(cudaStreamSynchronize(e->stream));
    CU_TRY(cudaStreamSynchronize(e->copy_stream));
    free_collect_buffers(e);
    CollectBuffers& b = e->buf;
    const size_t R = (size_t)B * T;
    int rc;
    if ((rc = dev_alloc(&b.cells, (size_t)B)) || (rc = dev_alloc(&b.meta, (size_t)B)) ||
        (rc = dev_alloc(&b.live_a, (size_t)B)) || (rc = dev_alloc(&b.live_b, (size_t)B)) ||
        (rc = dev_alloc(&b.n_live, (size_t)T + 1)) || (rc = dev_alloc(&b.logits, (size_t)B)) ||
        (rc = dev_alloc(&b.values, (size_t)B)) || (rc = dev_alloc(&b.rec_state, R)) ||
        (rc = dev_alloc(&b.rec_logits, R)) || (rc = dev_alloc(&b.rec_value, R)) ||
        (rc = dev_alloc(&b.rec_reward, R)) || (rc = dev_alloc(&b.rec_adv, R)) || (rc = dev_alloc(&b.rec_ret, R)) ||
        (rc = dev_alloc(&b.rec_action, R)) || (rc = dev_alloc(&b.rec_perm, R)) ||
        (rc = dev_alloc(&b.ep_len, (size_t)B)) || (rc = dev_alloc(&b.ep_off, (size_t)B)) ||
        (rc = dev_alloc(&b.stats, 4))) {
        free_collect_buffers(e);
        return rc;
    }
    for (auto& o : e->outs) {
        if ((rc = alloc_outset(&o, R, cells))) {
            free_collect_buffers(e);
            return rc;
        }
    }
    e->cap_B = B; e->cap_T = T; e->cap_R = (int64_t)R; e->cap_cells = cells;
    b.B = B; b.Tmax = T;
    return TWR_OK;
}

int twr_ensure_merged_buffers(twr_engine* e, int64_t R, int64_t E, int n_cells) {
    if (E > e->cap_mE) {
        dev_free(e->merged_ep_len);
        e->cap_mE = 0;
        int rc = dev_alloc(&e->merged_ep_len, (size_t)E);
        if (rc) return rc;
        e->cap_mE = E;
    }
    if (R <= e->cap_mR && n_cells <= e->cap_mcells) return TWR_OK;
    free_outset(e->merged);
    e->cap_mR = 0; e->cap_mcells = 0;
    int rc = alloc_outset(&e->merged, (size_t)R, n_cells);
    if (rc) { free_outset(e->merged); return rc; }
    e->cap_mR = R; e->cap_mcells = n_cells;
    return TWR_OK;
}

static uint64_t hint_key_of(const EnvParams& p, int64_t B) {
    uint64_t k = 1469598103934665603ull;
    const int64_t f[] = {p.kind, p.W, p.H, p.difficulty, p.depth_slope, p.max_depth, B};
    for (int64_t v : f) { k ^= (uint64_t)v; k *= 1099511628211ull; }
    return k;
}

// the start of a collect of B episodes into output set `which`: its counters zeroed, every env reset and listed live
static int begin_collect(twr_engine* e, const EnvParams& env, int64_t B, EnvIds ids, uint32_t cid, int which) {
    CollectBuffers& b = e->buf;
    b.B = B;
    select_outset(e, which);
    CU_TRY(cudaMemsetAsync(b.n_live, 0, sizeof(int32_t) * (size_t)(b.Tmax + 1), e->stream));
    CU_TRY(cudaMemsetAsync(b.stats, 0, sizeof(unsigned long long) * 4, e->stream));
    launch_envs_reset(e->stream, env, b.cells, b.meta, B, e->seed, ids, cid, b.live_a, b.n_live);
    return TWR_OK;
}

// forward n_fwd of a collect, between its pair of timing events when timing is on (twr_engine_set_timing)
static void launch_forward_timed(twr_engine* e, const PolicyDev& dev, const ForwardArgs& a, int n_fwd) {
    const bool timed = e->timing && 2 * n_fwd + 1 < (int)e->ev.size();
    if (timed) cudaEventRecord(e->ev[2 * n_fwd], e->stream);
    launch_forward(e, dev, a);
    if (timed) cudaEventRecord(e->ev[2 * n_fwd + 1], e->stream);
}

// TWISTERL_B200_TRACE=<chunk index>: zeroed pipeline counters for that chunk's launch (one buffer per engine), else NULL
static long long* trace_counters(twr_engine* e, int ci) {
    static const char* trace_env = getenv("TWISTERL_B200_TRACE");
    if (!trace_env || ci != atoi(trace_env)) return nullptr;
    if (!e->trace_buf) cudaMalloc(reinterpret_cast<void**>(&e->trace_buf), sizeof(long long) * TWR_DBG_WORDS);
    cudaMemsetAsync(e->trace_buf, 0, sizeof(long long) * TWR_DBG_WORDS, e->stream);
    return e->trace_buf;
}

// the counters of the traced launch (chunk ci of cnt steps over B envs) on stderr, once it has run
static void print_trace(twr_engine* e, int ci, int cnt, int64_t B) {
    std::vector<long long> h(TWR_DBG_WORDS);
    cudaMemcpyAsync(h.data(), e->trace_buf, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost, e->stream);
    cudaStreamSynchronize(e->stream);
    static const char* names[16] = {"mma total", "mma wait slot", "mma wait a1_full", "mma wait a2_full", "mma wait d2_empty", "lanes",
                                    "mma slot wait G1", "mma slot wait G1 first", "producer wait empty", "epi total", "epi wait d1_full",
                                    "epi wait d2_full", "epi wait a1_empty", "epi1 busy", "build_a1", "epi2+step busy"};
    fprintf(stderr, "[trace] chunk %d, %d steps, %lld live envs\n", ci, cnt, (long long)B);
    for (int k = 0; k < 16; ++k) {
        double sum = 0; int n = 0; long long mx = 0;
        for (int c = 0; c < TWR_DBG_CTAS; ++c) { const long long v = h[(size_t)c * 16 + k]; if (v) { sum += (double)v; ++n; if (v > mx) mx = v; } }
        fprintf(stderr, "[trace] %-24s cta0 %10lld  mean(nonzero) %12.1f  max %10lld\n", names[k], h[k], n ? sum / n : 0.0, mx);
    }
    const long long* tr = h.data() + TWR_DBG_TRACE;
    for (int item = 0; item < 8; ++item) {
        fprintf(stderr, "[trace] item %d:", item);
        for (int ev = 0; ev < 27; ++ev) if (tr[item * 32 + ev]) fprintf(stderr, " %d@%lld", ev, tr[item * 32 + ev] - tr[0]);
        fprintf(stderr, "\n");
    }
}

// Enqueue one (sub-)collect of B local episodes on the engine stream: reset -> T x (forward [+ step]) -> GAE ->
// offsets -> compaction into output set `which`.  No host synchronisation.
static int enqueue_collect(twr_engine* e, const EnvParams& env, const PolicyDev& dev, int64_t B, EnvIds ids, uint32_t cid,
                           float gamma, float lambda, int which, int* n_fwd_out, cudaEvent_t outset_free = nullptr) {
    CollectBuffers& b = e->buf;
    cudaStream_t st = e->stream;
    const int T = b.Tmax;
    int rc = begin_collect(e, env, B, ids, cid, which);
    if (rc) return rc;

    StepArgs sa{};
    sa.env = env; sa.seed = e->seed; sa.cid = cid; sa.ids = ids; sa.n_perms = dev.n_perms; sa.A = dev.A;
    ForwardArgs fa = forward_args(e, env, cid, ids, b.cells, B, b.logits, b.values);
    const bool fused = dev.tc_pack != nullptr;            // the tensor-core kernel runs the collect step in its epilogue
    int n_fwd = *n_fwd_out;
    if (fused) {
        // Persistent chunks: one launch covers `chunk` consecutive steps of every tile (envs stay with their
        // CTA pair, finished envs idle), then the live list is re-compacted.  Short episodes use chunk 1.
        // (ceil(T / 8), ceil(T / 2): T = horizon + 1 is odd for even horizons, and a trailing 1-step launch costs 160 us
        // where a step inside a persistent launch costs 45)
        int chunk = (T + 7) / 8 > 64 ? 64 : (T + 7) / 8;
        // Adaptive: when the previous collect of this (env, batch) shape kept >= 90 % of its envs alive past half of the
        // horizon, compacting every T/8 steps buys nothing and the launches are made 4x longer (results are identical
        // for any chunking; a policy that starts to finish early flips the hint back after one collect)
        e->hint_key = hint_key_of(env, B);
        {
            auto it = e->survive_half.find(e->hint_key);
            if (it != e->survive_half.end() && it->second >= 0.9f) chunk = (T + 1) / 2 > 256 ? 256 : (T + 1) / 2;
        }
        if (const char* c = getenv("TWISTERL_B200_CHUNK")) { const int v = atoi(c); if (v >= 1) chunk = v; }
        int ci_half = -1;
        int bal_delta = e->bal_delta;
        if (const char* c = getenv("TWISTERL_B200_BALANCE")) bal_delta = atoi(c);   // 0 switches the time-split schedule off
        CU_TRY(cudaMemsetAsync(b.ep_len, 0, sizeof(int32_t) * (size_t)B, st));
        int32_t* cur = b.live_a;
        int32_t* nxt = b.live_b;
        for (int t0 = 0, ci = 0; t0 < T; t0 += chunk, ++ci) {
            const int cnt = T - t0 < chunk ? T - t0 : chunk;
            if (ci_half < 0 && 2 * t0 >= T) ci_half = ci;          // first compaction boundary in the second half of the horizon
            fa.t = t0; fa.t_count = cnt; fa.live = cur; fa.n_live_ptr = b.n_live + ci;
            sa.t = t0;
            fa.fused = 1; fa.step = sa; fa.cb = b; fa.live_next = cnt == 1 ? nxt : nullptr;
            if (cnt == 1) { fa.cb.n_live = b.n_live + ci - t0; }   // collect_step_body appends at n_live[t+1]
            fa.bal_flags = nullptr; fa.bal_delta = 0;
            if (cnt >= 4 && e->bal_flags && bal_delta > 0) {
                CU_TRY(cudaMemsetAsync(e->bal_flags, 0, 1024 * sizeof(int32_t), st));
                fa.bal_flags = e->bal_flags; fa.bal_delta = bal_delta;
            }
            fa.dbg = trace_counters(e, ci);
            launch_forward_timed(e, dev, fa, n_fwd++);
            if (fa.dbg) print_trace(e, ci, cnt, B);
            if (cnt > 1) launch_compact_live(st, cur, b.n_live + ci, b.ep_len, B, nxt, b.n_live + ci + 1);
            int32_t* tmp = cur; cur = nxt; nxt = tmp;
        }
        // envs still alive at that boundary -> stats[3] (read back with the other statistics; feeds the chunk hint)
        if (ci_half >= 0) CU_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(b.stats) + 24, b.n_live + ci_half, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        e->hint_B = ci_half >= 0 ? B : 0;
    } else {
        e->hint_B = 0;
        for (int t = 0; t < T; ++t) {
            int32_t* cur = (t & 1) ? b.live_b : b.live_a;
            int32_t* nxt = (t & 1) ? b.live_a : b.live_b;
            fa.t = t; fa.live = cur; fa.n_live_ptr = b.n_live + t;
            sa.t = t;
            launch_forward_timed(e, dev, fa, n_fwd++);
            launch_collect_step(st, sa, b, cur, nxt);
        }
    }
    *n_fwd_out = n_fwd;
    launch_episode_offsets(st, b, ids);
    // only the compaction writes the output set: a pipelined caller's "its previous copy is done" event is awaited here,
    // not in front of the rollout
    if (outset_free) CU_TRY(cudaStreamWaitEvent(st, outset_free, 0));
    launch_compact_gae(st, env, b, dev.A, gamma, lambda);      // GAE rides on the compaction (one pass over the records)
    FWD_CHECK(e);
    return TWR_OK;
}

struct CollectPlan { EnvParams env; PolicyDev dev; int T; };

static int plan_collect(twr_engine* e, const twr_env_spec* spec, const twr_policy* p, int64_t num_episodes, CollectPlan* plan) {
    if (!e || !p) return fail(TWR_ERR_INVALID, "NULL argument");
    if (p->eng != e) return fail(TWR_ERR_INVALID, "policy belongs to another engine");
    e->last_kind = twr_engine::LAST_NONE;     // a collect that fails, even on its arguments, leaves nothing to gather
    // merge() errors on zero chunks (collector/collector.rs:41)
    if (num_episodes <= 0)
        return fail(TWR_ERR_INVALID, "Something went wrong. No data in collected data chunks to merge. ");
    if (num_episodes >= (1ll << 31)) return fail(TWR_ERR_INVALID, "num_episodes too large");
    int rc = check_spec(spec, &plan->env);
    if (rc) return rc;
    if (plan->env.kind == TWR_ENV_GRIDWORLD && plan->env.difficulty < 1)
        return fail(TWR_ERR_INVALID, "GridWorld reset needs difficulty >= 1 (the reference loops forever at 0)");
    if ((rc = check_policy_env(p, plan->env, &plan->dev))) return rc;
    plan->T = horizon_of(plan->env) + 1;
    return TWR_OK;
}

// the statistics words launch_publish_stats wrote for the collect just synchronised ([2] holds a double)
struct CollectStats { int64_t successes, n_records; double reward_sum; };
static CollectStats read_stats(const twr_engine* e) {
    CollectStats s{(int64_t)e->h_stats[0], (int64_t)e->h_stats[1], 0.0};
    memcpy(&s.reward_sum, &e->h_stats[2], sizeof(double));
    return s;
}

// the output set a collect just compacted into, as a twr_collected's device pointers
static twr_collected outset_view(const CollectBuffers& b) {
    twr_collected c{};
    c.obs = b.out_obs; c.logits = b.out_logits; c.values = b.out_values; c.rewards = b.out_rewards;
    c.advs = b.out_advs; c.rets = b.out_rets; c.actions = b.out_actions; c.perms = b.out_perms;
    return c;
}

// the end of a device-resident collect: its statistics to the host, then its result kept for twr_collected_to_host
static int finish_collect(twr_engine* e, const CollectPlan& plan, int64_t num_episodes, int kind, const twr_env_spec* spec,
                          uint32_t cid, twr_collected* out) {
    launch_publish_stats(e->stream, e->buf.stats, e->d_hstats);
    CU_TRY(cudaStreamSynchronize(e->stream));
    const CollectStats s = read_stats(e);
    twr_collected& c = e->last;
    c = outset_view(e->buf);
    c.n_records = s.n_records; c.num_episodes = num_episodes; c.n_cells = plan.env.N; c.num_actions = plan.dev.A;
    c.successes = s.successes; c.reward_sum = s.reward_sum; c.ep_len = e->ep_len_id;
    e->has_last = true;
    e->last_kind = kind; e->last_spec = *spec; e->last_cid = cid;
    *out = c;
    return TWR_OK;
}

static void finish_timing(twr_engine* e, int n_fwd) {
    if (!e->timing) return;
    float tot = 0.f, ms = 0.f;
    const int n = n_fwd < (int)e->ev.size() / 2 ? n_fwd : (int)e->ev.size() / 2;
    for (int t = 0; t < n; ++t) { cudaEventElapsedTime(&ms, e->ev[2 * t], e->ev[2 * t + 1]); tot += ms; }
    e->last_fwd_ms = tot; e->last_fwd_launches = n;
    cudaEventElapsedTime(&e->last_total_ms, e->ev_t0, e->ev_t1);
}

int twr_ppo_collect(twr_engine* e, const twr_env_spec* spec, const twr_policy* p, int64_t num_episodes, float gamma,
                    float lambda, twr_collected* out) {
    return twr_guard([&]() -> int {
    if (!out) return fail(TWR_ERR_INVALID, "NULL argument");
    CollectPlan plan;
    int rc = plan_collect(e, spec, p, num_episodes, &plan);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(e->device));
    if ((rc = ensure_collect_buffers(e, num_episodes, plan.T, plan.env.N, num_episodes))) return rc;
    cudaStream_t st = e->stream;
    e->has_last = false;
    e->buf.obs_u8 = 0;
    const uint32_t cid = e->collect_id++;
    // local episode 0 is the LAST episode id, local i is episode i-1: local order == merge order
    const EnvIds ids{(uint32_t)((int64_t)e->rank * num_episodes), (uint32_t)(num_episodes - 1), (uint32_t)num_episodes};
    if (e->timing) {
        while ((int)e->ev.size() < 2 * (plan.T + 1)) { cudaEvent_t ev; cudaEventCreate(&ev); e->ev.push_back(ev); }
        cudaEventRecord(e->ev_t0, st);
    }
    int n_fwd = 0;
    if ((rc = enqueue_collect(e, plan.env, plan.dev, num_episodes, ids, cid, gamma, lambda, 0, &n_fwd))) return rc;
    if (e->timing) cudaEventRecord(e->ev_t1, st);
    if ((rc = finish_collect(e, plan, num_episodes, twr_engine::LAST_PPO, spec, cid, out))) return rc;
    e->note_survival();
    finish_timing(e, n_fwd);
    return TWR_OK;
    });
}

// D2H of the R records `src` points at into dst, at record offset `at`
static int copy_out(cudaStream_t st, const twr_collected& src, const twr_host_buffers* dst, int64_t at, size_t R, int n_cells, int A) {
    if (dst->obs) CU_TRY(cudaMemcpyAsync(dst->obs + at * n_cells, src.obs, sizeof(uint16_t) * R * n_cells, cudaMemcpyDeviceToHost, st));
    else if (dst->obs_u8) CU_TRY(cudaMemcpyAsync(dst->obs_u8 + at * n_cells, src.obs, R * n_cells, cudaMemcpyDeviceToHost, st));
    if (dst->logits) CU_TRY(cudaMemcpyAsync(dst->logits + at * A, src.logits, sizeof(float) * R * A, cudaMemcpyDeviceToHost, st));
    if (dst->values) CU_TRY(cudaMemcpyAsync(dst->values + at, src.values, sizeof(float) * R, cudaMemcpyDeviceToHost, st));
    if (dst->rewards) CU_TRY(cudaMemcpyAsync(dst->rewards + at, src.rewards, sizeof(float) * R, cudaMemcpyDeviceToHost, st));
    if (dst->advs) CU_TRY(cudaMemcpyAsync(dst->advs + at, src.advs, sizeof(float) * R, cudaMemcpyDeviceToHost, st));
    if (dst->rets) CU_TRY(cudaMemcpyAsync(dst->rets + at, src.rets, sizeof(float) * R, cudaMemcpyDeviceToHost, st));
    if (dst->actions) CU_TRY(cudaMemcpyAsync(dst->actions + at, src.actions, R, cudaMemcpyDeviceToHost, st));
    if (dst->perms) CU_TRY(cudaMemcpyAsync(dst->perms + at, src.perms, R, cudaMemcpyDeviceToHost, st));
    return TWR_OK;
}

int twr_collected_to_host(twr_engine* e, const twr_host_buffers* dst) {
    return twr_guard([&]() -> int {
    if (!e || !dst) return fail(TWR_ERR_INVALID, "NULL argument");
    if (!e->has_last) return fail(TWR_ERR_STATE, "twr_collected_to_host: no collect has run on this engine");
    const twr_collected& c = e->last;
    const size_t R = (size_t)c.n_records;
    if ((int64_t)R > dst->capacity) return fail(TWR_ERR_INVALID, "host buffers too small for the collected records");
    if (!dst->obs && dst->obs_u8)
        return fail(TWR_ERR_UNSUPPORTED, "obs_u8 is produced by twr_ppo_collect_host only (the device-resident result holds u16 indices)");
    CU_TRY(cudaSetDevice(e->device));
    cudaStream_t st = e->stream;
    int rc = copy_out(st, c, dst, 0, R, c.n_cells, c.num_actions);    // what `last` describes: root's merged result after a gather
    if (rc) return rc;
    if (dst->ep_len) CU_TRY(cudaMemcpyAsync(dst->ep_len, c.ep_len, sizeof(int32_t) * (size_t)c.num_episodes, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return TWR_OK;
    });
}

// End-to-end collect with host buffers.  Large collects are split into sub-batches of consecutive local episodes so
// that the D2H copy of sub-batch k (copy stream) overlaps the rollout of sub-batch k+1.  For Puzzle envs the copy is
// 41 instead of 50 bytes per record: action, twist index and the three-valued reward cross PCIe as ONE byte and the
// advantages not at all (advs = rets - values, the very f32 subtraction of collector/ppo.rs:87-91); host threads
// rebuild the caller's rewards / advs / actions / perms arrays per sub-batch while later sub-batches roll out.
// Host side of CollectBuffers::pack_misc for records [a, b): `actions` holds action | reward code << 2 | (perm + 1) << 4;
// blocked so that every loop is a plain element-wise pass the host compiler vectorises.
static void expand_packed(uint8_t* __restrict__ actions, int8_t* __restrict__ perms, float* __restrict__ rewards, float* __restrict__ advs,
                          const float* __restrict__ rets, const float* __restrict__ values, float r_step, int64_t a, int64_t b) {
    constexpr int BK = 512;
    uint8_t m[BK];
    for (int64_t i0 = a; i0 < b; i0 += BK) {
        const int n = (int)std::min<int64_t>(BK, b - i0);
        memcpy(m, actions + i0, (size_t)n);
        for (int i = 0; i < n; ++i) actions[i0 + i] = (uint8_t)(m[i] & 3u);
        if (perms) for (int i = 0; i < n; ++i) perms[i0 + i] = (int8_t)((int)(m[i] >> 4) - 1);
        if (rewards)
            for (int i = 0; i < n; ++i) {
                const int c = (m[i] >> 2) & 3;
                rewards[i0 + i] = c == 2 ? 1.0f : (c == 1 ? -0.5f : r_step);       // puzzle.rs:171-177
            }
        if (advs) for (int i = 0; i < n; ++i) advs[i0 + i] = rets[i0 + i] - values[i0 + i];   // ppo.rs:87-91
    }
}

static std::vector<int64_t> host_collect_parts(twr_engine* e, int64_t num_episodes) {
    std::vector<int64_t> parts;
    if (const char* ps = getenv("TWISTERL_B200_E2E_PARTS")) {         // explicit sizes "a,b,c" (must sum to num_episodes)
        int64_t sum = 0;
        for (const char* q = ps; *q;) { char* end; const long long v = strtoll(q, &end, 10); if (end == q || v <= 0) break; parts.push_back(v); sum += v; q = *end ? end + 1 : end; }
        if (sum == num_episodes) return parts;
        parts.clear();
    }
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device);
    const int64_t round = (int64_t)(sms / 2) * 256;      // envs the pair kernel works on at once
    if (num_episodes < 32768 || e->precision == TWR_PREC_FP32 || round <= 0) { parts.push_back(num_episodes); return parts; }
    // Sub-batches of two kernel rounds -- the smallest shape the pair kernel runs at full rate (one round is a serial
    // chain of one tile per SM pair: 18 944 envs take 4.9 ms, 37 888 take 6.9 ms) -- and the remainder last, whose copy is
    // the exposed tail.  Measured on 65 536 envs (scripts/e2e_sweep.py): any finer or front-loaded split is slower.
    int64_t rem = num_episodes;
    while (rem > 2 * round) { parts.push_back(2 * round); rem -= 2 * round; }
    if (rem > 0) parts.push_back(rem);
    return parts;
}

int twr_ppo_collect_host(twr_engine* e, const twr_env_spec* spec, twr_policy* p, const twr_policy_desc* desc,
                         int64_t num_episodes, float gamma, float lambda, const twr_host_buffers* dst, twr_collected* out) {
    return twr_guard([&]() -> int {
    if (!e || !p || !dst || !out) return fail(TWR_ERR_INVALID, "NULL argument");
    int rc;
    if (desc && (rc = twr_policy_update(p, desc))) return rc;
    CollectPlan plan;
    if ((rc = plan_collect(e, spec, p, num_episodes, &plan))) return rc;
    const bool u8 = !dst->obs && dst->obs_u8;
    if (u8 && plan.dev.obs_size > 256) return fail(TWR_ERR_INVALID, "obs_u8 needs obs_size <= 256");
    CU_TRY(cudaSetDevice(e->device));
    const std::vector<int64_t> parts = host_collect_parts(e, num_episodes);
    if (parts.size() == 1 && !u8) {
        if ((rc = twr_ppo_collect(e, spec, p, num_episodes, gamma, lambda, out))) return rc;
        return twr_collected_to_host(e, dst);
    }
    if (parts.size() > TWR_MAX_SUBBATCH) return fail(TWR_ERR_INVALID, "too many sub-batches");
    int64_t Bmax = 0;
    for (int64_t v : parts) Bmax = v > Bmax ? v : Bmax;
    if ((rc = ensure_collect_buffers(e, Bmax, plan.T, plan.env.N, num_episodes))) return rc;
    // one byte for action / reward / twist when they fit: Puzzle rewards (three values) and at most 14 twists
    const bool pack = plan.env.kind == TWR_ENV_PUZZLE && plan.dev.n_perms <= 14 && dst->actions && (!dst->advs || (dst->rets && dst->values));
    const float reward_of_code[4] = {-0.5f / (float)plan.env.max_depth, -0.5f, 1.0f, 0.0f};     // puzzle.rs:171-177
    e->has_last = false;
    const uint32_t cid = e->collect_id++;
    const uint32_t base = (uint32_t)((int64_t)e->rank * num_episodes);
    int64_t at = 0, successes = 0, lo = 0;
    double reward_sum = 0.0;
    int n_fwd = 0;
    const bool timing = e->timing;
    e->timing = false;                                  // per-forward events are only kept for the device-resident path
    e->buf.obs_u8 = u8 ? 1 : 0;
    e->buf.pack_misc = pack ? 1 : 0;
    std::vector<std::thread> stages;                    // one per sub-batch: waits for its copy, then rebuilds the packed fields
    std::vector<std::function<void()>> deferred;        // stages whose thread could not be started: run on this thread at the end
    // TWISTERL_B200_E2E_TRACE=1: host-clock milestones of every sub-batch on stderr (ms since the call started)
    const bool trace = getenv("TWISTERL_B200_E2E_TRACE") != nullptr;
    const auto t_call = std::chrono::steady_clock::now();
    auto now_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count(); };
    std::vector<double> tr_enq, tr_done, tr_exp(parts.size(), 0.0);
    std::vector<size_t> tr_R;
    int hw = (int)std::thread::hardware_concurrency();
    int workers = hw / (2 * (e->world > 0 ? e->world : 1));
    workers = workers < 1 ? 1 : (workers > 16 ? 16 : workers);
    auto body = [&]() -> int {
        for (size_t k = 0; k < parts.size(); ++k) {
            const int64_t B = parts[k];
            const int which = (int)(k & 1);
            // global local index = lo + i; episode id = (lo + i + E - 1) mod E
            const EnvIds ids{base, (uint32_t)((lo + num_episodes - 1) % num_episodes), (uint32_t)num_episodes};
            int r2 = enqueue_collect(e, plan.env, plan.dev, B, ids, cid, gamma, lambda, which, &n_fwd,
                                     k >= 2 ? e->ev_copied[k - 2] : nullptr);        // output set `which` free again
            if (r2) return r2;
            if (trace) tr_enq.push_back(now_ms());
            launch_publish_stats(e->stream, e->buf.stats, e->d_hstats);
            CU_TRY(cudaEventRecord(e->ev_done[which], e->stream));
            CU_TRY(cudaStreamSynchronize(e->stream));       // record count of this sub-batch -> host offsets
            FWD_CHECK(e);
            e->note_survival();
            const CollectStats s = read_stats(e);
            const size_t R = (size_t)s.n_records;
            if (trace) { tr_done.push_back(now_ms()); tr_R.push_back(R); }
            successes += s.successes;
            reward_sum += s.reward_sum;
            if (at + (int64_t)R > dst->capacity) return fail(TWR_ERR_INVALID, "host buffers too small for the collected records");
            CU_TRY(cudaStreamWaitEvent(e->copy_stream, e->ev_done[which], 0));
            const twr_collected part = outset_view(e->buf);
            if (pack) {
                // the 9 bytes per record the host rebuild reads go first, so that it overlaps the bulk (obs, logits) of the
                // same sub-batch instead of trailing the last copy
                twr_host_buffers d2{};
                d2.values = dst->values; d2.rets = dst->rets; d2.actions = dst->actions;
                if ((r2 = copy_out(e->copy_stream, part, &d2, at, R, plan.env.N, plan.dev.A))) return r2;
                CU_TRY(cudaEventRecord(e->ev_small[k], e->copy_stream));
                twr_host_buffers d3{};
                d3.logits = dst->logits; d3.obs = dst->obs; d3.obs_u8 = dst->obs_u8;
                if ((r2 = copy_out(e->copy_stream, part, &d3, at, R, plan.env.N, plan.dev.A))) return r2;
            } else if ((r2 = copy_out(e->copy_stream, part, dst, at, R, plan.env.N, plan.dev.A))) return r2;
            CU_TRY(cudaEventRecord(e->ev_copied[k], e->copy_stream));
            if (pack) {
                cudaEvent_t ev = e->ev_small[k];
                const int dev_id = e->device;
                const int64_t at0 = at;
                const twr_host_buffers d = *dst;
                const float* rtab = reward_of_code;
                double* t_exp = trace ? &tr_exp[k] : nullptr;
                // the rebuild of one sub-batch; a thread that cannot be started (resource limits) is run inline instead --
                // no C++ exception may leave through the C boundary
                auto stage = [ev, dev_id, at0, R, d, rtab, workers, t_exp, t_call]() {
                    cudaSetDevice(dev_id);
                    cudaEventSynchronize(ev);
                    auto span = [&](int64_t a, int64_t b) { expand_packed(d.actions, d.perms, d.rewards, d.advs, d.rets, d.values, rtab[0], a, b); };
                    std::vector<std::thread> ws;
                    const int64_t per = ((int64_t)R + workers - 1) / workers;
                    for (int w = 1; w < workers; ++w) {
                        const int64_t a = at0 + w * per, b = std::min<int64_t>(at0 + (int64_t)R, a + per);
                        if (a >= b) continue;
                        try { ws.emplace_back(span, a, b); } catch (...) { span(a, b); }
                    }
                    span(at0, std::min<int64_t>(at0 + (int64_t)R, at0 + per));
                    for (auto& t : ws) t.join();
                    if (t_exp) *t_exp = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count();
                };
                try { stages.emplace_back(stage); } catch (...) { deferred.push_back(stage); }
            }
            at += (int64_t)R;
            lo += B;
        }
        if (dst->ep_len)
            CU_TRY(cudaMemcpyAsync(dst->ep_len, e->ep_len_id, sizeof(int32_t) * (size_t)num_episodes, cudaMemcpyDeviceToHost, e->copy_stream));
        CU_TRY(cudaStreamSynchronize(e->copy_stream));
        return TWR_OK;
    };
    rc = body();
    const double t_copies = trace ? now_ms() : 0.0;
    for (auto& t : stages) t.join();                    // every exit path: workers done, engine flags restored
    for (auto& f : deferred) f();
    if (trace && !rc) {
        for (size_t k = 0; k < tr_done.size(); ++k) {
            float copy_ms = 0.f;
            if (k > 0) cudaEventElapsedTime(&copy_ms, e->ev_copied[k - 1], e->ev_copied[k]);
            fprintf(stderr, "[e2e] part %zu: %lld envs, %zu records | enqueued %.2f  rollout done %.2f  copy end-to-end gap %.2f  expanded %.2f\n",
                    k, (long long)parts[k], tr_R[k], tr_enq[k], tr_done[k], copy_ms, tr_exp[k]);
        }
        fprintf(stderr, "[e2e] copies done %.2f  all done %.2f ms (pack %d, %d workers)\n", t_copies, now_ms(), (int)pack, workers);
    }
    e->buf.obs_u8 = 0; e->buf.pack_misc = 0;
    e->timing = timing;
    if (rc) { cudaStreamSynchronize(e->stream); cudaStreamSynchronize(e->copy_stream); return rc; }
    twr_collected c{};
    c.n_records = at; c.num_episodes = num_episodes; c.n_cells = plan.env.N; c.num_actions = plan.dev.A;
    c.successes = successes; c.reward_sum = reward_sum;    // device pointers stay NULL: the data now lives in `dst`
    *out = c;
    return TWR_OK;
    });
}


// ------------------------------------------------ batched MCTS driver (K6; also used by solve/evaluate) ---
// node pool of B trees x P nodes (+ per-env scratch) from the engine's cache, grown when a call needs more
static int mcts_acquire(twr_engine* e, int64_t B, int P, MctsPool* pool, MctsArgs* a) {
    if (P >= (1 << 20)) return fail(TWR_ERR_INVALID, "MCTS tree too large (num_mcts_searches * max_expand_depth must stay below 2^18)");
    MctsCache& c = e->mcts;
    const size_t n = (size_t)B * (size_t)P;
    if (n > c.cap_nodes || B > c.cap_B) {
        CU_TRY(cudaStreamSynchronize(e->stream));
        const size_t nn = n > c.cap_nodes ? n : c.cap_nodes;
        const int64_t nb = B > c.cap_B ? B : c.cap_B;
        mcts_release(e);
        int rc;
        if ((rc = dev_alloc(&c.cells, nn)) || (rc = dev_alloc(&c.meta, nn)) || (rc = dev_alloc(&c.parent, nn)) || (rc = dev_alloc(&c.node, nn)) ||
            (rc = dev_alloc(&c.n_nodes, (size_t)nb)) || (rc = dev_alloc(&c.fwd_list, (size_t)nb)) || (rc = dev_alloc(&c.fwd_env, (size_t)nb)) ||
            (rc = dev_alloc(&c.fwd_count, 2)) || (rc = dev_alloc(&c.cur_node, (size_t)nb)) || (rc = dev_alloc(&c.cur_value, (size_t)nb)) ||
            (rc = dev_alloc(&c.active, (size_t)nb)) || (rc = dev_alloc(&c.path, (size_t)nb * TWR_MCTS_PATH)) ||
            (rc = dev_alloc(&c.path_len, (size_t)nb)) || (rc = dev_alloc(&c.leaf_pos, (size_t)nb))) { mcts_release(e); return rc; }
        c.cap_nodes = nn; c.cap_B = nb;
    }
    pool->B = B; pool->P = P; pool->cells = c.cells; pool->meta = c.meta; pool->parent = c.parent;
    pool->node = c.node; pool->n_nodes = c.n_nodes; pool->path = c.path; pool->path_len = c.path_len;
    a->fwd_list = c.fwd_list; a->fwd_env = c.fwd_env; a->fwd_count = c.fwd_count; a->cur_node = c.cur_node;
    a->cur_value = c.cur_value; a->active = c.active; a->leaf_pos = c.leaf_pos;
    return TWR_OK;
}

static int mcts_pool_nodes(int A, int n_sims, int med) { return 1 + A * (n_sims * (med > 1 ? med : 1) + 1); }

// Policy::full_predict evaluates every twist: for a twisted policy, a constant [n_perms][B] array whose row pi holds pi
// (the perm_idx of twist pi's forward) and a.n_perms / a.twist_stride for the averaging; nothing for an untwisted one.
// The caller sizes the forward outputs a.logits / a.values for n_perms slices of B.
static int stage_twists(twr_engine* e, const PolicyDev& dev, int64_t B, Staging<int32_t>* idx, MctsArgs* a) {
    a->n_perms = dev.n_perms; a->twist_stride = B;
    if (dev.n_perms == 0) return TWR_OK;
    int rc = idx->alloc((size_t)dev.n_perms * (size_t)B);
    if (rc) return rc;
    std::vector<int32_t> h((size_t)dev.n_perms * (size_t)B);
    for (int pi = 0; pi < dev.n_perms; ++pi) std::fill(h.begin() + (size_t)pi * B, h.begin() + (size_t)(pi + 1) * B, pi);
    CU_TRY(cudaMemcpyAsync(idx->d, h.data(), sizeof(int32_t) * h.size(), cudaMemcpyHostToDevice, e->stream));
    return TWR_OK;
}

// forward output slices of B rows in a search: one per twist of a twisted policy (Policy::full_predict), else one
static size_t forward_slices(const PolicyDev& dev) { return dev.n_perms > 0 ? (size_t)dev.n_perms : 1; }

struct MctsOpt { int n_sims; float C; int max_expand_depth; };

// A search of B trees: its pool size checked before anything is allocated, the node pool from the engine's cache, the
// twist rows of full_predict and the options.  mcts_target then sets what it runs on.
static int mcts_reserve(twr_engine* e, const PolicyDev& dev, int64_t B, const MctsOpt& mo, Staging<int32_t>* twist_idx, MctsArgs* a) {
    const int P = mcts_pool_nodes(dev.A, mo.n_sims, mo.max_expand_depth);
    if ((double)B * P >= 2147483647.0)
        return fail(TWR_ERR_INVALID, "MCTS node pool too large (num_episodes * (1 + A*(n_sims*depth+1)) must be < 2^31)");
    *a = MctsArgs{};
    a->pool.A = dev.A;
    a->n_sims = mo.n_sims; a->max_expand_depth = mo.max_expand_depth; a->C = mo.C;
    int rc;
    if ((rc = mcts_acquire(e, B, P, &a->pool, a)) || (rc = stage_twists(e, dev, B, twist_idx, a))) return rc;
    return TWR_OK;
}

// what a search runs on: its start envs, its Philox streams and its forward outputs (forward_slices slices of B rows)
static void mcts_target(const twr_engine* e, MctsArgs* a, const EnvParams& env, uint32_t cid, EnvIds ids, const uint4* cells,
                        const uint32_t* meta, const float4* logits, const float* values) {
    a->env = env; a->seed = e->seed; a->cid = cid; a->ids = ids;
    a->env_cells = cells; a->env_meta = meta; a->logits = logits; a->values = values;
}

// the forward of a leaf batch: one launch, or for a twisted policy one per twist, twist pi's outputs in slice pi
static void launch_forward_twists(twr_engine* e, const PolicyDev& dev, const ForwardArgs& fa, const int32_t* twist_idx, int64_t stride) {
    if (dev.n_perms == 0) { launch_forward(e, dev, fa); return; }
    for (int pi = 0; pi < dev.n_perms; ++pi) {
        ForwardArgs f = fa;
        f.perm_idx = twist_idx + (size_t)pi * stride;
        f.logits = fa.logits + (size_t)pi * stride; f.values = fa.values + (size_t)pi * stride;
        launch_forward(e, dev, f);
    }
}

// predict_probs_mcts (rl/search.rs:104-189) for every live env, in lockstep over the simulations.  twist_idx: the array
// of stage_twists (NULL for an untwisted policy)
static void enqueue_mcts(twr_engine* e, const PolicyDev& dev, MctsArgs& a, const int32_t* live, const int32_t* n_live, int64_t B,
                         const int32_t* twist_idx) {
    cudaStream_t st = e->stream;
    // small batches: one persistent launch runs every simulation of the search (twr_mcts.cu, k_mcts_persistent)
    if (!getenv("TWISTERL_B200_MCTS_LOCKSTEP") && launch_mcts_persistent(st, a, dev, live, n_live, B)) return;
    ForwardArgs fa = forward_args(e, a.env, a.cid, a.ids, a.pool.cells, B, const_cast<float4*>(a.logits), const_cast<float*>(a.values));
    fa.live = a.fwd_list;
    auto forward = [&]() { launch_forward_twists(e, dev, fa, twist_idx, a.twist_stride); };
    launch_mcts_begin(st, a, live, n_live, B);
    fa.n_live_ptr = a.fwd_count;
    forward();
    launch_mcts_expand(st, a, 0, 0, 0, 0, B);
    if (a.max_expand_depth == 1 && a.n_sims > 0) {
        // one expansion round per simulation: expand/backup of simulation s and the descent of s+1 share a launch
        int which = 1;
        launch_mcts_select(st, a, live, n_live, 0, which, B);
        for (int sim = 0; sim < a.n_sims; ++sim) {
            fa.n_live_ptr = a.fwd_count + which;
            forward();
            if (sim + 1 < a.n_sims) { launch_mcts_expand_select(st, a, live, n_live, sim, which, B); which ^= 1; }
            else launch_mcts_expand(st, a, 1, sim, 0, which, B);
        }
        return;
    }
    int round = 1;
    for (int sim = 0; sim < a.n_sims; ++sim) {
        int which = round & 1;
        launch_mcts_select(st, a, live, n_live, sim, which, B);
        ++round;
        for (int d = 0; d < a.max_expand_depth; ++d) {
            if (d > 0) { which = round & 1; launch_mcts_pre(st, a, live, n_live, which, B); ++round; }
            fa.n_live_ptr = a.fwd_count + which;
            forward();
            launch_mcts_expand(st, a, 1, sim, d, which, B);
        }
    }
}


int twr_policy_full_predict(twr_engine* e, const twr_policy* p, twr_envs* v, float* probs, float* values) {
    return twr_guard([&]() -> int {
    if (!e || !p || !v || !probs || !values) return fail(TWR_ERR_INVALID, "NULL argument");
    if (p->eng != e || v->eng != e) return fail(TWR_ERR_INVALID, "policy/envs belong to another engine");
    if (v->n == 0) return TWR_OK;
    PolicyDev dev;
    int rc = check_policy_env(p, v->p, &dev);
    if (rc) return rc;
    const int64_t n = v->n;
    HostForward f;
    ForwardArgs fa;
    MctsArgs a{};
    a.env = v->p; a.pool.A = dev.A;
    Staging<float> d_probs, d_out; Staging<int32_t> twist_idx;
    if ((rc = f.stage(e, dev, v->p, v->cells, n, forward_slices(dev), nullptr, &fa)) || (rc = d_probs.alloc((size_t)n * dev.A)) ||
        (rc = d_out.alloc((size_t)n)) || (rc = stage_twists(e, dev, n, &twist_idx, &a))) return rc;
    // the leaf evaluation of the lockstep search: its forward launches, then its averaging and predict epilogue
    launch_forward_twists(e, dev, fa, twist_idx.d, n);
    a.logits = fa.logits; a.values = fa.values;
    launch_full_predict(e->stream, a, v->cells, v->meta, n, d_probs.d, d_out.d);
    FWD_CHECK(e);
    CU_TRY(cudaMemcpyAsync(probs, d_probs.d, sizeof(float) * (size_t)n * dev.A, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaMemcpyAsync(values, d_out.d, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
    });
}

// every env of a batch of n live: the list 0..n-1 and its count n at n_live[0]
static int upload_all_live(twr_engine* e, int32_t* live, int32_t* n_live, int64_t n) {
    std::vector<int32_t> iota((size_t)n);
    for (int64_t i = 0; i < n; ++i) iota[(size_t)i] = (int32_t)i;
    const int32_t n32 = (int32_t)n;
    CU_TRY(cudaMemcpyAsync(live, iota.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    CU_TRY(cudaMemcpyAsync(n_live, &n32, sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
    return TWR_OK;
}

// MCTS steps are expensive: every few steps the searching loops synchronise to stop once no env is left live
static int rollouts_ended(twr_engine* e, const int32_t* n_live, bool* ended) {
    int32_t left = 0;
    CU_TRY(cudaMemcpyAsync(&left, n_live, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    *ended = left == 0;
    return TWR_OK;
}

// ------------------------------------------------------------ evaluate / solve (f1) ---
// The best of S searches by the tuple order (success, reward) of solve.rs:94, starting from best = ((0.0, -inf), [])
// (solve.rs:82): writes it to (*bs, *br) and returns its index, or -1 when no search beats the start.
static int best_of(const uint8_t* success, const float* total, int64_t S, float* bs, float* br) {
    int best = -1;
    *bs = 0.0f; *br = -INFINITY;
    for (int64_t i = 0; i < S; ++i) {
        const float s1 = success[i] ? 1.0f : 0.0f, r1 = total[i];
        if (s1 > *bs || (s1 == *bs && r1 > *br)) { *bs = s1; *br = r1; best = (int)i; }
    }
    return best;
}

// Shared driver: B envs already initialised in (cells, meta); runs single_solve (rl/solve.rs:17-71) for all of
// them in lockstep.  Fills total[B], success[B], n_steps[B] and (optionally) the per-step action record.
static int run_solve(twr_engine* e, const EnvParams& env, const PolicyDev& dev, int64_t B, int T, EnvIds ids, uint32_t cid,
                     int deterministic, MctsOpt mo, uint4* cells, uint32_t* meta, float* total, uint8_t* success, int32_t* n_steps,
                     uint8_t* act_rec) {
    Staging<int32_t> live_a, live_b, n_live;
    Staging<float4> logits; Staging<float> values;
    int rc;
    // num_mcts_searches > 0: every step's action distribution is predict_probs_mcts of the current state
    MctsArgs ma{};
    Staging<float> mcts_probs; Staging<int32_t> mcts_vis, twist_idx;
    const bool search = mo.n_sims > 0;
    if (search && ((rc = mcts_reserve(e, dev, B, mo, &twist_idx, &ma)) || (rc = mcts_probs.alloc((size_t)B * dev.A)) ||
                   (rc = mcts_vis.alloc((size_t)B * dev.A)))) return rc;
    const size_t slices = search ? forward_slices(dev) : 1;
    if ((rc = live_a.alloc((size_t)B)) || (rc = live_b.alloc((size_t)B)) || (rc = n_live.alloc((size_t)T + 2)) ||
        (rc = logits.alloc(slices * (size_t)B)) || (rc = values.alloc(slices * (size_t)B))) return rc;
    cudaStream_t st = e->stream;
    CU_TRY(cudaMemsetAsync(n_live.d, 0, sizeof(int32_t) * (size_t)(T + 2), st));
    if ((rc = upload_all_live(e, live_a.d, n_live.d, B))) return rc;
    CU_TRY(cudaMemsetAsync(total, 0, sizeof(float) * (size_t)B, st));
    CU_TRY(cudaMemsetAsync(success, 0, (size_t)B, st));
    CU_TRY(cudaMemsetAsync(n_steps, 0, sizeof(int32_t) * (size_t)B, st));
    ForwardArgs fa = forward_args(e, env, cid, ids, cells, B, logits.d, values.d);
    SolveArgs sa{};
    sa.env = env; sa.seed = e->seed; sa.cid = cid; sa.ids = ids; sa.A = dev.A; sa.deterministic = deterministic; sa.B = B;
    sa.cells = cells; sa.meta = meta; sa.logits = logits.d; sa.n_live = n_live.d; sa.total = total; sa.success = success;
    sa.act_rec = act_rec; sa.n_steps = n_steps;
    if (search) {
        mcts_target(e, &ma, env, cid, ids, cells, meta, logits.d, values.d);
        sa.mcts_probs = mcts_probs.d;
    }
    for (int t = 0; t <= T; ++t) {          // at most T steps, then the terminal visit
        int32_t* cur = (t & 1) ? live_b.d : live_a.d;
        int32_t* nxt = (t & 1) ? live_a.d : live_b.d;
        if (search) {
            ma.t = t;
            enqueue_mcts(e, dev, ma, cur, n_live.d + t, B, twist_idx.d);
            launch_mcts_read(st, ma, B, mcts_probs.d, mcts_vis.d);
        } else {
            fa.t = t; fa.live = cur; fa.n_live_ptr = n_live.d + t;
            launch_forward(e, dev, fa);
        }
        sa.t = t;
        launch_solve_step(st, sa, cur, nxt);
        bool ended = false;
        if (search && (t & 3) == 3 && (rc = rollouts_ended(e, n_live.d + t + 1, &ended))) return rc;
        if (ended) break;
    }
    FWD_CHECK(e);
    CU_TRY(cudaStreamSynchronize(st));       // staging buffers are freed on return
    return TWR_OK;
}

int twr_evaluate(twr_engine* e, const twr_env_spec* spec, const twr_policy* p, int64_t num_episodes, int32_t deterministic,
                 int32_t num_searches, int32_t num_mcts_searches, float C, int32_t max_expand_depth,
                 float* success_rate, float* mean_reward) {
    return twr_evaluate_episodes(e, spec, p, num_episodes, deterministic, num_searches, num_mcts_searches, C, max_expand_depth,
                                 success_rate, mean_reward, nullptr, nullptr);
}

int twr_evaluate_episodes(twr_engine* e, const twr_env_spec* spec, const twr_policy* p, int64_t num_episodes, int32_t deterministic,
                          int32_t num_searches, int32_t num_mcts_searches, float C, int32_t max_expand_depth,
                          float* success_rate, float* mean_reward, float* best_success, float* best_reward) {
    return twr_guard([&]() -> int {
    if (!success_rate || !mean_reward) return fail(TWR_ERR_INVALID, "NULL argument");
    if (num_mcts_searches < 0 || max_expand_depth < 0) return fail(TWR_ERR_INVALID, "negative argument");
    const MctsOpt mo{num_mcts_searches, C, max_expand_depth};
    CollectPlan plan;
    if (num_episodes <= 0) { *success_rate = NAN; *mean_reward = NAN; return TWR_OK; }   // 0/0 in rl/evaluate.rs:47
    int rc = plan_collect(e, spec, p, num_episodes, &plan);
    if (rc) return rc;
    if (num_searches < 0) return fail(TWR_ERR_INVALID, "num_searches must be >= 0");
    const int S = num_searches;
    if (S == 0) { *success_rate = 0.0f; *mean_reward = -INFINITY; return TWR_OK; }       // solve() returns its initial best
    const int64_t B = num_episodes * S;
    if (B >= (1ll << 31)) return fail(TWR_ERR_INVALID, "num_episodes * num_searches too large");
    CU_TRY(cudaSetDevice(e->device));
    Staging<uint4> cells; Staging<uint32_t> meta; Staging<float> total; Staging<uint8_t> success; Staging<int32_t> n_steps;
    if ((rc = cells.alloc((size_t)B)) || (rc = meta.alloc((size_t)B)) || (rc = total.alloc((size_t)B)) ||
        (rc = success.alloc((size_t)B)) || (rc = n_steps.alloc((size_t)B))) return rc;
    const uint32_t cid = e->collect_id++;
    const uint32_t base = (uint32_t)((int64_t)e->rank * num_episodes);
    // every search of an episode starts from the same reset state (evaluate.rs:29-31 resets once, solve clones)
    EnvIds reset_ids{base, 0u, 0u, (uint32_t)S};
    launch_envs_reset(e->stream, plan.env, cells.d, meta.d, B, e->seed, reset_ids, cid, nullptr, nullptr);
    EnvIds ids{(uint32_t)((int64_t)e->rank * B), 0u, 0u, 0u};
    if ((rc = run_solve(e, plan.env, plan.dev, B, plan.T, ids, cid, deterministic, mo, cells.d, meta.d, total.d, success.d,
                        n_steps.d, nullptr))) return rc;
    std::vector<float> h_total((size_t)B); std::vector<uint8_t> h_succ((size_t)B);
    CU_TRY(cudaMemcpy(h_total.data(), total.d, sizeof(float) * (size_t)B, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(h_succ.data(), success.d, (size_t)B, cudaMemcpyDeviceToHost));
    float succ = 0.0f, rew = 0.0f;
    for (int64_t ep = 0; ep < num_episodes; ++ep) {
        float bs, br;
        best_of(h_succ.data() + ep * S, h_total.data() + ep * S, S, &bs, &br);
        succ += bs; rew += br;
        if (best_success) best_success[ep] = bs;
        if (best_reward) best_reward[ep] = br;
    }
    *success_rate = succ / (float)num_episodes;
    *mean_reward = rew / (float)num_episodes;
    return TWR_OK;
    });
}

int twr_solve(twr_engine* e, twr_envs* start, const twr_policy* p, int32_t deterministic, int32_t num_searches,
              int32_t num_mcts_searches, float C, int32_t max_expand_depth,
              float* success, float* reward, int32_t* actions, int32_t max_actions, int32_t* n_actions) {
    return twr_guard([&]() -> int {
    if (!e || !start || !p || !success || !reward || !n_actions) return fail(TWR_ERR_INVALID, "NULL argument");
    if (num_mcts_searches < 0 || max_expand_depth < 0) return fail(TWR_ERR_INVALID, "negative argument");
    const MctsOpt mo{num_mcts_searches, C, max_expand_depth};
    if (start->eng != e || p->eng != e) return fail(TWR_ERR_INVALID, "envs/policy belong to another engine");
    if (start->n != 1) return fail(TWR_ERR_INVALID, "twr_solve needs a batch of exactly one env holding the start state");
    *success = 0.0f; *reward = -INFINITY; *n_actions = 0;
    if (num_searches <= 0) return TWR_OK;
    PolicyDev dev;
    int rc = check_policy_env(p, start->p, &dev);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(e->device));
    int32_t depth = 0;
    if ((rc = twr_envs_depth(start, &depth))) return rc;
    const int T = depth;                                       // every step burns one unit of budget
    const int64_t B = num_searches;
    Staging<uint4> cells; Staging<uint32_t> meta; Staging<float> total; Staging<uint8_t> succ, act; Staging<int32_t> n_steps;
    if ((rc = cells.alloc((size_t)B)) || (rc = meta.alloc((size_t)B)) || (rc = total.alloc((size_t)B)) ||
        (rc = succ.alloc((size_t)B)) || (rc = n_steps.alloc((size_t)B)) || (rc = act.alloc((size_t)B * (size_t)(T + 1)))) return rc;
    launch_envs_broadcast(e->stream, start->cells, start->meta, cells.d, meta.d, B);
    const uint32_t cid = e->collect_id++;
    EnvIds ids{0x50000000u, 0u, 0u, 0u};
    if ((rc = run_solve(e, start->p, dev, B, T, ids, cid, deterministic, mo, cells.d, meta.d, total.d, succ.d, n_steps.d, act.d))) return rc;
    std::vector<float> h_total((size_t)B); std::vector<uint8_t> h_succ((size_t)B); std::vector<int32_t> h_n((size_t)B);
    CU_TRY(cudaMemcpy(h_total.data(), total.d, sizeof(float) * (size_t)B, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(h_succ.data(), succ.d, (size_t)B, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(h_n.data(), n_steps.d, sizeof(int32_t) * (size_t)B, cudaMemcpyDeviceToHost));
    const int best = best_of(h_succ.data(), h_total.data(), B, success, reward);
    if (best >= 0) {
        const int n = h_n[(size_t)best];
        *n_actions = n;
        if (actions) {
            if (n > max_actions) return fail(TWR_ERR_INVALID, "actions buffer too small");
            std::vector<uint8_t> col((size_t)(T + 1) * (size_t)B);
            CU_TRY(cudaMemcpy(col.data(), act.d, col.size(), cudaMemcpyDeviceToHost));
            for (int t = 0; t < n; ++t) actions[t] = col[(size_t)t * (size_t)B + (size_t)best];
        }
    }
    return TWR_OK;
    });
}


// ------------------------------------------------------------- AlphaZero (K6) ---
static int mcts_probs_impl(twr_engine* e, const twr_policy* p, twr_envs* v, int32_t n_sims, float C, int32_t max_expand_depth,
                           uint32_t env_id_base, uint32_t collect_id, int32_t t, float* probs, int32_t* visits, int32_t* trace);

int twr_mcts_probs(twr_engine* e, const twr_policy* p, twr_envs* v, int32_t n_sims, float C, int32_t max_expand_depth,
                   uint32_t env_id_base, uint32_t collect_id, int32_t t, float* probs, int32_t* visits) {
    return mcts_probs_impl(e, p, v, n_sims, C, max_expand_depth, env_id_base, collect_id, t, probs, visits, nullptr);
}

int twr_debug_mcts_trace(twr_engine* e, const twr_policy* p, twr_envs* v, int32_t n_sims, float C, int32_t max_expand_depth,
                         uint32_t env_id_base, uint32_t collect_id, int32_t t, float* probs, int32_t* visits, int32_t* trace) {
    if (!trace) return fail(TWR_ERR_INVALID, "NULL argument");
    return mcts_probs_impl(e, p, v, n_sims, C, max_expand_depth, env_id_base, collect_id, t, probs, visits, trace);
}

static int mcts_probs_impl(twr_engine* e, const twr_policy* p, twr_envs* v, int32_t n_sims, float C, int32_t max_expand_depth,
                           uint32_t env_id_base, uint32_t collect_id, int32_t t, float* probs, int32_t* visits, int32_t* trace) {
    if (!e || !p || !v || !probs || !visits) return fail(TWR_ERR_INVALID, "NULL argument");
    if (p->eng != e || v->eng != e) return fail(TWR_ERR_INVALID, "policy/envs belong to another engine");
    if (n_sims < 0 || max_expand_depth < 0 || t < 0) return fail(TWR_ERR_INVALID, "negative argument");
    if (v->n == 0) return TWR_OK;
    PolicyDev dev;
    int rc = check_policy_env(p, v->p, &dev);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(e->device));
    const int64_t B = v->n;
    MctsArgs a;
    Staging<float4> logits; Staging<float> values, d_probs; Staging<int32_t> live, n_live, d_vis, twist_idx;
    const size_t slices = forward_slices(dev);
    if ((rc = mcts_reserve(e, dev, B, MctsOpt{n_sims, C, max_expand_depth}, &twist_idx, &a)) ||
        (rc = logits.alloc(slices * (size_t)B)) || (rc = values.alloc(slices * (size_t)B)) || (rc = live.alloc((size_t)B)) ||
        (rc = n_live.alloc(1)) || (rc = d_probs.alloc((size_t)B * dev.A)) || (rc = d_vis.alloc((size_t)B * dev.A))) return rc;
    if ((rc = upload_all_live(e, live.d, n_live.d, B))) return rc;
    mcts_target(e, &a, v->p, collect_id, EnvIds{env_id_base, 0u, 0u, 0u}, v->cells, v->meta, logits.d, values.d);
    a.t = t;
    Staging<int32_t> d_trace;
    const size_t n_trace = (size_t)(n_sims > 0 ? n_sims : 1) * (size_t)B * 2;
    if (trace) {
        if ((rc = d_trace.alloc(n_trace))) return rc;
        CU_TRY(cudaMemsetAsync(d_trace.d, 0xFF, sizeof(int32_t) * n_trace, e->stream));
        a.trace = d_trace.d;
    }
    enqueue_mcts(e, dev, a, live.d, n_live.d, B, twist_idx.d);
    launch_mcts_read(e->stream, a, B, d_probs.d, d_vis.d);
    FWD_CHECK(e);
    if (trace) CU_TRY(cudaMemcpyAsync(trace, d_trace.d, sizeof(int32_t) * (size_t)n_sims * (size_t)B * 2, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaMemcpyAsync(probs, d_probs.d, sizeof(float) * (size_t)B * dev.A, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaMemcpyAsync(visits, d_vis.d, sizeof(int32_t) * (size_t)B * dev.A, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    return TWR_OK;
}

int twr_az_collect(twr_engine* e, const twr_env_spec* spec, const twr_policy* p, int64_t num_episodes, int32_t num_mcts_searches,
                   float C, int32_t max_expand_depth, twr_collected* out) {
    return twr_guard([&]() -> int {
    if (!out) return fail(TWR_ERR_INVALID, "NULL argument");
    CollectPlan plan;
    int rc = plan_collect(e, spec, p, num_episodes, &plan);
    if (rc) return rc;
    if (num_mcts_searches < 0 || max_expand_depth < 0) return fail(TWR_ERR_INVALID, "negative argument");
    if (plan.dev.n_perms > 0) return fail(TWR_ERR_UNSUPPORTED, "MCTS with twists (full_predict over all perms) is not implemented; the AZ trainer clears them (rl/az.py:24-26)");
    CU_TRY(cudaSetDevice(e->device));
    const int64_t B = num_episodes;
    const int T = plan.T;
    MctsArgs a;
    Staging<int32_t> no_twists;                 // stays empty: twists are refused above
    if ((rc = mcts_reserve(e, plan.dev, B, MctsOpt{num_mcts_searches, C, max_expand_depth}, &no_twists, &a)) ||
        (rc = ensure_collect_buffers(e, B, T, plan.env.N, B))) return rc;
    CollectBuffers& b = e->buf;
    cudaStream_t st = e->stream;
    e->has_last = false;
    b.obs_u8 = 0;
    const uint32_t cid = e->collect_id++;
    const EnvIds ids{(uint32_t)((int64_t)e->rank * B), (uint32_t)(B - 1), (uint32_t)B, 0u};
    if ((rc = begin_collect(e, plan.env, B, ids, cid, 0))) return rc;
    mcts_target(e, &a, plan.env, cid, ids, b.cells, b.meta, b.logits, b.values);
    for (int t = 0; t < T; ++t) {
        int32_t* cur = (t & 1) ? b.live_b : b.live_a;
        int32_t* nxt = (t & 1) ? b.live_a : b.live_b;
        a.t = t;
        enqueue_mcts(e, plan.dev, a, cur, b.n_live + t, B, nullptr);
        launch_az_finish(st, a, b, cur, nxt);
        bool ended = false;
        if ((t & 7) == 7 && (rc = rollouts_ended(e, b.n_live + t + 1, &ended))) return rc;
        if (ended) break;
    }
    launch_az_remaining(st, b);
    launch_episode_offsets(st, b, ids);
    launch_compact(st, plan.env, b, plan.dev.A);
    FWD_CHECK(e);
    return finish_collect(e, plan, num_episodes, twr_engine::LAST_AZ, spec, cid, out);
    });
}

int twr_host_alloc(void** ptr, int64_t bytes) {
    if (!ptr || bytes < 0) return fail(TWR_ERR_INVALID, "bad argument");
    CU_TRY(cudaHostAlloc(ptr, (size_t)(bytes ? bytes : 1), cudaHostAllocDefault));
    return TWR_OK;
}
void twr_host_free(void* ptr) { if (ptr) cudaFreeHost(ptr); }

}  // extern "C"
