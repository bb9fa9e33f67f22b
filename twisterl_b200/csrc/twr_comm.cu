// twr_comm.cu -- multi-GPU plumbing of the C ABI (SURVEY.md 8e): one engine per GPU, envs sharded with no data-path
// collective during the rollout; NCCL over NVLink carries the per-iteration weight broadcast, the statistics reduction
// and, for a trainer on one rank, the gather of every rank's collected records into that rank's memory.
//
// NCCL is bound at RUN time (dlopen of libnccl.so.2, or the path in TWISTERL_B200_NCCL_LIB): a host process that already
// loaded NCCL (PyTorch ships one) shares that copy, and a single-GPU host needs no NCCL at all.  Only the prototypes of
// <nccl.h> are used at compile time.
#include "twr_private.cuh"

#include <dlfcn.h>
#include <nccl.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

extern "C" int twr_set_error(int code, const char* msg);

namespace {

struct Nccl {
    void* handle = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclBroadcast) Broadcast = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclGetVersion) GetVersion = nullptr;
    // optional: only twr_gather_collected uses them, and a libnccl without them leaves every other entry point working
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclSend) Send = nullptr;
    decltype(&ncclRecv) Recv = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    std::string why;
};
Nccl g_nccl;
std::once_flag g_nccl_once;

const Nccl& nccl() {
    std::call_once(g_nccl_once, [] {
        const char* names[] = {getenv("TWISTERL_B200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (!n || !*n) continue;
            g_nccl.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (g_nccl.handle) break;
            g_nccl.why = dlerror();
        }
        if (!g_nccl.handle) return;
        auto sym = [&](const char* s) { void* p = dlsym(g_nccl.handle, s); if (!p) g_nccl.why = std::string("missing symbol ") + s; return p; };
        g_nccl.GetUniqueId = reinterpret_cast<decltype(&ncclGetUniqueId)>(sym("ncclGetUniqueId"));
        g_nccl.CommInitRank = reinterpret_cast<decltype(&ncclCommInitRank)>(sym("ncclCommInitRank"));
        g_nccl.CommDestroy = reinterpret_cast<decltype(&ncclCommDestroy)>(sym("ncclCommDestroy"));
        g_nccl.Broadcast = reinterpret_cast<decltype(&ncclBroadcast)>(sym("ncclBroadcast"));
        g_nccl.AllReduce = reinterpret_cast<decltype(&ncclAllReduce)>(sym("ncclAllReduce"));
        g_nccl.GetErrorString = reinterpret_cast<decltype(&ncclGetErrorString)>(sym("ncclGetErrorString"));
        g_nccl.GetVersion = reinterpret_cast<decltype(&ncclGetVersion)>(sym("ncclGetVersion"));
        if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.Broadcast || !g_nccl.AllReduce ||
            !g_nccl.GetErrorString) {
            dlclose(g_nccl.handle);
            g_nccl.handle = nullptr;
            return;
        }
        g_nccl.AllGather = reinterpret_cast<decltype(&ncclAllGather)>(dlsym(g_nccl.handle, "ncclAllGather"));
        g_nccl.Send = reinterpret_cast<decltype(&ncclSend)>(dlsym(g_nccl.handle, "ncclSend"));
        g_nccl.Recv = reinterpret_cast<decltype(&ncclRecv)>(dlsym(g_nccl.handle, "ncclRecv"));
        g_nccl.GroupStart = reinterpret_cast<decltype(&ncclGroupStart)>(dlsym(g_nccl.handle, "ncclGroupStart"));
        g_nccl.GroupEnd = reinterpret_cast<decltype(&ncclGroupEnd)>(dlsym(g_nccl.handle, "ncclGroupEnd"));
    });
    return g_nccl;
}

int no_nccl() { return twr_set_error(TWR_ERR_UNSUPPORTED, ("NCCL is not available: " + nccl().why).c_str()); }
int nccl_fail(const char* what, ncclResult_t r) {
    return twr_set_error(TWR_ERR_CUDA, (std::string(what) + ": " + nccl().GetErrorString(r)).c_str());
}
#define CU_TRY(expr)                                                                                        \
    do {                                                                                                    \
        cudaError_t _e = (expr);                                                                            \
        if (_e != cudaSuccess) return twr_set_error(TWR_ERR_CUDA, (std::string(#expr) + ": " + cudaGetErrorString(_e)).c_str()); \
    } while (0)

static_assert(sizeof(ncclUniqueId) == TWR_COMM_ID_BYTES, "TWR_COMM_ID_BYTES must be sizeof(ncclUniqueId)");

// One rank's header of twr_gather_collected, int64 words.  Every rank all-gathers it before any record moves and reaches
// the same verdict from the same bytes.  Words H_KIND .. H_EPISODES and H_SEED .. H_ROOT must agree across ranks.
enum : int {
    H_HAS = 0,        // 1: `last` is this rank's own device-resident collect
    H_KIND,           // twr_engine::LastKind
    H_SPEC,           // 6 words: the twr_env_spec the collect ran on
    H_CELLS = H_SPEC + 6, H_ACTIONS, H_EPISODES,
    H_RECORDS, H_HEAD,  // records, and of them the first episode's (the rank's last episode id, see twr_gather_collected)
    H_SUCCESSES, H_REWARD_SUM /* double bits */,
    H_SEED, H_PRECISION, H_CID, H_ROOT,
    H_FAIL,           // non-zero: this rank's own preparation failed (a twr_status); every rank returns it, none moves data
    TWR_GATHER_HDR
};

}  // namespace

extern "C" {

int twr_comm_version(void) {
    int v = 0;
    if (!nccl().handle || !nccl().GetVersion || nccl().GetVersion(&v) != ncclSuccess) return 0;
    return v;
}

int twr_comm_unique_id(uint8_t* id) {
    if (!id) return twr_set_error(TWR_ERR_INVALID, "id is NULL");
    if (!nccl().handle) return no_nccl();
    ncclUniqueId u;
    const ncclResult_t r = nccl().GetUniqueId(&u);
    if (r != ncclSuccess) return nccl_fail("ncclGetUniqueId", r);
    memcpy(id, &u, sizeof(u));
    return TWR_OK;
}

int twr_comm_init(twr_engine* e, const uint8_t* id) {
    if (!e || !id) return twr_set_error(TWR_ERR_INVALID, "NULL argument");
    if (e->comm) return twr_set_error(TWR_ERR_STATE, "twr_comm_init: this engine already has a communicator");
    if (!nccl().handle) return no_nccl();
    CU_TRY(cudaSetDevice(e->device));
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    ncclComm_t c = nullptr;
    const ncclResult_t r = nccl().CommInitRank(&c, e->world, u, e->rank);
    if (r != ncclSuccess) return nccl_fail("ncclCommInitRank", r);
    e->comm = c;
    if (!e->d_stats) CU_TRY(cudaMalloc(reinterpret_cast<void**>(&e->d_stats), TWR_COMM_MAX_STATS * sizeof(double)));
    if (!e->d_gather) CU_TRY(cudaMalloc(reinterpret_cast<void**>(&e->d_gather), ((size_t)e->world * TWR_GATHER_HDR + 1) * sizeof(int64_t)));
    return TWR_OK;
}

void twr_comm_destroy(twr_engine* e) {
    if (!e) return;
    if (e->comm && nccl().handle) {
        cudaSetDevice(e->device);
        cudaStreamSynchronize(e->stream);
        nccl().CommDestroy(static_cast<ncclComm_t>(e->comm));
    }
    e->comm = nullptr;
    if (e->d_stats) { cudaFree(e->d_stats); e->d_stats = nullptr; }
    if (e->d_gather) { cudaFree(e->d_gather); e->d_gather = nullptr; }
}

int twr_broadcast_weights(twr_engine* e, twr_policy* p, int32_t root) {
    if (!e || !p) return twr_set_error(TWR_ERR_INVALID, "NULL argument");
    if (p->eng != e) return twr_set_error(TWR_ERR_INVALID, "policy belongs to another engine");
    if (root < 0 || root >= e->world) return twr_set_error(TWR_ERR_INVALID, "root out of range");
    CU_TRY(cudaSetDevice(e->device));
    if (e->world > 1) {
        if (!e->comm) return twr_set_error(TWR_ERR_STATE, "twr_broadcast_weights: call twr_comm_init first");
        const ncclResult_t r = nccl().Broadcast(p->d_blob, p->d_blob, (size_t)p->blob_floats, ncclFloat32, root,
                                                static_cast<ncclComm_t>(e->comm), e->stream);
        if (r != ncclSuccess) return nccl_fail("ncclBroadcast", r);
    }
    // every rank (the root included) rebuilds the kernels' operand layouts from the blob it now holds
    return twr_policy_update_from_device(p, p->d_blob);
}

int twr_allreduce_stats(twr_engine* e, double* stats, int32_t n, int32_t op) {
    if (!e || !stats) return twr_set_error(TWR_ERR_INVALID, "NULL argument");
    if (n < 1 || n > TWR_COMM_MAX_STATS) return twr_set_error(TWR_ERR_INVALID, "n must be in 1..TWR_COMM_MAX_STATS");
    if (op != TWR_REDUCE_SUM && op != TWR_REDUCE_MAX) return twr_set_error(TWR_ERR_INVALID, "op must be TWR_REDUCE_SUM or TWR_REDUCE_MAX");
    if (e->world == 1) return TWR_OK;
    if (!e->comm) return twr_set_error(TWR_ERR_STATE, "twr_allreduce_stats: call twr_comm_init first");
    CU_TRY(cudaSetDevice(e->device));
    CU_TRY(cudaMemcpyAsync(e->d_stats, stats, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    const ncclResult_t r = nccl().AllReduce(e->d_stats, e->d_stats, (size_t)n, ncclFloat64, op == TWR_REDUCE_MAX ? ncclMax : ncclSum,
                                            static_cast<ncclComm_t>(e->comm), e->stream);
    if (r != ncclSuccess) return nccl_fail("ncclAllReduce", r);
    CU_TRY(cudaMemcpyAsync(stats, e->d_stats, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));       // the reduced numbers are read by the host (what a trainer logs); this
                                                    // also keeps a rank from queueing the next step behind a slower peer
    return TWR_OK;
}

// Rank r's local result is [episode (r+1)E-1][episodes rE .. (r+1)E-2] (EnvIds{rank*E, E-1, E} of the collects): a head of
// one episode, then a tail.  ONE collect of W*E episodes lays out [WE-1][0 .. WE-2], i.e.
// head_{W-1}, tail_0, head_0, tail_1, head_1, ..., tail_{W-1}: each rank's two pieces go straight to their merged offsets.
int twr_gather_collected(twr_engine* e, int32_t root, twr_collected* out) {
    if (!e || !out) return twr_set_error(TWR_ERR_INVALID, "NULL argument");
    if (root < 0 || root >= e->world) return twr_set_error(TWR_ERR_INVALID, "root out of range");
    const bool local = e->has_last && (e->last_kind == twr_engine::LAST_PPO || e->last_kind == twr_engine::LAST_AZ);
    static const char* no_result = "twr_gather_collected: rank %d holds no device-resident collect result (no twr_ppo_collect / "
                                   "twr_az_collect has succeeded since its last collect call, or it already holds a gathered result)";
    char msg[256];
    if (e->world == 1) {
        if (!local) { snprintf(msg, sizeof msg, no_result, e->rank); return twr_set_error(TWR_ERR_STATE, msg); }
        *out = e->last;
        return TWR_OK;
    }
    if (!e->comm) return twr_set_error(TWR_ERR_STATE, "twr_gather_collected: call twr_comm_init first");
    const Nccl& n = nccl();
    if (!n.AllGather || !n.Send || !n.Recv || !n.GroupStart || !n.GroupEnd)
        return twr_set_error(TWR_ERR_UNSUPPORTED, "twr_gather_collected: this libnccl lacks ncclAllGather / ncclSend / ncclRecv / ncclGroupStart / ncclGroupEnd");
    CU_TRY(cudaSetDevice(e->device));
    cudaStream_t st = e->stream;
    ncclComm_t comm = static_cast<ncclComm_t>(e->comm);
    const int W = e->world;
    const twr_collected& c = e->last;

    // 1. agreement: every rank's header to every rank
    int64_t h[TWR_GATHER_HDR] = {};
    h[H_ROOT] = root;
    std::string own_failure;       // a local failure travels in the header instead of leaving the peers in the all-gather
    if (local) {
        int32_t head = 0;
        cudaError_t ce = cudaMemcpyAsync(&head, c.ep_len + (c.num_episodes - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) {
            h[H_FAIL] = TWR_ERR_CUDA;
            own_failure = std::string("twr_gather_collected: reading the first episode's length: ") + cudaGetErrorString(ce);
        }
        const twr_env_spec& s = e->last_spec;
        const int64_t spec[6] = {s.kind, s.width, s.height, s.difficulty, s.depth_slope, s.max_depth};
        h[H_HAS] = 1; h[H_KIND] = e->last_kind;
        for (int k = 0; k < 6; ++k) h[H_SPEC + k] = spec[k];
        h[H_CELLS] = c.n_cells; h[H_ACTIONS] = c.num_actions; h[H_EPISODES] = c.num_episodes;
        h[H_RECORDS] = c.n_records; h[H_HEAD] = head; h[H_SUCCESSES] = c.successes;
        memcpy(&h[H_REWARD_SUM], &c.reward_sum, sizeof(double));
        h[H_SEED] = (int64_t)e->seed; h[H_PRECISION] = e->precision; h[H_CID] = e->last_cid;
    }
    std::vector<int64_t> all((size_t)W * TWR_GATHER_HDR);
    int64_t* d_mine = e->d_gather + (size_t)e->rank * TWR_GATHER_HDR;
    CU_TRY(cudaMemcpyAsync(d_mine, h, sizeof(h), cudaMemcpyHostToDevice, st));
    ncclResult_t r = n.AllGather(d_mine, e->d_gather, TWR_GATHER_HDR, ncclInt64, comm, st);
    if (r != ncclSuccess) return nccl_fail("ncclAllGather", r);
    CU_TRY(cudaMemcpyAsync(all.data(), e->d_gather, sizeof(int64_t) * all.size(), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    auto hdr = [&](int rk, int word) { return all[(size_t)rk * TWR_GATHER_HDR + word]; };
    for (int rk = 0; rk < W; ++rk)
        if (hdr(rk, H_FAIL)) {
            if (rk == e->rank) return twr_set_error((int)hdr(rk, H_FAIL), own_failure.c_str());
            snprintf(msg, sizeof msg, "twr_gather_collected: rank %d failed before the exchange", rk);
            return twr_set_error((int)hdr(rk, H_FAIL), msg);
        }
    for (int rk = 0; rk < W; ++rk)
        if (!hdr(rk, H_HAS)) { snprintf(msg, sizeof msg, no_result, rk); return twr_set_error(TWR_ERR_STATE, msg); }
    static const struct { int lo, hi; const char* what; } agree[] = {
        {H_KIND, H_KIND + 1, "collect kind (PPO / AZ)"}, {H_SPEC, H_SPEC + 6, "env spec"}, {H_CELLS, H_ACTIONS + 1, "shape"},
        {H_EPISODES, H_EPISODES + 1, "num_episodes"}, {H_SEED, H_SEED + 1, "seed"}, {H_PRECISION, H_PRECISION + 1, "precision"},
        {H_CID, H_CID + 1, "collect id"}, {H_ROOT, H_ROOT + 1, "root"}};
    for (int rk = 1; rk < W; ++rk)
        for (const auto& a : agree)
            for (int k = a.lo; k < a.hi; ++k)
                if (hdr(rk, k) != hdr(0, k)) {
                    snprintf(msg, sizeof msg, "twr_gather_collected: the ranks ran different collects (%s of rank %d differs from rank 0's)", a.what, rk);
                    return twr_set_error(TWR_ERR_INVALID, msg);
                }

    // 2. root sizes its merged buffers; every rank learns whether that worked before anything is sent
    const int64_t E = hdr(0, H_EPISODES);
    const int cells = (int)hdr(0, H_CELLS), A = (int)hdr(0, H_ACTIONS);
    int64_t R_total = 0, successes = 0;
    double reward_sum = 0.0;
    for (int rk = 0; rk < W; ++rk) {
        double rs;
        memcpy(&rs, &all[(size_t)rk * TWR_GATHER_HDR + H_REWARD_SUM], sizeof(double));
        R_total += hdr(rk, H_RECORDS); successes += hdr(rk, H_SUCCESSES); reward_sum += rs;
    }
    const bool is_root = e->rank == root;
    int64_t verdict = is_root ? twr_ensure_merged_buffers(e, R_total, (int64_t)W * E, cells) : 0;
    int64_t* d_verdict = e->d_gather + (size_t)W * TWR_GATHER_HDR;
    CU_TRY(cudaMemcpyAsync(d_verdict, &verdict, sizeof(int64_t), cudaMemcpyHostToDevice, st));
    r = n.Broadcast(d_verdict, d_verdict, 1, ncclInt64, root, comm, st);
    if (r != ncclSuccess) return nccl_fail("ncclBroadcast", r);
    CU_TRY(cudaMemcpyAsync(&verdict, d_verdict, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if (verdict != TWR_OK)
        return is_root ? (int)verdict : twr_set_error((int)verdict, "twr_gather_collected: the root rank could not allocate the merged result");

    // 3. the records: two pieces per field per rank, each received at its merged offset
    std::vector<int64_t> head_at(W), tail_at(W);
    int64_t pos = hdr(W - 1, H_HEAD);
    head_at[W - 1] = 0;
    for (int rk = 0; rk < W; ++rk) {
        tail_at[rk] = pos; pos += hdr(rk, H_RECORDS) - hdr(rk, H_HEAD);
        if (rk < W - 1) { head_at[rk] = pos; pos += hdr(rk, H_HEAD); }
    }
    const twr_engine::OutSet& m = e->merged;
    const struct { const void* src; void* dst; size_t rec_bytes; } fields[] = {
        {c.obs, m.obs, sizeof(uint16_t) * cells}, {c.logits, m.logits, sizeof(float) * A}, {c.values, m.values, sizeof(float)},
        {c.rewards, m.rewards, sizeof(float)}, {c.advs, m.advs, sizeof(float)}, {c.rets, m.rets, sizeof(float)},
        {c.actions, m.actions, 1}, {c.perms, m.perms, 1}};
    // every piece of rank rk, in one order on both ends of each send / receive pair: fn(rk, src byte offset, dst, bytes)
    auto for_each_piece = [&](auto&& fn) -> int {
        for (int rk = 0; rk < W; ++rk) {
            const int64_t hd = hdr(rk, H_HEAD), tl = hdr(rk, H_RECORDS) - hd;
            for (const auto& f : fields) {
                char* dst = static_cast<char*>(f.dst);
                int rc;
                if ((rc = fn(rk, f.src, 0, dst + head_at[rk] * f.rec_bytes, hd * f.rec_bytes)) ||
                    (rc = fn(rk, f.src, hd * f.rec_bytes, dst + tail_at[rk] * f.rec_bytes, tl * f.rec_bytes))) return rc;
            }
            const int rc = fn(rk, c.ep_len, 0, e->merged_ep_len + rk * E, (size_t)E * sizeof(int32_t));   // by episode id
            if (rc) return rc;
        }
        return TWR_OK;
    };
    r = n.GroupStart();
    if (r != ncclSuccess) return nccl_fail("ncclGroupStart", r);
    int rc = for_each_piece([&](int rk, const void* src, size_t off, void* dst, size_t bytes) -> int {
        if (rk == root || bytes == 0) return TWR_OK;
        ncclResult_t q = ncclSuccess;
        if (is_root) q = n.Recv(dst, bytes, ncclUint8, rk, comm, st);
        else if (rk == e->rank) q = n.Send(static_cast<const char*>(src) + off, bytes, ncclUint8, root, comm, st);
        return q == ncclSuccess ? TWR_OK : nccl_fail(is_root ? "ncclRecv" : "ncclSend", q);
    });
    r = n.GroupEnd();                              // closes the group on an error too
    if (rc) return rc;
    if (r != ncclSuccess) return nccl_fail("ncclGroupEnd", r);
    if (is_root)              // root's own shard, after its receives are posted: a failure here leaves no peer waiting
        rc = for_each_piece([&](int rk, const void* src, size_t off, void* dst, size_t bytes) -> int {
            if (rk != root || bytes == 0) return TWR_OK;
            CU_TRY(cudaMemcpyAsync(dst, static_cast<const char*>(src) + off, bytes, cudaMemcpyDeviceToDevice, st));
            return TWR_OK;
        });
    if (rc) { cudaStreamSynchronize(st); return rc; }
    CU_TRY(cudaStreamSynchronize(st));

    if (is_root) {
        twr_collected mc{};
        mc.n_records = R_total; mc.num_episodes = (int64_t)W * E; mc.n_cells = cells; mc.num_actions = A;
        mc.successes = successes; mc.reward_sum = reward_sum;
        mc.obs = m.obs; mc.logits = m.logits; mc.values = m.values; mc.rewards = m.rewards; mc.advs = m.advs;
        mc.rets = m.rets; mc.actions = m.actions; mc.perms = m.perms; mc.ep_len = e->merged_ep_len;
        e->last = mc;
        e->last_kind = twr_engine::LAST_MERGED;
    }
    *out = e->last;
    return TWR_OK;
}

}  // extern "C"
