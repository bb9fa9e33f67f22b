// twr_private.cuh -- the opaque handles of include/twisterl_b200.h, shared by the translation units that implement the ABI
// (twr_engine.cu: engine / policy / env / collect; twr_comm.cu: NCCL plumbing).
#pragma once
#include "../../include/twisterl_b200.h"
#include "twr_kernels.cuh"

#include <map>
#include <vector>

// MCTS working set of an engine (node pool + per-env scratch), kept between calls: AZ collects / MCTS-guided evaluation
// re-allocating ~1 GB per call cost more in cudaMalloc / cudaFree (and their implicit synchronisation) than the searches
struct MctsCache {
    uint4* cells = nullptr; uint4* node = nullptr; uint32_t* meta = nullptr;
    int32_t *parent = nullptr, *n_nodes = nullptr, *fwd_list = nullptr, *fwd_env = nullptr, *fwd_count = nullptr, *cur_node = nullptr,
            *path = nullptr, *path_len = nullptr, *leaf_pos = nullptr;
    uint8_t* active = nullptr; float* cur_value = nullptr;
    size_t cap_nodes = 0; int64_t cap_B = 0;
};

struct twr_engine {
    int device = 0, precision = 0, rank = 0, world = 1;
    int tc_terms = 0;            // ForwardArgs::tc_terms of every tensor-core forward of this engine (0 = all split terms)
    int tc_flags = 0;            // TWISTERL_B200_TC_FLAGS: experiment switches of the pair kernel OR-ed into ForwardArgs::dbg_flags
    bool launch_error = false;   // a forward launch could not be made since the last check (see FWD_CHECK)
    uint64_t seed = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    uint32_t collect_id = 0;
    long long launches0 = 0;
    // collect buffers: working set + two compacted-output sets (double buffered for the pipelined host collect)
    CollectBuffers buf{};
    struct OutSet { uint16_t* obs = nullptr; float* logits = nullptr; float* values = nullptr; float* rewards = nullptr;
                    float* advs = nullptr; float* rets = nullptr; uint8_t* actions = nullptr; int8_t* perms = nullptr; };
    OutSet outs[2];
    int32_t* ep_len_id = nullptr; int64_t cap_E = 0;
    int64_t cap_B = 0; int cap_T = 0; int64_t cap_R = 0; int cap_cells = 0;
    cudaStream_t copy_stream = nullptr;
    std::map<uint64_t, float> survive_half;   // (env, batch) shape -> fraction of envs alive past half the horizon, last collect
    uint64_t hint_key = 0; int64_t hint_B = 0;
    void note_survival() {                    // call after h_stats of an enqueue_collect has landed
        if (hint_B > 0) survive_half[hint_key] = (float)((double)(h_stats[3] & 0xFFFFFFFFull) / (double)hint_B);
    }
    int32_t* bal_flags = nullptr;   // hand-off counters of the balanced pair-kernel schedule (one per CTA pair)
    int bal_delta = 3;
#define TWR_MAX_SUBBATCH 64
    cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_copied[TWR_MAX_SUBBATCH] = {}, ev_small[TWR_MAX_SUBBATCH] = {};
    unsigned long long* h_stats = nullptr;   // pinned, mapped
    unsigned long long* d_hstats = nullptr;  // its device address
    bool has_last = false;
    twr_collected last{};
    // what `last` holds, and the spec and collect id it was collected with (twr_gather_collected checks that every rank
    // ran the same collect)
    enum LastKind { LAST_NONE = 0, LAST_PPO = 1, LAST_AZ = 2, LAST_MERGED = 3 };
    int last_kind = LAST_NONE;
    twr_env_spec last_spec{};
    uint32_t last_cid = 0;
    // the gathered result on the root rank: engine-owned and grow-only, separate from outs[], which the pipelined host
    // collect double-buffers
    OutSet merged;
    int32_t* merged_ep_len = nullptr;
    int64_t cap_mR = 0, cap_mE = 0; int cap_mcells = 0;
    // timing
    bool timing = false;
    std::vector<cudaEvent_t> ev;
    float last_fwd_ms = 0.f, last_total_ms = 0.f; int64_t last_fwd_launches = 0;
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    // NCCL plumbing (twr_comm.cu): communicator over the `world` engines of a job, device scratch for the stats reduction
    void* comm = nullptr;
    double* d_stats = nullptr;
    int64_t* d_gather = nullptr;      // twr_gather_collected: every rank's header (world x TWR_GATHER_HDR words) + root's verdict
    MctsCache mcts;
    long long* trace_buf = nullptr;   // device counters of a traced forward launch (TWISTERL_B200_TRACE)
};

// root's merged output buffers for R records of n_cells cells over E episodes (twr_engine.cu; grow-only)
extern "C" int twr_ensure_merged_buffers(twr_engine* e, int64_t R, int64_t E, int n_cells);

struct twr_policy {
    twr_engine* eng = nullptr;
    PolicyDev dev{};
    float* d_blob = nullptr;
    int64_t blob_floats = 0;
    int32_t* d_obs_perms = nullptr;
    int32_t* d_act_perms = nullptr;
    void* tc_pack = nullptr;
    int64_t off_emb_b = 0;
    std::vector<int64_t> off_w, off_b;   // blob offsets of every Linear (common..., action_net..., value_net...)
};

struct twr_envs {
    twr_engine* eng = nullptr;
    EnvParams p{};
    int64_t n = 0;
    uint4* cells = nullptr;
    uint32_t* meta = nullptr;
};

