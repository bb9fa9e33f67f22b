// twisterl_b200.hpp -- C++17 host side above the C ABI (twisterl_b200.h), header only.
//
// The reference's collection path is compiled Rust; its toolchain is absent from this image, so this header is the
// compiled-language mirror of the reference's own types for that path, name for name:
//
//   twisterl::Linear / EmbeddingBag / Sequential / Policy   rust/src/nn/layers.rs:10-49, nn/modules.rs:16-34, nn/policy.rs:20-32
//   twisterl::CollectedData (+ merge)                        rust/src/collector/collector.rs:22-88
//   twisterl::Collector { collect(env, policy) }             rust/src/collector/collector.rs:90-92 (trait Collector)
//   twisterl::PPOCollector / AZCollector                     rust/src/collector/ppo.rs:40-126, collector/az.rs:49-130
//   twisterl::evaluate / solve                               rust/src/rl/evaluate.rs:22-89, rl/solve.rs:73-101
//
// An env is named by its constructor arguments (twr_env_spec, the device stand-in for Box<dyn Env>): Puzzle(...) and
// GridWorld(...) below build it.  Every failure of the library is thrown as twisterl::Error carrying twr_last_error()
// -- the anyhow::Error -> PyRuntimeError of the reference (python_interface/error_mapping.rs:29-33).  There is no CPU
// fallback: without a Blackwell device Engine's constructor throws.
#pragma once

#include "twisterl_b200.h"

#include <cstdint>
#include <map>
#include <array>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

namespace twisterl {

struct Error : std::runtime_error {
    int status;
    Error(int st, const std::string& what) : std::runtime_error(what), status(st) {}
};
inline void check(int rc) {
    if (rc != TWR_OK) throw Error(rc, twr_last_error());
}

// ---------------------------------------------------------------------------------------------- envs ---
inline twr_env_spec Puzzle(int width, int height, int difficulty, int depth_slope, int max_depth) {   // envs/puzzle.rs:34-42
    return twr_env_spec{TWR_ENV_PUZZLE, width, height, difficulty, depth_slope, max_depth};
}
inline twr_env_spec GridWorld(int width, int height, int max_steps, int difficulty) {                  // grid_world/src/lib.rs:23-41
    return twr_env_spec{TWR_ENV_GRIDWORLD, width, height, difficulty, 0, max_steps};
}

// -------------------------------------------------------------------------------------------- engine ---
class Engine {
public:
    explicit Engine(int device = 0, twr_precision precision = TWR_PREC_F16X2, uint64_t seed = 0x5EED5EEDull, int rank = 0,
                    int world = 1, void* stream = nullptr) : rank_(rank) {
        twr_engine_cfg cfg{device, (int32_t)precision, seed, rank, world, stream};
        check(twr_engine_create(&cfg, &h_));
    }
    ~Engine() { if (h_) twr_engine_destroy(h_); }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    twr_engine* handle() const { return h_; }
    int rank() const { return rank_; }
    void synchronize() { check(twr_engine_synchronize(h_)); }
    void set_collect_id(uint32_t id) { check(twr_engine_set_collect_id(h_, id)); }   // pins the Philox streams of the next collect
    int64_t launch_count() const { return twr_engine_launch_count(h_); }

    // ---- multi-GPU plumbing (one Engine per GPU, rank / world from the constructor): NCCL through the C ABI
    static std::array<uint8_t, TWR_COMM_ID_BYTES> comm_unique_id() {      // rank 0 creates it; the host ships the bytes to every rank
        std::array<uint8_t, TWR_COMM_ID_BYTES> id{};
        check(twr_comm_unique_id(id.data()));
        return id;
    }
    void comm_init(const std::array<uint8_t, TWR_COMM_ID_BYTES>& id) { check(twr_comm_init(h_, id.data())); }   // collective
    // in-place sum / max over the ranks of a few host doubles (episodes, successes, reward sum, records, ...)
    void allreduce_stats(std::vector<double>& stats, twr_reduce_op op = TWR_REDUCE_SUM) {
        check(twr_allreduce_stats(h_, stats.data(), (int32_t)stats.size(), (int32_t)op));
    }

private:
    twr_engine* h_ = nullptr;
    int rank_ = 0;
};

// ------------------------------------------------------------------------------------------------ nn ---
struct Linear {                      // nn.Linear(weights_vector, bias_vector, apply_relu): weights = W.T.flatten()
    std::vector<float> weights, bias;
    bool apply_relu = false;
    int out() const { return (int)bias.size(); }
    int in() const { return bias.empty() ? 0 : (int)(weights.size() / bias.size()); }
};
using Sequential = std::vector<Linear>;
struct EmbeddingBag {                // nn.EmbeddingBag(vec_vectors, bias_vector, apply_relu, obs_shape, conv_dim)
    std::vector<std::vector<float>> vectors;
    std::vector<float> bias;
    bool apply_relu = true;
    std::vector<int> obs_shape;      // one entry: BasicPolicy; two: Conv1dPolicy (nn/layers.rs:63-77)
    int conv_dim = 0;
};
struct PolicyWeights {               // nn.Policy(embeddings, common, action_net, value_net, obs_perms, act_perms)
    EmbeddingBag embeddings;
    Sequential common, action_net, value_net;
    std::vector<std::vector<int32_t>> obs_perms, act_perms;
};

class Policy {
public:
    Policy(Engine& eng, const PolicyWeights& w) : eng_(&eng) { with_desc(w, [&](const twr_policy_desc& d) { check(twr_policy_create(eng.handle(), &d, &h_)); }); }
    // straight from a safetensors checkpoint of the reference's BasicPolicy / Conv1dPolicy state dict (native reader)
    static std::unique_ptr<Policy> from_safetensors(Engine& eng, const std::string& path, const std::vector<int32_t>& obs_shape = {},
                                                    int conv_dim = 0, const std::vector<std::vector<int32_t>>& obs_perms = {},
                                                    const std::vector<std::vector<int32_t>>& act_perms = {}) {
        std::vector<int32_t> op, ap;
        for (const auto& p : obs_perms) op.insert(op.end(), p.begin(), p.end());
        for (const auto& p : act_perms) ap.insert(ap.end(), p.begin(), p.end());
        std::unique_ptr<Policy> pol(new Policy(eng));
        check(twr_policy_create_from_safetensors(eng.handle(), path.c_str(), obs_shape.empty() ? nullptr : obs_shape.data(),
                                                 (int32_t)obs_shape.size(), conv_dim, op.empty() ? nullptr : op.data(),
                                                 ap.empty() ? nullptr : ap.data(), (int32_t)obs_perms.size(), &pol->h_));
        return pol;
    }
    ~Policy() { if (h_) twr_policy_destroy(h_); }
    Policy(const Policy&) = delete;
    Policy& operator=(const Policy&) = delete;
    // in-place weight refresh (what sync_rs_policy rebuilds from scratch in the reference, rl/algorithm.py:91-93)
    void update(const PolicyWeights& w) { with_desc(w, [&](const twr_policy_desc& d) { check(twr_policy_update(h_, &d)); }); }
    // rank `root`'s parameters into this policy on every rank (ncclBroadcast on the engine stream) + operand refresh
    void broadcast_from(int root = 0) { check(twr_broadcast_weights(eng_->handle(), h_, root)); }
    twr_policy* handle() const { return h_; }
    Engine& engine() const { return *eng_; }

private:
    explicit Policy(Engine& eng) : eng_(&eng) {}
    template <class F>
    static void with_desc(const PolicyWeights& w, F&& f) {
        const EmbeddingBag& e = w.embeddings;
        std::vector<float> flat;
        const size_t v = e.vectors.empty() ? 0 : e.vectors[0].size();
        flat.reserve(e.vectors.size() * v);
        for (const auto& row : e.vectors) {
            if (row.size() != v) throw Error(TWR_ERR_INVALID, "EmbeddingBag vectors must have equal lengths");
            flat.insert(flat.end(), row.begin(), row.end());
        }
        auto lin = [](const Sequential& s) {
            std::vector<twr_linear_desc> d;
            for (const Linear& l : s) d.push_back(twr_linear_desc{l.weights.data(), l.bias.data(), l.in(), l.out(), l.apply_relu ? 1 : 0});
            return d;
        };
        const std::vector<twr_linear_desc> c = lin(w.common), a = lin(w.action_net), vn = lin(w.value_net);
        std::vector<int32_t> op, ap;
        for (const auto& p : w.obs_perms) op.insert(op.end(), p.begin(), p.end());
        for (const auto& p : w.act_perms) ap.insert(ap.end(), p.begin(), p.end());
        twr_policy_desc d{};
        d.emb_vectors = flat.data(); d.emb_bias = e.bias.data();
        d.obs_size = (int32_t)e.vectors.size(); d.emb_size = (int32_t)e.bias.size(); d.emb_apply_relu = e.apply_relu ? 1 : 0;
        d.obs_shape_len = (int32_t)e.obs_shape.size();
        for (size_t i = 0; i < e.obs_shape.size() && i < 2; ++i) d.obs_shape[i] = e.obs_shape[i];
        d.conv_dim = e.conv_dim;
        d.common = c.data(); d.n_common = (int32_t)c.size();
        d.action_net = a.data(); d.n_action = (int32_t)a.size();
        d.value_net = vn.data(); d.n_value = (int32_t)vn.size();
        d.n_perms = (int32_t)w.obs_perms.size();
        d.obs_perms = op.empty() ? nullptr : op.data(); d.act_perms = ap.empty() ? nullptr : ap.data();
        f(d);
    }
    Engine* eng_;
    twr_policy* h_ = nullptr;
};

// ----------------------------------------------------------------------------------------- collector ---
struct CollectedData {                                                    // collector/collector.rs:22-30
    std::vector<std::vector<size_t>> obs;
    std::vector<std::vector<float>> logits;
    std::vector<float> values, rewards;
    std::vector<size_t> actions;
    std::vector<std::optional<size_t>> perms;
    std::map<std::string, std::vector<float>> additional_data;
    // extras of the device path (not part of the reference struct)
    std::vector<int32_t> ep_len;
    int64_t successes = 0;
    double reward_sum = 0.0;

    void merge(const CollectedData& o) {                                  // collector/collector.rs:48-88
        obs.insert(obs.end(), o.obs.begin(), o.obs.end());
        logits.insert(logits.end(), o.logits.begin(), o.logits.end());
        values.insert(values.end(), o.values.begin(), o.values.end());
        rewards.insert(rewards.end(), o.rewards.begin(), o.rewards.end());
        actions.insert(actions.end(), o.actions.begin(), o.actions.end());
        perms.insert(perms.end(), o.perms.begin(), o.perms.end());
        for (const auto& kv : o.additional_data) {
            auto& dst = additional_data[kv.first];
            dst.insert(dst.end(), kv.second.begin(), kv.second.end());
        }
    }
};

struct Collector {                                                        // trait Collector, collector/collector.rs:90-92
    virtual ~Collector() = default;
    virtual CollectedData collect(const twr_env_spec& env, Policy& policy) = 0;
};

namespace detail {
template <class T>
struct Pinned {                      // page-locked destination so the D2H copies overlap the next sub-batch's rollout
    T* p = nullptr;
    explicit Pinned(size_t n) { void* q = nullptr; check(twr_host_alloc(&q, (int64_t)(n * sizeof(T)))); p = static_cast<T*>(q); }
    ~Pinned() { twr_host_free(p); }
    Pinned(const Pinned&) = delete;
    Pinned& operator=(const Pinned&) = delete;
};
}  // namespace detail

class PPOCollector : public Collector {                                   // collector/ppo.rs:40-126
public:
    PPOCollector(size_t num_episodes, float gamma, float lambda, size_t num_cores = 1)
        : num_episodes(num_episodes), gamma(gamma), lambda(lambda), num_cores(num_cores) {}
    size_t num_episodes;
    float gamma, lambda;
    size_t num_cores;                // accepted for compatibility: episodes spread over the SMs, not over a rayon pool

    CollectedData collect(const twr_env_spec& env, Policy& policy) override {
        const int64_t cap = twr_max_records(&env, (int64_t)num_episodes);
        if (cap < 0) throw Error(TWR_ERR_INVALID, twr_last_error());
        const size_t n = (size_t)env.width * env.height, C = (size_t)cap;
        const bool u8 = n * n <= 256;                                     // one-byte observation indices when they fit
        detail::Pinned<uint8_t> obs8(u8 ? C * n : 1), actions(C);
        detail::Pinned<uint16_t> obs16(u8 ? 1 : C * n);
        detail::Pinned<float> logits(C * 4), values(C), rewards(C), advs(C), rets(C);
        detail::Pinned<int8_t> perms(C);
        detail::Pinned<int32_t> ep_len(num_episodes ? num_episodes : 1);
        twr_host_buffers dst{cap, u8 ? nullptr : obs16.p, logits.p, values.p, rewards.p, advs.p, rets.p, actions.p, perms.p, ep_len.p,
                             u8 ? obs8.p : nullptr};
        twr_collected c{};
        check(twr_ppo_collect_host(policy.engine().handle(), &env, policy.handle(), nullptr, (int64_t)num_episodes, gamma, lambda, &dst, &c));
        const size_t R = (size_t)c.n_records, A = (size_t)c.num_actions;
        CollectedData d;
        d.obs.resize(R); d.logits.resize(R);
        for (size_t r = 0; r < R; ++r) {
            d.obs[r].resize(n);
            for (size_t i = 0; i < n; ++i) d.obs[r][i] = u8 ? (size_t)obs8.p[r * n + i] : (size_t)obs16.p[r * n + i];
            d.logits[r].assign(logits.p + r * A, logits.p + (r + 1) * A);
        }
        d.values.assign(values.p, values.p + R);
        d.rewards.assign(rewards.p, rewards.p + R);
        d.actions.assign(actions.p, actions.p + R);
        d.perms.resize(R);
        for (size_t r = 0; r < R; ++r) d.perms[r] = perms.p[r] < 0 ? std::nullopt : std::optional<size_t>((size_t)perms.p[r]);
        d.additional_data["advs"].assign(advs.p, advs.p + R);             // ppo.rs:94-96
        d.additional_data["rets"].assign(rets.p, rets.p + R);
        d.ep_len.assign(ep_len.p, ep_len.p + num_episodes);
        d.successes = c.successes; d.reward_sum = c.reward_sum;
        return d;                                                         // already in merge order [last, 0, 1, .., n-2]
    }
};

class AZCollector : public Collector {                                    // collector/az.rs:49-130
public:
    AZCollector(size_t num_episodes, size_t num_mcts_searches, float C, size_t max_expand_depth, size_t num_cores = 1)
        : num_episodes(num_episodes), num_mcts_searches(num_mcts_searches), C(C), max_expand_depth(max_expand_depth), num_cores(num_cores) {}
    size_t num_episodes, num_mcts_searches;
    float C;
    size_t max_expand_depth, num_cores;

    CollectedData collect(const twr_env_spec& env, Policy& policy) override {
        twr_collected c{};
        check(twr_az_collect(policy.engine().handle(), &env, policy.handle(), (int64_t)num_episodes, (int32_t)num_mcts_searches, C,
                             (int32_t)max_expand_depth, &c));
        const size_t R = (size_t)c.n_records, n = (size_t)c.n_cells, A = (size_t)c.num_actions;
        std::vector<uint16_t> obs(R * n + 1);
        std::vector<float> probs(R * A + 1), rets(R + 1);
        std::vector<int32_t> ep_len(num_episodes ? num_episodes : 1);
        twr_host_buffers dst{(int64_t)R, obs.data(), probs.data(), nullptr, nullptr, nullptr, rets.data(), nullptr, nullptr, ep_len.data(), nullptr};
        check(twr_collected_to_host(policy.engine().handle(), &dst));
        CollectedData d;                                                  // az.rs:97-104: obs, probs in .logits, perms None, the rest empty
        d.obs.resize(R); d.logits.resize(R); d.perms.assign(R, std::nullopt);
        for (size_t r = 0; r < R; ++r) {
            d.obs[r].assign(obs.begin() + r * n, obs.begin() + (r + 1) * n);
            d.logits[r].assign(probs.begin() + r * A, probs.begin() + (r + 1) * A);
        }
        d.additional_data["remaining_values"].assign(rets.begin(), rets.begin() + R);
        d.ep_len.assign(ep_len.begin(), ep_len.begin() + num_episodes);
        d.successes = c.successes; d.reward_sum = c.reward_sum;
        return d;
    }
};

// Collective over the ranks, each of which has just run a device-resident collect (twr_ppo_collect / twr_az_collect) of
// the same shape: rank `root` receives every rank's episodes, merged in the order ONE collect of all of them lays out
// (twr_gather_collected), as CollectedData shaped like PPOCollector::collect's, or with `az` like AZCollector::collect's
// (MCTS distributions in `logits`, additional_data["remaining_values"], perms None, no values / rewards / actions).
// The other ranks get an empty CollectedData.
inline CollectedData gather_collected(Engine& eng, int root = 0, bool az = false) {
    twr_collected c{};
    check(twr_gather_collected(eng.handle(), root, &c));
    CollectedData d;
    if (eng.rank() != root) return d;
    const size_t R = (size_t)c.n_records, n = (size_t)c.n_cells, A = (size_t)c.num_actions, E = (size_t)c.num_episodes;
    std::vector<uint16_t> obs(R * n + 1);
    std::vector<float> logits(R * A + 1), values(R + 1), rewards(R + 1), advs(R + 1), rets(R + 1);
    std::vector<uint8_t> actions(R + 1);
    std::vector<int8_t> perms(R + 1);
    d.ep_len.resize(E);
    twr_host_buffers dst{(int64_t)R, obs.data(), logits.data(), values.data(), rewards.data(), advs.data(), rets.data(),
                         actions.data(), perms.data(), d.ep_len.data(), nullptr};
    check(twr_collected_to_host(eng.handle(), &dst));
    d.obs.resize(R); d.logits.resize(R); d.perms.resize(R);
    for (size_t r = 0; r < R; ++r) {
        d.obs[r].assign(obs.begin() + r * n, obs.begin() + (r + 1) * n);
        d.logits[r].assign(logits.begin() + r * A, logits.begin() + (r + 1) * A);
        d.perms[r] = az || perms[r] < 0 ? std::nullopt : std::optional<size_t>((size_t)perms[r]);
    }
    d.successes = c.successes; d.reward_sum = c.reward_sum;
    if (az) {                                                             // az.rs:97-104, as AZCollector::collect
        d.additional_data["remaining_values"].assign(rets.begin(), rets.begin() + R);
        return d;
    }
    d.values.assign(values.begin(), values.begin() + R);
    d.rewards.assign(rewards.begin(), rewards.begin() + R);
    d.actions.assign(actions.begin(), actions.begin() + R);
    d.additional_data["advs"].assign(advs.begin(), advs.begin() + R);
    d.additional_data["rets"].assign(rets.begin(), rets.begin() + R);
    return d;
}

// A batch of envs of one spec on the device (the parity API of the C header): reset / set_state / step / queries
class Envs {
public:
    Envs(Engine& eng, const twr_env_spec& spec, int64_t n) : n_(n), cells_(spec.width * spec.height) { check(twr_envs_create(eng.handle(), &spec, n, &h_)); }
    ~Envs() { if (h_) twr_envs_destroy(h_); }
    Envs(const Envs&) = delete;
    Envs& operator=(const Envs&) = delete;
    twr_envs* handle() const { return h_; }
    void set_state(const std::vector<int64_t>& states) { check(twr_envs_set_state(h_, states.data())); }        // [n][cells]
    void reset(uint32_t env_id_base = 0, uint32_t collect_id = 0) { check(twr_envs_reset(h_, env_id_base, collect_id)); }
    void step(const std::vector<int32_t>& actions) { check(twr_envs_step(h_, actions.data())); }
    std::vector<int64_t> get_state() { std::vector<int64_t> s((size_t)(n_ * cells_)); check(twr_envs_get_state(h_, s.data())); return s; }
    std::vector<int32_t> observe() { std::vector<int32_t> o((size_t)(n_ * cells_)); check(twr_envs_observe(h_, o.data())); return o; }
    std::vector<float> reward() { std::vector<float> r((size_t)n_); check(twr_envs_reward(h_, r.data())); return r; }
    std::vector<uint8_t> is_final() { std::vector<uint8_t> f((size_t)n_); check(twr_envs_is_final(h_, f.data())); return f; }

private:
    twr_envs* h_ = nullptr;
    int64_t n_;
    int cells_;
};

// rl/solve.rs:73-101: best of num_searches rollouts from the state held by the one-env batch `start`
// -> ((success, reward), actions)
inline std::pair<std::pair<float, float>, std::vector<size_t>> solve(Envs& start, Policy& policy, bool deterministic, size_t num_searches,
                                                                     size_t num_mcts_searches = 0, float C = 1.41f,
                                                                     size_t max_expand_depth = 1, size_t max_actions = 4096) {
    float s = 0.f, r = 0.f;
    int32_t n = 0;
    std::vector<int32_t> acts(max_actions);
    check(twr_solve(policy.engine().handle(), start.handle(), policy.handle(), deterministic ? 1 : 0, (int32_t)num_searches,
                    (int32_t)num_mcts_searches, C, (int32_t)max_expand_depth, &s, &r, acts.data(), (int32_t)max_actions, &n));
    return {{s, r}, std::vector<size_t>(acts.begin(), acts.begin() + n)};
}

// rl/evaluate.rs:22-89 -> (success rate, mean reward); `seed` and `num_cores` of the reference signature have no effect here
inline std::pair<float, float> evaluate(const twr_env_spec& env, Policy& policy, size_t num_episodes, bool deterministic,
                                        size_t num_searches, size_t num_mcts_searches = 0, float C = 1.41f, size_t max_expand_depth = 1) {
    float s = 0.f, r = 0.f;
    check(twr_evaluate(policy.engine().handle(), &env, policy.handle(), (int64_t)num_episodes, deterministic ? 1 : 0, (int32_t)num_searches,
                       (int32_t)num_mcts_searches, C, (int32_t)max_expand_depth, &s, &r));
    return {s, r};
}

}  // namespace twisterl
