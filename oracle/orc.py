"""ctypes binding of the CPU oracle (oracle/twr_oracle.c).

TEST INFRASTRUCTURE ONLY.  Importers allowed: tests/, __graft_entry__.smoke(), and
bench.py's cpu_baseline / --impl reference legs.  Nothing under twisterl_b200/ imports this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SO = _HERE / "_build" / "libtwr_oracle.so"

ENV_PUZZLE, ENV_GRIDWORLD = 0, 1
RNG_RESET, RNG_PERM, RNG_SAMPLE, RNG_SOLVE = 0, 1, 2, 3
NET_COMMON, NET_ACTION, NET_VALUE = 0, 1, 2
MAX_CELLS = 64


def build(force: bool = False) -> Path:
    srcs = [_HERE / "twr_oracle.c", _HERE / "twr_oracle.h", _HERE / "Makefile"]
    stale = (not _SO.exists()) or any(s.stat().st_mtime > _SO.stat().st_mtime for s in srcs)
    if force or stale:
        subprocess.run(["make", "-C", str(_HERE), "-B"], check=True, capture_output=True)
    return _SO


class EnvSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
                ("difficulty", C.c_int32), ("depth_slope", C.c_int32), ("max_depth", C.c_int32)]


class _Env(C.Structure):
    _fields_ = [("spec", EnvSpec), ("cells", C.c_int64 * MAX_CELLS), ("zx", C.c_int32), ("zy", C.c_int32),
                ("depth", C.c_int64), ("ax", C.c_int32), ("ay", C.c_int32), ("gx", C.c_int32),
                ("gy", C.c_int32), ("tx", C.c_int32), ("ty", C.c_int32), ("steps_left", C.c_int64)]


class _Collected(C.Structure):
    _fields_ = [("n_records", C.c_int64), ("num_episodes", C.c_int32), ("n_cells", C.c_int32),
                ("num_actions", C.c_int32), ("ep_len", C.POINTER(C.c_int32)), ("obs", C.POINTER(C.c_int32)),
                ("logits", C.POINTER(C.c_float)), ("values", C.POINTER(C.c_float)),
                ("rewards", C.POINTER(C.c_float)), ("advs", C.POINTER(C.c_float)),
                ("rets", C.POINTER(C.c_float)), ("actions", C.POINTER(C.c_int32)),
                ("perms", C.POINTER(C.c_int32))]


_lib = None


def lib():
    global _lib
    if _lib is None:
        try:
            build()
            _lib = C.CDLL(str(_SO))
        except OSError:
            build(force=True)
            _lib = C.CDLL(str(_SO))
        L = _lib
        L.orc_u32_to_unit_f32.restype = C.c_float
        L.orc_u32_to_unit_f32.argtypes = [C.c_uint32]
        L.orc_env_reward.restype = C.c_float
        L.orc_policy_new.restype = C.c_void_p
        L.orc_policy_free.argtypes = [C.c_void_p]
        L.orc_env_reset.argtypes = [C.POINTER(_Env), C.c_uint64, C.c_uint32, C.c_uint32]
        L.orc_gae.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
        L.orc_solve.argtypes = [C.POINTER(_Env), C.c_void_p, C.c_int32, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32,
                                C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p, C.POINTER(C.c_int32)]
        L.orc_evaluate.argtypes = [C.POINTER(EnvSpec), C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_uint32,
                                   C.c_uint32, C.c_uint32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p, C.c_void_p]
        L.orc_solve_mcts.argtypes = [C.POINTER(_Env), C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_int32,
                                     C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                     C.c_void_p, C.POINTER(C.c_int32)]
        L.orc_evaluate_mcts.argtypes = [C.POINTER(EnvSpec), C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                        C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_float),
                                        C.POINTER(C.c_float), C.c_void_p, C.c_void_p]
        L.orc_ppo_collect.argtypes = [C.POINTER(EnvSpec), C.c_void_p, C.c_int32, C.c_float, C.c_float,
                                      C.c_uint64, C.c_uint32, C.c_uint32, C.c_int32, C.POINTER(_Collected)]
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def philox(ctr, key) -> np.ndarray:
    c = (C.c_uint32 * 4)(*[int(x) & 0xFFFFFFFF for x in ctr])
    k = (C.c_uint32 * 2)(*[int(x) & 0xFFFFFFFF for x in key])
    o = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(c, k, o)
    return np.array(list(o), dtype=np.uint32)


def u32_to_unit_f32(w: int) -> float:
    return float(lib().orc_u32_to_unit_f32(int(w) & 0xFFFFFFFF))


def puzzle_spec(width, height, difficulty, depth_slope, max_depth) -> EnvSpec:
    return EnvSpec(ENV_PUZZLE, width, height, difficulty, depth_slope, max_depth)


def gridworld_spec(width, height, max_steps, difficulty) -> EnvSpec:
    return EnvSpec(ENV_GRIDWORLD, width, height, difficulty, 0, max_steps)


class Env:
    """One scalar env, driven exactly like the reference's `Box<dyn Env>`."""

    def __init__(self, spec: EnvSpec):
        self._e = _Env()
        lib().orc_env_init(C.byref(self._e), C.byref(spec))

    @property
    def spec(self) -> EnvSpec:
        return self._e.spec

    def num_actions(self): return int(lib().orc_env_num_actions(C.byref(self._e)))
    def num_cells(self): return int(lib().orc_env_num_cells(C.byref(self._e)))
    def obs_shape(self): n = self.num_cells(); return [n, n]

    @property
    def difficulty(self): return int(lib().orc_env_get_difficulty(C.byref(self._e)))

    @difficulty.setter
    def difficulty(self, d): lib().orc_env_set_difficulty(C.byref(self._e), int(d))

    def set_state(self, state):
        a = np.ascontiguousarray(state, dtype=np.int64)
        lib().orc_env_set_state(C.byref(self._e), _p(a, C.c_int64), len(a))

    def reset(self, seed=0, env_id=0, collect_id=0):
        lib().orc_env_reset(C.byref(self._e), int(seed), int(env_id), int(collect_id))

    def step(self, action): lib().orc_env_step(C.byref(self._e), int(action))

    def masks(self):
        m = np.zeros(self.num_actions(), dtype=np.uint8)
        lib().orc_env_masks(C.byref(self._e), _p(m, C.c_uint8))
        return [bool(x) for x in m]

    def is_final(self): return bool(lib().orc_env_is_final(C.byref(self._e)))
    def success(self): return bool(lib().orc_env_success(C.byref(self._e)))
    def reward(self): return float(lib().orc_env_reward(C.byref(self._e)))

    def observe(self):
        o = np.zeros(self.num_cells(), dtype=np.int32)
        lib().orc_env_observe(C.byref(self._e), _p(o, C.c_int32))
        return o.tolist()

    def get_state(self):
        b = np.zeros(self.num_cells(), dtype=np.int64)
        lib().orc_env_get_state(C.byref(self._e), _p(b, C.c_int64))
        return b.tolist()

    @property
    def depth(self):
        return int(self._e.depth if self._e.spec.kind == ENV_PUZZLE else self._e.steps_left)

    @property
    def zero_location(self):
        return (int(self._e.zx), int(self._e.zy))


class Policy:
    """Restated `twisterl.nn.Policy`; weights in the exact layouts `to_rust()` hands over."""

    def __init__(self):
        self._h = C.c_void_p(lib().orc_policy_new())
        self.num_actions = None

    def __del__(self):
        if getattr(self, "_h", None):
            try:
                lib().orc_policy_free(self._h)
            except Exception:                      # interpreter shutdown: module globals are already gone
                pass
            self._h = None

    def set_embedding(self, vectors, bias, apply_relu=True, obs_shape=None, conv_dim=0):
        v = np.ascontiguousarray(vectors, dtype=np.float32)
        b = np.ascontiguousarray(bias, dtype=np.float32)
        shape = np.ascontiguousarray(obs_shape if obs_shape is not None else [v.shape[0]], dtype=np.int32)
        rc = lib().orc_policy_set_embedding(self._h, _p(v, C.c_float), v.shape[0], v.shape[1], _p(b, C.c_float),
                                            len(b), int(apply_relu), _p(shape, C.c_int32), len(shape), int(conv_dim))
        assert rc == 0

    def add_linear(self, which, weights_vector, bias, apply_relu):
        w = np.ascontiguousarray(weights_vector, dtype=np.float32).ravel()
        b = np.ascontiguousarray(bias, dtype=np.float32)
        rc = lib().orc_policy_add_linear(self._h, which, _p(w, C.c_float), len(w), _p(b, C.c_float), len(b),
                                         int(apply_relu))
        assert rc == 0
        if which == NET_ACTION:
            self.num_actions = len(b)

    def set_perms(self, obs_perms, act_perms):
        op = np.ascontiguousarray(obs_perms, dtype=np.int32)
        ap = np.ascontiguousarray(act_perms, dtype=np.int32)
        n = op.shape[0] if op.size else 0
        lib().orc_policy_set_perms(self._h, _p(op, C.c_int32), _p(ap, C.c_int32), n,
                                   op.shape[1] if n else 0, ap.shape[1] if n else 0)

    @classmethod
    def from_torch_state_dict(cls, sd, obs_perms=(), act_perms=()):
        """BasicPolicy state_dict -> oracle policy, mirroring nn/utils.py:17-59 (to_rust export)."""
        g = lambda k: np.asarray(sd[k], dtype=np.float32)
        p = cls()
        p.set_embedding(g("embeddings.weight").T, g("embeddings.bias"), True)
        for net, which in (("common", NET_COMMON), ("action", NET_ACTION), ("value", NET_VALUE)):
            idxs = sorted({int(k.split(".")[1]) for k in sd if k.startswith(net + ".")})
            for n, i in enumerate(idxs):
                w = g(f"{net}.{i}.weight")
                relu = (net == "common") or (n + 1 < len(idxs))
                p.add_linear(which, w.T.flatten(), g(f"{net}.{i}.bias"), relu)
        if len(obs_perms):
            p.set_perms(obs_perms, act_perms)
        return p

    @classmethod
    def from_conv1d_state_dict(cls, sd, obs_shape, conv_dim, obs_perms=(), act_perms=()):
        """Conv1dPolicy weights -> oracle policy, mirroring embeddingbag_to_rust's Conv1d branch
        (src/twisterl/nn/utils.py:68-75): vectors = conv weight [v, n_in, 1] squeezed and transposed, zero bias."""
        g = lambda k: np.asarray(sd[k], dtype=np.float32)
        p = cls()
        w = g("conv_layer.weight")[:, :, 0]
        p.set_embedding(w.T, np.zeros(w.shape[0] * obs_shape[1 - conv_dim], np.float32), True, list(obs_shape), conv_dim)
        for net, which in (("common", NET_COMMON), ("action", NET_ACTION), ("value", NET_VALUE)):
            p.add_linear(which, g(f"{net}.0.weight").T.flatten(), g(f"{net}.0.bias"), net == "common")
        if len(obs_perms):
            p.set_perms(obs_perms, act_perms)
        return p

    def _call(self, fn, obs, masks, perm):
        o = np.ascontiguousarray(obs, dtype=np.int32)
        out = np.zeros(256, dtype=np.float32)
        val = C.c_float()
        if masks is None:
            n = fn(self._h, _p(o, C.c_int32), len(o), int(perm), _p(out, C.c_float), C.byref(val))
        else:
            m = np.ascontiguousarray(masks, dtype=np.uint8)
            if perm is None:
                n = fn(self._h, _p(o, C.c_int32), len(o), _p(m, C.c_uint8), _p(out, C.c_float), C.byref(val))
            else:
                n = fn(self._h, _p(o, C.c_int32), len(o), _p(m, C.c_uint8), int(perm), _p(out, C.c_float),
                       C.byref(val))
        assert n >= 0
        return out[:n].copy(), np.float32(val.value)

    def raw_predict(self, obs, perm=-1): return self._call(lib().orc_policy_raw_predict, obs, None, perm)
    def forward(self, obs, masks, perm=-1): return self._call(lib().orc_policy_forward, obs, masks, perm)
    def predict(self, obs, masks, perm=-1): return self._call(lib().orc_policy_predict, obs, masks, perm)
    def full_predict(self, obs, masks): return self._call(lib().orc_policy_full_predict, obs, masks, None)


def argmax(v) -> int:
    a = np.ascontiguousarray(v, dtype=np.float32)
    return int(lib().orc_argmax(_p(a, C.c_float), len(a)))


def sample_from_logits(logits, uniforms) -> int:
    l = np.ascontiguousarray(logits, dtype=np.float32)
    u = np.ascontiguousarray(uniforms, dtype=np.float32)
    return int(lib().orc_sample_from_logits(_p(l, C.c_float), len(l), _p(u, C.c_float)))


def gae(rewards, values, gamma, lam):
    r = np.ascontiguousarray(rewards, dtype=np.float32)
    v = np.ascontiguousarray(values, dtype=np.float32)
    adv = np.zeros_like(r); ret = np.zeros_like(r)
    lib().orc_gae(r.ctypes.data, v.ctypes.data, len(r), gamma, lam, adv.ctypes.data, ret.ctypes.data)
    return adv, ret


def merge_order(n) -> np.ndarray:
    o = np.zeros(n, dtype=np.int32)
    lib().orc_merge_order(n, _p(o, C.c_int32))
    return o


def ppo_collect(spec: EnvSpec, policy: Policy, num_episodes, gamma, lam, seed=0, collect_id=0, env_id_base=0,
                num_threads=None) -> dict:
    if num_threads is None:
        num_threads = os.cpu_count() or 1
    c = _Collected()
    rc = lib().orc_ppo_collect(C.byref(spec), policy._h, int(num_episodes), float(gamma), float(lam), int(seed),
                               int(collect_id), int(env_id_base), int(num_threads), C.byref(c))
    if rc != 0:
        raise RuntimeError("oracle ppo_collect failed")
    R, nc, na = c.n_records, c.n_cells, c.num_actions
    arr = lambda ptr, shape, dt: np.ctypeslib.as_array(ptr, shape=shape).astype(dt, copy=True)
    out = dict(
        n_records=int(R), ep_len=arr(c.ep_len, (c.num_episodes,), np.int32),
        obs=arr(c.obs, (R, nc), np.int32), logits=arr(c.logits, (R, na), np.float32),
        values=arr(c.values, (R,), np.float32), rewards=arr(c.rewards, (R,), np.float32),
        advs=arr(c.advs, (R,), np.float32), rets=arr(c.rets, (R,), np.float32),
        actions=arr(c.actions, (R,), np.int32), perms=arr(c.perms, (R,), np.int32))
    lib().orc_collected_free(C.byref(c))
    return out


def time_ppo_collect(spec: EnvSpec, policy: Policy, num_episodes, gamma, lam, seed, collect_id, num_threads):
    """Run the collect and free it without copying out: (n_records, seconds).  Used by bench.py."""
    import time
    c = _Collected()
    t0 = time.perf_counter()
    rc = lib().orc_ppo_collect(C.byref(spec), policy._h, int(num_episodes), float(gamma), float(lam), int(seed),
                               int(collect_id), 0, int(num_threads), C.byref(c))
    dt = time.perf_counter() - t0
    if rc != 0:
        raise RuntimeError("oracle ppo_collect failed")
    n = int(c.n_records)
    lib().orc_collected_free(C.byref(c))
    return n, dt


def solve(env: Env, policy: Policy, deterministic, num_searches, seed=0, collect_id=0, id0=0, num_mcts_searches=0,
          c_puct=1.41, max_expand_depth=1):
    """((success, reward), actions) like collector.solve (rl/solve.rs:73-101), from the env's current state."""
    acts = np.zeros(4096, dtype=np.int32)
    s, r, n = C.c_float(), C.c_float(), C.c_int32()
    lib().orc_solve_mcts(C.byref(env._e), policy._h, int(bool(deterministic)), int(num_searches), int(num_mcts_searches),
                         float(c_puct), int(max_expand_depth), int(seed), int(collect_id),
                         int(id0), C.byref(s), C.byref(r), acts.ctypes.data, C.byref(n))
    return (float(s.value), float(r.value)), acts[: n.value].tolist()


class _AzCollected(C.Structure):
    _fields_ = [("n_records", C.c_int64), ("num_episodes", C.c_int32), ("n_cells", C.c_int32), ("num_actions", C.c_int32),
                ("ep_len", C.POINTER(C.c_int32)), ("obs", C.POINTER(C.c_int32)), ("probs", C.POINTER(C.c_float)),
                ("rewards", C.POINTER(C.c_float)), ("actions", C.POINTER(C.c_int32)),
                ("remaining_values", C.POINTER(C.c_float))]


def mcts_probs(env: Env, policy: Policy, n_sims, c_puct, max_expand_depth, seed=0, collect_id=0, stream_id=0, t=0):
    """(probs, visit counts) of predict_probs_mcts (rl/search.rs:104-189) from the env's current state."""
    probs = np.zeros(policy.num_actions, dtype=np.float32)
    visits = np.zeros(policy.num_actions, dtype=np.int32)
    f = lib().orc_mcts_probs
    f.argtypes = [C.POINTER(_Env), C.c_void_p, C.c_int32, C.c_float, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int32,
                  C.c_void_p, C.c_void_p]
    f(C.byref(env._e), policy._h, int(n_sims), float(c_puct), int(max_expand_depth), int(seed), int(collect_id),
      int(stream_id), int(t), probs.ctypes.data, visits.ctypes.data)
    return probs, visits


def mcts_trace(env: Env, policy: Policy, n_sims, c_puct, max_expand_depth, seed=0, collect_id=0, stream_id=0, t=0,
               path_lengths=False):
    """mcts_probs plus the per-simulation trace: (probs, visits, leaf[n_sims], backed_up_node[n_sims], margin[n_sims]),
    with path_lengths=True also path_len[n_sims], the number of nodes each simulation's backup updated (root and
    backed-up node included)."""
    probs = np.zeros(policy.num_actions, dtype=np.float32)
    visits = np.zeros(policy.num_actions, dtype=np.int32)
    leaf = np.zeros(max(n_sims, 1), dtype=np.int32); child = np.zeros(max(n_sims, 1), dtype=np.int32)
    margin = np.zeros(max(n_sims, 1), dtype=np.float32); path_len = np.zeros(max(n_sims, 1), dtype=np.int32)
    f = lib().orc_mcts_trace
    f.argtypes = [C.POINTER(_Env), C.c_void_p, C.c_int32, C.c_float, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int32,
                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    f.restype = None
    f(C.byref(env._e), policy._h, int(n_sims), float(c_puct), int(max_expand_depth), int(seed), int(collect_id),
      int(stream_id), int(t), probs.ctypes.data, visits.ctypes.data, leaf.ctypes.data, child.ctypes.data, margin.ctypes.data,
      path_len.ctypes.data)
    out = (probs, visits, leaf[:n_sims], child[:n_sims], margin[:n_sims])
    return out + (path_len[:n_sims],) if path_lengths else out


def az_collect(spec: EnvSpec, policy: Policy, num_episodes, n_sims, c_puct, max_expand_depth, seed=0, collect_id=0,
               env_id_base=0) -> dict:
    c = _AzCollected()
    f = lib().orc_az_collect
    f.argtypes = [C.POINTER(EnvSpec), C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_uint64, C.c_uint32,
                  C.c_uint32, C.POINTER(_AzCollected)]
    if f(C.byref(spec), policy._h, int(num_episodes), int(n_sims), float(c_puct), int(max_expand_depth), int(seed),
         int(collect_id), int(env_id_base), C.byref(c)) != 0:
        raise RuntimeError("oracle az_collect failed")
    R, nc, na = c.n_records, c.n_cells, c.num_actions
    arr = lambda ptr, shape, dt: np.ctypeslib.as_array(ptr, shape=shape).astype(dt, copy=True)
    out = dict(n_records=int(R), ep_len=arr(c.ep_len, (c.num_episodes,), np.int32), obs=arr(c.obs, (R, nc), np.int32),
               probs=arr(c.probs, (R, na), np.float32), rewards=arr(c.rewards, (R,), np.float32),
               actions=arr(c.actions, (R,), np.int32), remaining_values=arr(c.remaining_values, (R,), np.float32))
    lib().orc_az_collected_free(C.byref(c))
    return out


def evaluate(spec: EnvSpec, policy: Policy, num_episodes, deterministic, num_searches, seed=0, collect_id=0,
             reset_base=0, search_base=0, num_mcts_searches=0, c_puct=1.41, max_expand_depth=1):
    """(success_rate, mean_reward, per-episode best success, per-episode best reward) (rl/evaluate.rs:22-89)."""
    bs = np.zeros(num_episodes, dtype=np.float32); bt = np.zeros(num_episodes, dtype=np.float32)
    s, r = C.c_float(), C.c_float()
    lib().orc_evaluate_mcts(C.byref(spec), policy._h, int(num_episodes), int(bool(deterministic)), int(num_searches),
                            int(num_mcts_searches), float(c_puct), int(max_expand_depth), int(seed),
                            int(collect_id), int(reset_base), int(search_base), C.byref(s), C.byref(r), bs.ctypes.data,
                            bt.ctypes.data)
    return float(s.value), float(r.value), bs, bt


def evaluate_margins(spec: EnvSpec, policy: Policy, num_episodes, deterministic, num_searches, seed=0, collect_id=0,
                     reset_base=0, search_base=0, num_mcts_searches=0, c_puct=1.41, max_expand_depth=1):
    """(per-episode best success, best reward, smallest decision margin) -- see orc_evaluate_margins."""
    bs = np.zeros(num_episodes, dtype=np.float32); bt = np.zeros(num_episodes, dtype=np.float32)
    mm = np.zeros(num_episodes, dtype=np.float32)
    f = lib().orc_evaluate_margins
    f.argtypes = [C.POINTER(EnvSpec), C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_uint64,
                  C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    f.restype = None
    f(C.byref(spec), policy._h, int(num_episodes), int(bool(deterministic)), int(num_searches), int(num_mcts_searches),
      float(c_puct), int(max_expand_depth), int(seed), int(collect_id), int(reset_base), int(search_base),
      bs.ctypes.data, bt.ctypes.data, mm.ctypes.data)
    return bs, bt, mm
