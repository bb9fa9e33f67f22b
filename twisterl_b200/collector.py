"""Host mirror of `twisterl.twisterl.collector` (rust/src/python_interface/collector.rs).

`PPOCollector(num_episodes, gamma, lambda, num_cores).collect(env, policy)` keeps the reference's
constructor keywords and blocking call; the work happens in `twr_ppo_collect` on the device and the
result comes back as NumPy arrays (`*_array` attributes) that the list-valued properties of
`CollectedData` wrap for drop-in compatibility.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .env import spec_from_env
from .nn import Policy


class CollectedData:
    """`collector.CollectedData(obs, logits, values, rewards, actions, perms=None)`
    (python_interface/collector.rs:24-137).  List-valued getters copy, like the PyO3 ones."""

    def __init__(self, obs, logits, values, rewards, actions, perms=None):
        self._obs, self._logits = obs, logits
        self._values, self._rewards, self._actions = values, rewards, actions
        self._perms = perms if perms is not None else [-1] * len(obs)
        self._additional: dict[str, object] = {}
        self.stats: dict = {}

    # ---- array views (zero-copy when the data came from the device path)
    @property
    def obs_array(self): return np.asarray(self._obs)
    @property
    def logits_array(self): return np.asarray(self._logits, dtype=np.float32)
    @property
    def values_array(self): return np.asarray(self._values, dtype=np.float32)
    @property
    def rewards_array(self): return np.asarray(self._rewards, dtype=np.float32)
    @property
    def actions_array(self): return np.asarray(self._actions)
    @property
    def perms_array(self): return np.asarray(self._perms)

    def additional_array(self, key): return np.asarray(self._additional[key], dtype=np.float32)

    # ---- reference properties
    @staticmethod
    def _ls(x):
        return x.tolist() if isinstance(x, np.ndarray) else list(x)

    obs = property(lambda s: s._ls(s._obs), lambda s, v: setattr(s, "_obs", v))
    logits = property(lambda s: s._ls(s._logits), lambda s, v: setattr(s, "_logits", v))
    values = property(lambda s: s._ls(s._values), lambda s, v: setattr(s, "_values", v))
    rewards = property(lambda s: s._ls(s._rewards), lambda s, v: setattr(s, "_rewards", v))
    actions = property(lambda s: s._ls(s._actions), lambda s, v: setattr(s, "_actions", v))

    @property
    def perms(self):
        return [int(p) if p is not None and int(p) >= 0 else -1 for p in self._ls(self._perms)]

    @perms.setter
    def perms(self, v):
        self._perms = [(-1 if (p is None or int(p) < 0) else int(p)) for p in v]

    @property
    def additional_data(self):
        return {k: self._ls(v) for k, v in self._additional.items()}

    @additional_data.setter
    def additional_data(self, d):
        self._additional = dict(d)

    def get_additional_data_item(self, key):
        v = self._additional.get(key)
        return None if v is None else self._ls(v)

    def set_additional_data_item(self, key, value):
        self._additional[key] = value

    def merge(self, other: "CollectedData") -> None:
        """CollectedData::merge (collector/collector.rs:70-88): append every vector."""
        cat = lambda a, b: (np.concatenate([np.asarray(a), np.asarray(b)]) if isinstance(a, np.ndarray)
                            else list(a) + self._ls(b))
        self._obs, self._logits = cat(self._obs, other._obs), cat(self._logits, other._logits)
        self._values, self._rewards = cat(self._values, other._values), cat(self._rewards, other._rewards)
        self._actions, self._perms = cat(self._actions, other._actions), cat(self._perms, other._perms)
        for k, v in other._additional.items():
            self._additional[k] = cat(self._additional[k], v) if k in self._additional else v


def _host_buffers(cap: int, n_cells: int, n_actions: int, num_episodes: int, pinned: bool, obs_u8: bool = False):
    """Caller-owned host buffers of one collect.  `obs_u8` asks twr_ppo_collect_host for one-byte observation
    indices (obs_size <= 256) through twr_host_buffers.obs_u8 instead of the u16 `obs` field."""
    mk = (lambda shape, dt: _lib.PinnedArray(shape, dt)) if pinned else None
    fields = dict(obs=((cap, n_cells), np.uint8 if obs_u8 else np.uint16), logits=((cap, n_actions), np.float32), values=((cap,), np.float32),
                  rewards=((cap,), np.float32), advs=((cap,), np.float32), rets=((cap,), np.float32),
                  actions=((cap,), np.uint8), perms=((cap,), np.int8), ep_len=((num_episodes,), np.int32))
    holders, arrays = {}, {}
    for k, (shape, dt) in fields.items():
        if pinned:
            holders[k] = mk(shape, dt)
            arrays[k] = holders[k].array
        else:
            arrays[k] = np.empty(shape, dtype=dt)
    ptr = {k: C.c_void_p(arrays[k].ctypes.data) for k in arrays}
    hb = _lib.HostBuffers(cap, None if obs_u8 else ptr["obs"], *[ptr[k] for k in
                          ("logits", "values", "rewards", "advs", "rets", "actions", "perms", "ep_len")],
                          ptr["obs"] if obs_u8 else None)
    return hb, arrays, holders


def torch_views(c: _lib.Collected, device: int, dense_obs: bool = True) -> dict:
    """Torch CUDA tensors over the device-resident result `c` describes (a collect, or root's gathered result of
    twr_gather_collected), aliasing the engine's buffers: valid until the next collect / gather on that engine.
    Keys: obs (dense one-hot float [R, obs_size] or int64 indices [R, cells]), logits, actions, advs, rets, perms,
    values, rewards, stats."""
    import torch
    R, N, A = int(c.n_records), int(c.n_cells), int(c.num_actions)
    dev = torch.device("cuda", int(device))

    def view(ptr, shape, typestr):
        class _H:
            __cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (int(ptr), False), "version": 2}
        return torch.as_tensor(_H(), device=dev)

    idx = view(c.obs, (R, N), "<u2").to(torch.int64)
    out = {"logits": view(c.logits, (R, A), "<f4"), "values": view(c.values, (R,), "<f4"),
           "rewards": view(c.rewards, (R,), "<f4"), "advs": view(c.advs, (R,), "<f4"), "rets": view(c.rets, (R,), "<f4"),
           "actions": view(c.actions, (R,), "|u1").to(torch.int64), "perms": view(c.perms, (R,), "|i1").to(torch.int64)}
    if dense_obs:
        obs = torch.zeros((R, N * N), dtype=torch.float32, device=dev)
        obs.scatter_(1, idx, 1.0)
        out["obs"] = obs
    else:
        out["obs"] = idx
    out["stats"] = dict(episodes=int(c.num_episodes), successes=int(c.successes), reward_sum=float(c.reward_sum), records=R)
    return out


class PyBaseCollector:
    """`collector.PyBaseCollector` (python_interface/collector.rs:139-152)."""

    def collect(self, env, policy):
        raise NotImplementedError


class PPOCollector(PyBaseCollector):
    """`collector.PPOCollector(num_episodes, gamma, lambda, num_cores)` (python_interface/collector.rs:154-170;
    PPOCollector::collect rust/src/collector/ppo.rs:108-126).  `num_cores` is accepted for
    compatibility: episodes are spread over the GPU's SMs instead of a rayon pool."""

    _ARGS = ("num_episodes", "gamma", "lambda", "num_cores")

    def __init__(self, *args, **kwargs):
        if len(args) > len(self._ARGS):
            raise TypeError(f"PPOCollector takes {len(self._ARGS)} arguments")
        vals = dict(zip(self._ARGS, args))
        for k, v in kwargs.items():
            if k == "engine":
                continue
            if k not in self._ARGS:
                raise TypeError(f"PPOCollector() got an unexpected keyword argument '{k}'")
            if k in vals:
                raise TypeError(f"PPOCollector() got multiple values for argument '{k}'")
            vals[k] = v
        missing = [k for k in self._ARGS if k not in vals]
        if missing:
            raise TypeError(f"PPOCollector() missing required argument: '{missing[0]}'")
        self.num_episodes = int(vals["num_episodes"])
        self.gamma, self.lambda_ = float(vals["gamma"]), float(vals["lambda"])
        self.num_cores = int(vals["num_cores"])
        if self.num_episodes < 0 or self.num_cores < 0:
            raise OverflowError("can't convert negative int to unsigned")
        self._engine = kwargs.get("engine")
        self.pinned = False

    @property
    def engine(self) -> _lib.Engine:
        return self._engine or _lib.default_engine()

    def collect_device(self, env, policy: Policy) -> _lib.Collected:
        """Run the collect and leave the result in device memory (pointers in the returned struct)."""
        spec = spec_from_env(env)
        eng = self.engine
        out = _lib.Collected()
        _lib.check(_lib.load().twr_ppo_collect(eng._h, C.byref(spec), policy.device_handle(eng), self.num_episodes,
                                               self.gamma, self.lambda_, C.byref(out)))
        return out

    def collect_torch(self, env, policy: Policy, dense_obs: bool = True):
        """Device hand-off for a GPU trainer (SURVEY.md 8f row f2): run the collect and return torch CUDA tensors that
        alias the engine's output buffers (valid until the next collect on this engine) -- what
        `PPO.data_to_torch` (src/twisterl/rl/ppo.py:25-61) builds through Python lists and an H2D copy.
        Keys: see `torch_views`."""
        return torch_views(self.collect_device(env, policy), self.engine.device, dense_obs)

    def collect(self, env, policy: Policy) -> CollectedData:
        if not isinstance(policy, Policy):
            raise TypeError("argument 'policy': expected twisterl.nn.Policy")
        return self.to_host(self.collect_device(env, policy))

    def to_host(self, c: _lib.Collected) -> CollectedData:
        """CollectedData of the engine's last device-resident result, which `c` describes (twr_collected_to_host)."""
        eng = self.engine
        R = int(c.n_records)
        hb, arr, holders = _host_buffers(R, c.n_cells, c.num_actions, int(c.num_episodes), self.pinned)
        _lib.check(_lib.load().twr_collected_to_host(eng._h, C.byref(hb)))
        data = CollectedData(arr["obs"], arr["logits"], arr["values"], arr["rewards"], arr["actions"], arr["perms"])
        data.set_additional_data_item("advs", arr["advs"])
        data.set_additional_data_item("rets", arr["rets"])
        data.ep_len = arr["ep_len"]
        data.stats = dict(episodes=int(c.num_episodes), successes=int(c.successes), reward_sum=float(c.reward_sum),
                          records=R)
        data._holders = holders
        return data


class AZCollector(PyBaseCollector):
    """`collector.AZCollector(num_episodes, num_mcts_searches, C, max_expand_depth, num_cores)`
    (python_interface/collector.rs:172-188; AZCollector::collect rust/src/collector/az.rs:112-130): batched MCTS on the
    device, leaves evaluated by the same forward kernel as the PPO path."""

    def __init__(self, num_episodes, num_mcts_searches, C, max_expand_depth, num_cores, *, engine=None):
        self.num_episodes, self.num_mcts_searches = int(num_episodes), int(num_mcts_searches)
        self.C, self.max_expand_depth, self.num_cores = float(C), int(max_expand_depth), int(num_cores)
        self._engine = engine

    @property
    def engine(self) -> _lib.Engine:
        return self._engine or _lib.default_engine()

    def collect_device(self, env, policy: Policy) -> _lib.Collected:
        """Run the collect and leave the result in device memory (pointers in the returned struct)."""
        if not isinstance(policy, Policy):
            raise TypeError("argument 'policy': expected twisterl.nn.Policy")
        spec = spec_from_env(env)
        eng = self.engine
        c = _lib.Collected()
        _lib.check(_lib.load().twr_az_collect(eng._h, C.byref(spec), policy.device_handle(eng), self.num_episodes,
                                              self.num_mcts_searches, self.C, self.max_expand_depth, C.byref(c)))
        return c

    def collect(self, env, policy: Policy) -> CollectedData:
        return self.to_host(self.collect_device(env, policy))

    def to_host(self, c: _lib.Collected) -> CollectedData:
        """CollectedData of the engine's last device-resident result, which `c` describes (twr_collected_to_host)."""
        eng = self.engine
        R = int(c.n_records)
        hb, arr, holders = _host_buffers(R, c.n_cells, c.num_actions, int(c.num_episodes), False)
        _lib.check(_lib.load().twr_collected_to_host(eng._h, C.byref(hb)))
        # az.rs:97-104: obs, probs (in .logits), perms all None; values / rewards / actions stay empty
        data = CollectedData(arr["obs"], arr["logits"], [], [], [], np.full(R, -1, dtype=np.int8))
        data.set_additional_data_item("remaining_values", arr["rets"])
        data.ep_len = arr["ep_len"]
        data.step_rewards, data.step_actions = arr["rewards"], arr["actions"]    # extras, not part of the reference object
        data.stats = dict(episodes=int(c.num_episodes), successes=int(c.successes), reward_sum=float(c.reward_sum), records=R)
        return data


def solve(env, policy, deterministic, num_searches, num_mcts_searches, C, max_expand_depth):
    """`collector.solve` (python_interface/env.rs:180-191; rl/solve.rs:73-101): best of `num_searches` rollouts
    from the env's CURRENT state -> ((success, reward), actions)."""
    spec_from_env(env)                       # rejects envs without a device implementation
    eng = _lib.default_engine()
    import ctypes as ct
    batch = env._b()
    if batch.engine is not eng:
        raise RuntimeError("env state lives on another engine")
    cap = int(batch.depth()[0]) + 1
    acts = np.zeros(cap, dtype=np.int32)
    succ, rew, n = ct.c_float(), ct.c_float(), ct.c_int32()
    _lib.check(_lib.load().twr_solve(eng._h, batch._h, policy.device_handle(eng), int(bool(deterministic)), int(num_searches),
                                     int(num_mcts_searches), float(C), int(max_expand_depth),
                                     ct.byref(succ), ct.byref(rew), _lib.ptr(acts), cap, ct.byref(n)))
    return (float(succ.value), float(rew.value)), [int(a) for a in acts[: n.value]]


def evaluate(env, policy, num_episodes, deterministic, num_searches, num_mcts_searches, seed, C, max_expand_depth,
             num_cores):
    """`collector.evaluate` (python_interface/env.rs:194-207; rl/evaluate.rs:22-89) -> (success rate, mean reward).
    `seed` is ignored like in the reference; `num_cores` is accepted for compatibility."""
    spec = spec_from_env(env)
    eng = _lib.default_engine()
    import ctypes as ct
    s, r = ct.c_float(), ct.c_float()
    _lib.check(_lib.load().twr_evaluate(eng._h, ct.byref(spec), policy.device_handle(eng), int(num_episodes),
                                        int(bool(deterministic)), int(num_searches), int(num_mcts_searches), float(C),
                                        int(max_expand_depth), ct.byref(s), ct.byref(r)))
    return float(s.value), float(r.value)
