"""twisterl_b200 -- B200-native rollout engine behind twisteRL's `twisterl.twisterl` API.

Submodules mirror the reference's PyO3 module (rust/src/python_interface/python_bindings.rs:55-77):
`env`, `nn`, `collector`.  `install_as_twisterl()` registers this package as `twisterl.twisterl`
(and the example crate's `grid_world`), so the reference's Python half (trainers, configs,
checkpoint loading) runs unmodified on top of the CUDA engine.
"""
from __future__ import annotations

import sys
import types

from . import _lib, collector, env, nn
from ._lib import Engine, configure, default_engine

__all__ = ["env", "nn", "collector", "Engine", "configure", "default_engine", "install_as_twisterl", "accelerate"]
__version__ = "0.1.0"


def install_as_twisterl() -> types.ModuleType:
    """Make `from twisterl import twisterl` / `import grid_world` resolve to this engine."""
    mod = types.ModuleType("twisterl.twisterl")
    mod.__doc__ = "twisterl_b200 standing in for the Rust extension twisterl.twisterl"
    mod.env, mod.nn, mod.collector = env, nn, collector
    sys.modules["twisterl.twisterl"] = mod
    for sub in ("env", "nn", "collector"):
        sys.modules[f"twisterl.twisterl.{sub}"] = getattr(mod, sub)
    gw = types.ModuleType("grid_world")
    gw.GridWorld = env.GridWorld
    sys.modules["grid_world"] = gw
    pkg = sys.modules.get("twisterl")
    if pkg is not None:
        pkg.twisterl = mod
    return mod


def accelerate(algorithm, comm=None):
    """Opt-in fast paths for a reference `twisterl.rl` Algorithm object that already runs on this engine (SURVEY.md 8f
    rows f2 / f3).  The reference's source stays untouched; three of the INSTANCE's methods are replaced:

    * `sync_rs_policy` (rl/algorithm.py:91-93): the live CUDA parameters are copied device-to-device into the engine's
      policy (`nn.Policy.update_from_torch`) instead of `to_rust()`'s trip through Python lists;
    * `collect` + `data_to_torch` (rl/algorithm.py:101-104, rl/ppo.py:25-61; PPO only): the collect stays on the device
      (`PPOCollector.collect_torch`) and the training tensors are built there -- same tuple, same arithmetic
      (advantage normalisation, Categorical log-probs of the recorded masked logits) as the reference's data_to_torch.

    With a `dist.Comm` (on the root rank), `collect` runs on every rank's GPU: `algorithm.collector.num_episodes`
    is the total, sharded over the ranks and gathered to this one (`dist.ShardedCollector`, kept as
    `algorithm.sharded_collector`; its `close()` stops the other ranks, which run its `serve`).  PPO collects through
    `collect_torch`, AZ through `collect`.

    Returns the algorithm."""
    import time
    import types

    def timed(fn):                                     # the reference's @timed contract: (result, seconds)
        def wrapper(self, *a, **kw):
            t0 = time.perf_counter_ns()
            out = fn(self, *a, **kw)
            return out, (time.perf_counter_ns() - t0) / 1e9
        return wrapper

    def sync_rs_policy(self):
        try:
            self.rs_pol.update_from_torch(self.policy)
        except (NotImplementedError, AttributeError):  # other embedding kinds: the reference's own export
            self.rs_pol = self.policy.to_rust()

    algorithm.sync_rs_policy = types.MethodType(timed(sync_rs_policy), algorithm)
    sharded = None
    if comm is not None:
        from .dist import ShardedCollector
        sharded = algorithm.sharded_collector = ShardedCollector(algorithm.collector, comm)
    if isinstance(getattr(algorithm, "collector", None), collector.PPOCollector):
        def collect(self):
            return (sharded or self.collector).collect_torch(self.env, self.rs_pol, dense_obs=True)

        def data_to_torch(self, data):
            import torch
            advs = data["advs"]
            with torch.no_grad():
                if self.config["training"].get("normalize_advantage", False):
                    advs = (advs - advs.mean()) / (advs.std() + 1e-8)
                log_probs = torch.distributions.Categorical(logits=data["logits"]).log_prob(data["actions"])
            return data["obs"], log_probs, data["actions"], advs, data["rets"], data["perms"]

        algorithm.collect = types.MethodType(timed(collect), algorithm)
        algorithm.data_to_torch = types.MethodType(timed(data_to_torch), algorithm)
    elif sharded is not None:
        def collect(self):
            return sharded.collect(self.env, self.rs_pol)

        algorithm.collect = types.MethodType(timed(collect), algorithm)
    return algorithm
