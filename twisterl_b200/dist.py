"""Multi-GPU plumbing: one process per GPU, independent env shards, replicated weights.

The rollout itself has no exchange step (episodes are independent, SURVEY.md section 8e); per iteration there is one
broadcast of the flat fp32 weight blob from the trainer rank and one all-reduce of a small statistics vector, and a
trainer on one rank receives every rank's episodes with one gather (`ShardedCollector`).  On the GPUs these are NCCL
calls made by the library itself (`twr_broadcast_weights` / `twr_allreduce_stats` / `twr_gather_collected` of the C ABI,
on the engine's stream) -- what a Rust or C++ host would call; `torch.distributed` (gloo, CPU) only carries the 128-byte
NCCL unique id from rank 0 to the other ranks and the ShardedCollector's per-iteration command, and stands in for NCCL in
the CPU tests of this host logic.
"""
from __future__ import annotations

import copy
import ctypes as C
import os

import numpy as np

STATS_FIELDS = ("episodes", "successes", "reward_sum", "records")


def env_id_base(rank: int, num_episodes: int) -> int:
    """First global env id of this rank's shard: rank r owns [r*E, (r+1)*E).  The Philox streams are keyed
    by global env id, so a rollout does not depend on how many GPUs it was sharded over."""
    return int(rank) * int(num_episodes)


def _stats_dict(v) -> dict:
    return {"episodes": int(v[0]), "successes": int(v[1]), "reward_sum": float(v[2]), "records": int(v[3]),
            "success_rate": v[1] / max(v[0], 1.0), "mean_reward": v[2] / max(v[0], 1.0)}


class Comm:
    """The exchanges of one rank.  `engine` given: NCCL through the C ABI (the communicator lives in the engine);
    `engine=None`: torch.distributed's default group (gloo in the CPU tests).  world == 1: every call is a no-op."""

    def __init__(self, engine=None, rank: int | None = None, world: int | None = None):
        self.engine = engine
        self.rank = int(os.environ.get("RANK", "0")) if rank is None else int(rank)
        self.world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else int(world)
        self.backend = "none"
        if self.world == 1:
            return
        import torch.distributed as dist
        if not dist.is_initialized():                  # bootstrap channel only (MASTER_ADDR / MASTER_PORT from the launcher)
            dist.init_process_group("gloo", rank=self.rank, world_size=self.world)
        self._dist = dist
        if engine is None:
            self.backend = "gloo"
            return
        from . import _lib
        if (engine.rank, engine.world) != (self.rank, self.world):
            raise ValueError("engine rank/world differ from the launcher's")
        L = _lib.load()
        uid = np.zeros(128, np.uint8)
        if self.rank == 0:
            _lib.check(L.twr_comm_unique_id(_lib.ptr(uid)))
        box = [uid.tobytes()]
        dist.broadcast_object_list(box, src=0)
        uid = np.frombuffer(box[0], np.uint8).copy()
        _lib.check(L.twr_comm_init(engine._h, _lib.ptr(uid)))
        self.backend = f"nccl {L.twr_comm_version()} via the C ABI"

    # ---- per-iteration exchanges -----------------------------------------------------------------
    def broadcast_weights(self, target, root: int = 0):
        """NCCL path: `target` is a policy handle (twr_policy*) -- rank `root`'s blob reaches every engine and the operand
        layouts are rebuilt.  gloo path: `target` is a torch tensor, broadcast in place."""
        if self.engine is not None:
            from . import _lib
            _lib.check(_lib.load().twr_broadcast_weights(self.engine._h, target, int(root)))
        elif self.world > 1:
            self._dist.broadcast(target, src=root)
        return target

    def allreduce(self, values, op: str = "sum") -> list:
        v = np.ascontiguousarray(values, dtype=np.float64)
        if self.world == 1:
            return v.tolist()
        if self.engine is not None:
            from . import _lib
            _lib.check(_lib.load().twr_allreduce_stats(self.engine._h, _lib.ptr(v), int(v.size), 1 if op == "max" else 0))
            return v.tolist()
        import torch
        t = torch.from_numpy(v)
        self._dist.all_reduce(t, op=self._dist.ReduceOp.MAX if op == "max" else self._dist.ReduceOp.SUM)
        return t.tolist()

    def allreduce_stats(self, episodes: int, successes: int, reward_sum: float, records: int) -> dict:
        return _stats_dict(self.allreduce([episodes, successes, reward_sum, records]))

    def gather_collected(self, root: int = 0):
        """twr_gather_collected: collective over the ranks, each of which has just run a device-resident collect of the
        same shape.  Returns the `_lib.Collected` struct: on `root` the merged result of every rank (in the order one
        collect of all their episodes lays out), elsewhere the rank's own result.  Needs the engine (NCCL) path."""
        if self.engine is None:
            raise RuntimeError("gather_collected needs a Comm over an engine")
        from . import _lib
        c = _lib.Collected()
        _lib.check(_lib.load().twr_gather_collected(self.engine._h, int(root), C.byref(c)))
        return c

    def max_over_ranks(self, x: float) -> float:
        return float(self.allreduce([x], op="max")[0])

    def barrier(self):
        if self.world > 1:
            self.allreduce([0.0])

    def close(self):
        if self.engine is not None and self.world > 1 and getattr(self.engine, "_h", None):
            from . import _lib
            _lib.load().twr_comm_destroy(self.engine._h)
        if self.world > 1 and self._dist.is_initialized():
            self._dist.destroy_process_group()


STOP = -1          # ShardedCollector command: the workers leave serve()


class ShardedCollector:
    """A `PPOCollector` / `AZCollector` of `collector.num_episodes` episodes IN TOTAL, sharded over the `comm.world` engines
    of a job: rank r collects the global episode ids [r*E, (r+1)*E), E = total / world, and rank `root` receives every
    shard, merged in the order one collect of all of them on one engine lays out -- byte for byte that collect, for the
    same seed, collect id and precision.

    Root calls `collect` / `collect_torch`; every other rank calls `serve`.  Each iteration root broadcasts one command over
    the gloo group (its env's difficulty, or STOP, and the collect id), then the weights; every rank pins that collect id
    on its engine, collects its shard and joins the gather.  The collect ids are this object's own counter, starting at
    `collect_id` and advancing by one per iteration: whatever else root's engine runs between iterations (an evaluate,
    a solve) leaves the ranks' Philox streams in step.  A rank whose collect raised still joins the gather, so no rank is
    left waiting, and re-raises afterwards (the gather fails alike on every rank).  `close()` on root stops the workers."""

    def __init__(self, collector, comm: Comm, root: int = 0, collect_id: int = 0):
        total = int(collector.num_episodes)
        if total <= 0 or total % comm.world:
            raise ValueError(f"ShardedCollector: {total} episodes do not split into {comm.world} equal shards "
                             "(global episode ids are rank * shard + i)")
        if not 0 <= int(root) < comm.world:
            raise ValueError("root out of range")
        self.comm, self.root = comm, int(root)
        self.local = copy.copy(collector)
        self.local.num_episodes = total // comm.world
        if comm.engine is not None:
            self.local._engine = comm.engine
        self.collect_id = int(collect_id)
        self._stopped = False

    @property
    def is_root(self) -> bool:
        return self.comm.rank == self.root

    def _command(self, cmd: int = 0, collect_id: int = 0) -> tuple[int, int]:
        """Root: sends (`cmd`, `collect_id`) to every rank, `cmd` an env difficulty >= 0 or STOP; other ranks: return
        the pair root sent."""
        if self.comm.world == 1:
            return int(cmd), int(collect_id)
        import torch
        t = torch.tensor([int(cmd), int(collect_id)], dtype=torch.int64)
        self.comm._dist.broadcast(t, src=self.root)
        return int(t[0]), int(t[1])

    def _iteration(self, env, policy, difficulty: int, collect_id: int):
        env.difficulty = difficulty
        eng = self.comm.engine
        self.comm.broadcast_weights(policy.device_handle(eng), root=self.root)
        eng.set_collect_id(collect_id)
        err = None
        try:
            self.local.collect_device(env, policy)
        except Exception as exc:
            err = exc
        try:
            c = self.comm.gather_collected(self.root)
        except RuntimeError as gather_err:
            if err is not None:
                raise err from gather_err
            raise
        if err is not None:
            raise err
        return c

    def _root_iteration(self, env, policy):
        if not self.is_root:
            raise RuntimeError("ShardedCollector: only the root rank collects; the other ranks call serve()")
        if self._stopped:
            raise RuntimeError("ShardedCollector: closed")
        cmd = self._command(int(env.difficulty), self.collect_id)
        self.collect_id += 1
        return self._iteration(env, policy, *cmd)

    def collect(self, env, policy):
        """Root: one sharded collect of every rank, as the wrapped collector's `CollectedData` of all episodes."""
        return self.local.to_host(self._root_iteration(env, policy))

    def collect_torch(self, env, policy, dense_obs: bool = True) -> dict:
        """Root: one sharded PPO collect of every rank, as torch CUDA tensors on root's device over the gathered result
        (`collector.torch_views`; valid until the next collect or gather on root's engine)."""
        from .collector import PPOCollector, torch_views
        if not isinstance(self.local, PPOCollector):
            raise TypeError("collect_torch needs a PPOCollector")
        return torch_views(self._root_iteration(env, policy), self.comm.engine.device, dense_obs)

    def serve(self, env, policy) -> int:
        """The other ranks: collect and send a shard per root iteration until root closes.  Returns the iterations served."""
        if self.is_root:
            raise RuntimeError("ShardedCollector: the root rank collects; serve() is for the other ranks")
        n = 0
        while (cmd := self._command())[0] != STOP:
            self._iteration(env, policy, *cmd)
            n += 1
        return n

    def close(self):
        """Root: stops the workers (once)."""
        if self.is_root and not self._stopped:
            self._stopped = True
            self._command(STOP)
