"""Host logic of dist.ShardedCollector that needs no device: the equal-shard check and the per-iteration command protocol
between the root rank and the serving ranks, over a world_size-2 gloo group (the device collect and the gather are
replaced by recorders)."""
import os
import socket
from types import SimpleNamespace

import pytest
import torch.multiprocessing as mp


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


class _FakeCollector:
    def __init__(self, num_episodes):
        self.num_episodes = num_episodes

    def to_host(self, c):
        return c


def test_total_must_split_into_equal_shards():
    from twisterl_b200 import dist as twd
    two = SimpleNamespace(rank=0, world=2, engine=None)
    with pytest.raises(ValueError, match="equal shards"):
        twd.ShardedCollector(_FakeCollector(7), two)
    with pytest.raises(ValueError, match="equal shards"):
        twd.ShardedCollector(_FakeCollector(0), two)
    with pytest.raises(ValueError, match="root"):
        twd.ShardedCollector(_FakeCollector(8), two, root=2)
    sc = twd.ShardedCollector(_FakeCollector(8), two)
    assert sc.local.num_episodes == 4 and sc.local is not sc and sc.is_root and sc.collect_id == 0


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    from twisterl_b200 import dist as twd
    comm = twd.Comm()
    seen = []
    sc = twd.ShardedCollector(_FakeCollector(6 * world), comm, collect_id=40 if rank == 0 else 7)   # root's counter rules
    sc._iteration = lambda env, policy, difficulty, cid: seen.append([difficulty, cid]) or ("merged", difficulty)
    out = {"shard": sc.local.num_episodes}
    if rank == 0:
        with_err = []
        try:
            sc.serve(None, None)
        except RuntimeError as exc:
            with_err.append(str(exc))
        env = SimpleNamespace(difficulty=3)
        out["first"] = sc.collect(env, None)
        env.difficulty = 5
        out["second"] = sc.collect(env, None)
        sc.close()
        sc.close()                                  # the stop goes out once
        try:
            sc.collect(env, None)
        except RuntimeError as exc:
            with_err.append(str(exc))
        out["errors"] = with_err
    else:
        try:
            sc.collect(SimpleNamespace(difficulty=1), None)
        except RuntimeError as exc:
            out["errors"] = [str(exc)]
        out["served"] = sc.serve(None, None)
    out["seen"] = seen
    comm.barrier()                                  # a second stop from root would have been taken for this
    q.put((rank, out))
    comm.close()


def test_command_protocol_two_ranks():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = dict(q.get(timeout=120) for _ in procs)
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
                p.join()
    assert [p.exitcode for p in procs] == [0, 0]
    root, worker = res[0], res[1]
    assert root["shard"] == worker["shard"] == 6
    assert root["first"] == ("merged", 3) and root["second"] == ("merged", 5)
    assert root["seen"] == worker["seen"] == [[3, 40], [5, 41]]      # root's collect ids reach every rank
    assert worker["served"] == 2
    assert "serve() is for the other ranks" in root["errors"][0] and "closed" in root["errors"][1]
    assert "only the root rank collects" in worker["errors"][0]
