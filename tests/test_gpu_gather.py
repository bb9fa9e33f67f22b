"""Multi-GPU gather (twr_gather_collected, dist.ShardedCollector): one process per GPU, W engines each collect E episodes
and rank 0 receives all of them.  Every random draw is keyed by the global episode id (DESIGN.md section 3), so the
merged result must equal, byte for byte, one engine's collect of W*E episodes with the same seed, precision and collect
id -- a differing byte is a defect of that invariance, not a tolerance to widen.  The ranks also agree on every refusal
(no rank is left blocked in a collective), and the sharded collector keeps them in lockstep over iterations.

W = 2, and W = torch.cuda.device_count() when that is larger (up to 8).  Every rank runs all cases in one spawn per W;
rank 0 writes what it received under a temporary directory, and the parent compares with its own single-engine collect.
"""
import hashlib
import json
import os
import socket
import time
import traceback
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

from helpers import synth_state_dict, trained15, transpose_twists

pytestmark = pytest.mark.gpu

SEED = 0x5EED0017
GAMMA = LAM = 0.995
PRECISIONS = ("f16f8c", "fp32")           # the CTA-pair tensor-core kernel and the fp32 SIMT kernel
# name, env (kind, constructor args), episodes per rank, twists
PPO_CASES = [
    ("puzzle15_d32", ("puzzle", 4, 4, 32, 2, 256), 300, False),
    ("puzzle15_d32_twists", ("puzzle", 4, 4, 32, 2, 256), 300, True),
    ("puzzle8", ("puzzle", 3, 3, 6, 2, 256), 300, False),
    ("gridworld5", ("gridworld", 5, 5, 64, 10), 300, False),
    # several tiles per CTA pair per rank (74 pairs x 256 envs a round on a B200), chunks of >= 4 steps: the balanced
    # schedule of the pair kernel runs on every shard and on the single-engine collect alike
    ("puzzle15_d16_large", ("puzzle", 4, 4, 16, 2, 256), 40960, False),
]
AZ_ENV, AZ_EPISODES, AZ_SIMS = ("puzzle", 3, 3, 4, 2, 16), 24, 8
ERR_EPISODES = 64
SHARD_EPISODES, SHARD_CID, SHARD_DIFFICULTIES = 200, 900, (3, 5)
SAVE_LIMIT = 32 << 20                       # larger arrays travel as a SHA-256 digest
JOIN_TIMEOUT = 900


def _cid(i, j):
    return 100 + 10 * i + j


def _env(spec, add_perms=False):
    import twisterl_b200 as tw
    kind, *a = spec
    return tw.env.Puzzle(*a, add_perms=add_perms) if kind == "puzzle" else tw.env.GridWorld(*a)


def _policy(spec, twists, seed=21):
    from parity import make_policies
    kind, w, h = spec[:3]
    if (kind, w, h) == ("puzzle", 4, 4):
        _, sd = trained15()
        obs = 256
    else:
        obs = 81 if kind == "puzzle" else 625
        sd = synth_state_dict(seed, obs, 512, 256 if kind == "puzzle" else 128, 4)
    return make_policies(sd, obs, *(transpose_twists(4) if twists else ((), ())))[0]


def _ppo_arrays(d):
    return {"obs": d.obs_array, "logits": d.logits_array, "values": d.values_array, "rewards": d.rewards_array,
            "advs": d.additional_array("advs"), "rets": d.additional_array("rets"), "actions": d.actions_array,
            "perms": d.perms_array, "ep_len": d.ep_len}


def _az_arrays(d):
    return {"obs": d.obs_array, "logits": d.logits_array, "remaining_values": d.additional_array("remaining_values"),
            "rewards": np.asarray(d.step_rewards), "actions": np.asarray(d.step_actions), "ep_len": d.ep_len}


def _save(path, arrays, stats):
    out = {"stats": json.dumps(stats)}
    for k, a in arrays.items():
        a = np.ascontiguousarray(a)
        out[k] = a if a.nbytes <= SAVE_LIMIT else np.array(f"sha256:{a.dtype.str}:{a.shape}:" + hashlib.sha256(a.tobytes()).hexdigest())
    np.savez(path, **out)


def _assert_same(path, arrays, stats):
    """Rank 0's saved arrays / statistics against the single-engine collect's: bytes equal, reward sums to 1e-12."""
    z = np.load(path)
    got = json.loads(str(z["stats"]))
    for k in ("episodes", "records", "successes"):
        assert got[k] == stats[k], (k, got[k], stats[k])
    assert abs(got["reward_sum"] - stats["reward_sum"]) <= 1e-12 * max(1.0, abs(stats["reward_sum"]))
    for k, a in arrays.items():
        if a is None:
            continue
        a = np.ascontiguousarray(a)
        g = z[k]
        if g.dtype.kind == "U":
            assert str(g) == f"sha256:{a.dtype.str}:{a.shape}:" + hashlib.sha256(a.tobytes()).hexdigest(), k
            continue
        assert g.dtype == a.dtype and g.shape == a.shape, (k, g.dtype, g.shape, a.dtype, a.shape)
        gb, ab = g.reshape(len(g), -1).view(np.uint8), a.reshape(len(a), -1).view(np.uint8)
        bad = np.flatnonzero((gb != ab).any(axis=1))
        assert bad.size == 0, f"{k}: {bad.size} rows differ, first at {bad[:8].tolist()}"


def _torch_arrays(t):
    """collect_torch output as host arrays in the dtypes of CollectedData's (observation indices only when they were
    asked for: dense_obs=False)."""
    a = {k: t[k].cpu().numpy() for k in ("logits", "values", "rewards", "advs", "rets")}
    if not t["obs"].is_floating_point():
        a["obs"] = t["obs"].cpu().numpy().astype(np.uint16)
    a["actions"] = t["actions"].cpu().numpy().astype(np.uint8)
    a["perms"] = t["perms"].cpu().numpy().astype(np.int8)
    return a


def _evaluate(eng, env, pol):
    """collector.evaluate on `eng` (it advances the engine's collect id, as a trainer's curriculum check does)."""
    import ctypes as C
    import twisterl_b200 as tw
    from twisterl_b200 import _lib
    spec = tw.env.spec_from_env(env)
    s, r = C.c_float(), C.c_float()
    _lib.check(_lib.load().twr_evaluate(eng._h, C.byref(spec), pol.device_handle(eng), 64, 0, 1, 0, 1.41, 1,
                                        C.byref(s), C.byref(r)))


# ------------------------------------------------------------------------------------------------ ranks ---
def _gather_error(comm, root=0):
    try:
        comm.gather_collected(root)
        return None
    except RuntimeError as exc:
        return str(exc)


def _run_rank(rank, world, out):
    import ctypes as C
    import twisterl_b200 as tw
    from twisterl_b200 import _lib, collector as twc, dist as twd
    L = _lib.load()
    engs = {p: tw.Engine(device=rank, precision=p, seed=SEED, rank=rank, world=world) for p in PRECISIONS}
    comms = {p: twd.Comm(engs[p]) for p in PRECISIONS}
    res = {"own": {}}

    # 1. PPO: every case, both forward kernels
    for i, (name, spec, E, twists) in enumerate(PPO_CASES):
        for j, prec in enumerate(PRECISIONS):
            eng = engs[prec]
            pol = _policy(spec, twists)
            col = tw.collector.PPOCollector(E, GAMMA, LAM, 1, engine=eng)
            eng.set_collect_id(_cid(i, j))
            own = col.collect_device(_env(spec, twists), pol)
            c = comms[prec].gather_collected(0)
            if rank == 0:
                d = col.to_host(c)
                _save(out / f"ppo-{name}-{prec}.npz", _ppo_arrays(d), d.stats)
            else:                                   # the other ranks keep their own result
                res["own"][f"{name}-{prec}"] = [int(c.num_episodes), int(c.n_records) == int(own.n_records), c.obs == own.obs]
            pol.release()

    # 2. AZ (lock-step MCTS on every rank: the persistent kernel is chosen by batch size)
    for j, prec in enumerate(PRECISIONS):
        eng = engs[prec]
        pol = _policy(AZ_ENV, False)
        col = tw.collector.AZCollector(AZ_EPISODES, AZ_SIMS, 1.41, 1, 1, engine=eng)
        eng.set_collect_id(_cid(len(PPO_CASES), j))
        col.collect_device(_env(AZ_ENV), pol)
        c = comms[prec].gather_collected(0)
        if rank == 0:
            d = col.to_host(c)
            _save(out / f"az-{prec}.npz", _az_arrays(d), d.stats)
        pol.release()

    # 3. refusals: the same error on every rank, nobody left waiting
    eng, comm = engs["f16f8c"], comms["f16f8c"]
    spec = ("puzzle", 4, 4, 8, 2, 256)
    pol = _policy(spec, False)
    env = _env(spec)
    errs = {}
    tw.collector.PPOCollector(ERR_EPISODES + rank, GAMMA, LAM, 1, engine=eng).collect_device(env, pol)
    errs["unequal_episodes"] = _gather_error(comm)
    if rank == 1:                               # pipelined host collect of two sub-batches: no device-resident result
        os.environ["TWISTERL_B200_E2E_PARTS"] = f"{ERR_EPISODES // 2},{ERR_EPISODES // 2}"
        s = tw.env.spec_from_env(env)
        cap = int(L.twr_max_records(C.byref(s), ERR_EPISODES))
        hb, _arr, _ = twc._host_buffers(cap, 16, 4, ERR_EPISODES, pinned=False)
        o = _lib.Collected()
        _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(s), pol.device_handle(eng), None, ERR_EPISODES, GAMMA, LAM,
                                          C.byref(hb), C.byref(o)))
        del os.environ["TWISTERL_B200_E2E_PARTS"]
    else:
        tw.collector.PPOCollector(ERR_EPISODES, GAMMA, LAM, 1, engine=eng).collect_device(env, pol)
    errs["pipelined_host_collect"] = _gather_error(comm)
    tw.collector.PPOCollector(ERR_EPISODES, GAMMA, LAM, 1, engine=eng).collect_device(env, pol)
    errs["root_out_of_range"] = _gather_error(comm, root=world)
    errs["then_valid"] = _gather_error(comm)
    errs["root_holds_merged"] = _gather_error(comm)
    res["errors"] = errs
    pol.release()

    # 4. ShardedCollector: two iterations, difficulty changed in between; every rank starts from different weights and
    # collect id, and root evaluates on the same engine before each iteration (which advances only root's own id)
    pol = _policy(("puzzle", 3, 3), False, seed=300 + rank)
    env = _env(("puzzle", 3, 3, 1, 2, 256))
    eng.set_collect_id(rank * 1000)
    sc = twd.ShardedCollector(tw.collector.PPOCollector(world * SHARD_EPISODES, GAMMA, LAM, 1), comm,
                              collect_id=SHARD_CID if rank == 0 else 0)
    local = []
    collect_device = sc.local.collect_device

    def recording(env_, pol_):
        c = collect_device(env_, pol_)
        local.append([int(env_.difficulty), int(c.n_records)])
        return c
    sc.local.collect_device = recording
    if rank == 0:
        env.difficulty = SHARD_DIFFICULTIES[0]
        _evaluate(eng, env, pol)
        d = sc.collect(env, pol)
        _save(out / "sharded-1.npz", _ppo_arrays(d), d.stats)
        env.difficulty = SHARD_DIFFICULTIES[1]
        _evaluate(eng, env, pol)
        t = sc.collect_torch(env, pol, dense_obs=False)
        res["sharded_torch"] = [t["stats"]["records"], int(t["obs"].shape[0]), t["stats"]["episodes"]]
        _save(out / "sharded-2.npz", _torch_arrays(t), t["stats"])
        sc.close()
    else:
        res["served"] = sc.serve(env, pol)
    res["sharded_local"] = local
    pol.release()

    # 5. accelerate(algorithm, comm): a trainer's collect on root goes through the sharded collector (PPO: collect_torch,
    # AZ: collect), with an evaluate on root's engine before each collect
    for kind, spec, total in (("ppo", ("puzzle", 3, 3, 3, 2, 256), world * SHARD_EPISODES), ("az", AZ_ENV, world * AZ_EPISODES)):
        pol = _policy(spec, False)
        env = _env(spec)
        col = (tw.collector.PPOCollector(total, GAMMA, LAM, 1) if kind == "ppo"
               else tw.collector.AZCollector(total, AZ_SIMS, 1.41, 1, 1))
        if rank == 0:
            algo = SimpleNamespace(collector=col, env=env, rs_pol=pol, policy=None, config={"training": {}})
            tw.accelerate(algo, comm)
            got = []
            for _ in range(2):
                _evaluate(eng, env, pol)
                data, _secs = algo.collect()
                got.append(data["stats"] if kind == "ppo" else data.stats)
            algo.sharded_collector.close()
            res[f"accelerate_{kind}"] = got
        else:
            res[f"accelerate_{kind}_served"] = twd.ShardedCollector(col, comm).serve(env, pol)
        pol.release()

    for c in comms.values():
        c.close()
    for e in engs.values():
        e.close()
    return res


def _child(rank, world, port, outdir):
    out = Path(outdir)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      TWISTERL_B200_MCTS_LOCKSTEP="1", TWISTERL_B200_MCTS_DEBUG="1")
    fd = os.open(out / f"stderr{rank}.txt", os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    os.dup2(fd, 2)                              # the library's [mcts] lines and any traceback
    try:
        res = _run_rank(rank, world, out)
    except BaseException:
        traceback.print_exc()
        raise
    (out / f"rank{rank}.json").write_text(json.dumps(res))


# ------------------------------------------------------------------------------------------------ parent ---
def _worlds():
    try:
        import torch
        n = torch.cuda.device_count()
    except Exception:
        n = 0
    return [2] + ([min(n, 8)] if min(n, 8) > 2 else [])


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture(scope="module", params=_worlds(), ids=lambda w: f"W{w}")
def run(request, tmp_path_factory):
    import torch
    import torch.multiprocessing as mp
    from twisterl_b200 import _lib
    world = request.param
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    if _lib.load().twr_comm_version() == 0:
        pytest.skip("NCCL is not available")
    out = tmp_path_factory.mktemp(f"gather_w{world}")
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_child, args=(r, world, port, str(out))) for r in range(world)]
    for p in procs:
        p.start()
    deadline = time.time() + JOIN_TIMEOUT
    try:                                        # until all are done, one has failed (its peers would wait in NCCL), or time is up
        while time.time() < deadline and any(p.is_alive() for p in procs) and not any(p.exitcode for p in procs):
            time.sleep(1.0)
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=30)
            if p.is_alive():
                p.kill()
                p.join()
    logs = {r: (out / f"stderr{r}.txt").read_text()[-4000:] if (out / f"stderr{r}.txt").exists() else "" for r in range(world)}
    bad = [r for r, p in enumerate(procs) if p.exitcode != 0]
    assert not bad, "\n".join(f"rank {r} exit {procs[r].exitcode}:\n{logs[r]}" for r in bad)
    ranks = [json.loads((out / f"rank{r}.json").read_text()) for r in range(world)]
    return world, out, ranks, logs


_ref_engines = {}


def _ref_engine(prec):
    import twisterl_b200 as tw
    if prec not in _ref_engines:
        _ref_engines[prec] = tw.Engine(device=0, precision=prec, seed=SEED)
    return _ref_engines[prec]


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("case", PPO_CASES, ids=[c[0] for c in PPO_CASES])
def test_ppo_gather_equals_one_collect(run, case, prec):
    import twisterl_b200 as tw
    world, out, ranks, _ = run
    i, j = PPO_CASES.index(case), PRECISIONS.index(prec)
    name, spec, E, twists = case
    eng = _ref_engine(prec)
    pol = _policy(spec, twists)
    eng.set_collect_id(_cid(i, j))
    d = tw.collector.PPOCollector(world * E, GAMMA, LAM, 1, engine=eng).collect(_env(spec, twists), pol)
    pol.release()
    assert d.stats["episodes"] == world * E
    _assert_same(out / f"ppo-{name}-{prec}.npz", _ppo_arrays(d), d.stats)
    if twists:
        assert set(np.unique(d.perms_array)) == {0, 1}
    for r in range(1, world):                      # the other ranks' `out` is their own result, unchanged
        assert ranks[r]["own"][f"{name}-{prec}"] == [E, True, True]


@pytest.mark.parametrize("prec", PRECISIONS)
def test_az_gather_equals_one_collect(run, prec, monkeypatch, capfd):
    import twisterl_b200 as tw
    world, out, _, logs = run
    monkeypatch.setenv("TWISTERL_B200_MCTS_LOCKSTEP", "1")
    monkeypatch.setenv("TWISTERL_B200_MCTS_DEBUG", "1")
    eng = _ref_engine(prec)
    pol = _policy(AZ_ENV, False)
    eng.set_collect_id(_cid(len(PPO_CASES), PRECISIONS.index(prec)))
    d = tw.collector.AZCollector(world * AZ_EPISODES, AZ_SIMS, 1.41, 1, 1, engine=eng).collect(_env(AZ_ENV), pol)
    pol.release()
    _assert_same(out / f"az-{prec}.npz", _az_arrays(d), d.stats)
    # the lock-step search ran everywhere: with TWISTERL_B200_MCTS_DEBUG the persistent kernel announces itself
    assert "[mcts] persistent" not in capfd.readouterr().err
    assert not any("[mcts] persistent" in log for log in logs.values())


def test_refusals_are_uniform(run):
    world, _, ranks, _ = run
    for key, code_text in (("unequal_episodes", "num_episodes of rank"), ("pipelined_host_collect", "rank 1 holds no device-resident"),
                           ("root_out_of_range", "root out of range"), ("root_holds_merged", "rank 0 holds no device-resident")):
        msgs = [r["errors"][key] for r in ranks]
        assert all(m is not None and code_text in m for m in msgs), (key, msgs)
        assert len(set(msgs)) == 1, (key, msgs)
    assert all(r["errors"]["then_valid"] is None for r in ranks)


def test_sharded_collector(run):
    import twisterl_b200 as tw
    world, out, ranks, _ = run
    assert all(r["served"] == len(SHARD_DIFFICULTIES) for r in ranks[1:])
    for r in ranks:                                 # every rank collected at the difficulty root sent
        assert [x[0] for x in r["sharded_local"]] == list(SHARD_DIFFICULTIES)
    totals = [sum(r["sharded_local"][k][1] for r in ranks) for k in range(len(SHARD_DIFFICULTIES))]
    assert ranks[0]["sharded_torch"] == [totals[1], totals[1], world * SHARD_EPISODES]
    # each iteration is one collect of all episodes with root's weights (the others started from their own) at root's
    # counter's collect id, whatever root evaluated in between
    eng = _ref_engine("f16f8c")
    pol = _policy(("puzzle", 3, 3), False, seed=300)
    for k, difficulty in enumerate(SHARD_DIFFICULTIES):
        eng.set_collect_id(SHARD_CID + k)
        d = tw.collector.PPOCollector(world * SHARD_EPISODES, GAMMA, LAM, 1, engine=eng).collect(
            _env(("puzzle", 3, 3, difficulty, 2, 256)), pol)
        assert d.stats["records"] == totals[k]
        _assert_same(out / f"sharded-{k + 1}.npz", _ppo_arrays(d) | ({} if k == 0 else {"ep_len": None}), d.stats)
    pol.release()
    for kind, per_rank in (("ppo", SHARD_EPISODES), ("az", AZ_EPISODES)):
        assert all(r[f"accelerate_{kind}_served"] == 2 for r in ranks[1:])
        assert [st["episodes"] for st in ranks[0][f"accelerate_{kind}"]] == [world * per_rank] * 2


@pytest.mark.parametrize("prec", PRECISIONS)
def test_shards_in_merge_order_equal_one_collect(prec):
    """The layout twr_gather_collected relies on, on one GPU: W engines configured as ranks 0..W-1 of W collect E
    episodes each; their results placed head_{W-1}, tail_0, head_0, ..., tail_{W-1} (head_r = the first ep_len[E-1]
    records of rank r) and their ep_len concatenated equal one engine's collect of W*E episodes, byte for byte."""
    import twisterl_b200 as tw
    W, E, cid = 3, 300, 77
    name, spec, _, twists = PPO_CASES[1]
    ref_eng = tw.Engine(device=0, precision=prec, seed=SEED)
    pol = _policy(spec, twists)
    ref_eng.set_collect_id(cid)
    ref = tw.collector.PPOCollector(W * E, GAMMA, LAM, 1, engine=ref_eng).collect(_env(spec, twists), pol)
    pol.release()
    ref_eng.close()
    shards = []
    for r in range(W):
        eng = tw.Engine(device=0, precision=prec, seed=SEED, rank=r, world=W)
        pol = _policy(spec, twists)
        eng.set_collect_id(cid)
        d = tw.collector.PPOCollector(E, GAMMA, LAM, 1, engine=eng).collect(_env(spec, twists), pol)
        shards.append(_ppo_arrays(d))
        pol.release()
        eng.close()
    heads = [int(s["ep_len"][E - 1]) for s in shards]
    for k, a in _ppo_arrays(ref).items():
        if k == "ep_len":
            got = np.concatenate([s[k] for s in shards])
        else:
            pieces = [shards[W - 1][k][:heads[W - 1]]]
            for r in range(W):
                pieces.append(shards[r][k][heads[r]:])
                if r < W - 1:
                    pieces.append(shards[r][k][:heads[r]])
            got = np.concatenate(pieces)
        assert got.dtype == a.dtype and got.shape == a.shape, k
        assert np.array_equal(got.view(np.uint8), np.ascontiguousarray(a).view(np.uint8)), k


@pytest.mark.parametrize("kind", ["ppo", "az"])
def test_accelerate_with_comm_keeps_collect_ids_across_evaluations(kind, monkeypatch):
    """accelerate(algorithm, comm) routes the trainer's collect through the sharded collector (PPO: collect_torch, AZ:
    collect).  An evaluate on the same engine before each collect, as a curriculum check does, advances the engine's
    own collect id; the sharded collects still run at the collector's ids (500, 501), i.e. equal the plain collects pinned
    there.  One GPU: a communicator of world 1."""
    import twisterl_b200 as tw
    from twisterl_b200 import dist as twd
    monkeypatch.setenv("TWISTERL_B200_MCTS_LOCKSTEP", "1")
    spec = ("puzzle", 3, 3, 3, 2, 256) if kind == "ppo" else AZ_ENV

    def collector():
        return (tw.collector.PPOCollector(400, GAMMA, LAM, 1) if kind == "ppo"
                else tw.collector.AZCollector(AZ_EPISODES, AZ_SIMS, 1.41, 1, 1))
    eng = tw.Engine(device=0, precision="f16f8c", seed=SEED)
    pol, env = _policy(spec, False), _env(spec)
    algo = SimpleNamespace(collector=collector(), env=env, rs_pol=pol, policy=None, config={"training": {}})
    tw.accelerate(algo, twd.Comm(eng, rank=0, world=1))
    algo.sharded_collector.collect_id = 500
    got = []
    for _ in range(2):
        _evaluate(eng, env, pol)
        data, _secs = algo.collect()
        got.append(_torch_arrays(data) if kind == "ppo" else _az_arrays(data))
    algo.sharded_collector.close()
    pol.release()
    eng.close()
    ref_eng = tw.Engine(device=0, precision="f16f8c", seed=SEED)
    pol = _policy(spec, False)
    col = collector()
    col._engine = ref_eng
    for k in range(2):
        ref_eng.set_collect_id(500 + k)
        d = col.collect(env, pol)
        ref = _ppo_arrays(d) if kind == "ppo" else _az_arrays(d)
        for name, a in got[k].items():
            assert np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(ref[name]).view(np.uint8)), (k, name)
    pol.release()
    ref_eng.close()


def test_world_one_returns_the_local_result():
    """world == 1: no communicator, the local result comes back unchanged; nothing to gather is refused."""
    import ctypes as C
    import twisterl_b200 as tw
    from twisterl_b200 import _lib, dist as twd
    eng = tw.Engine(device=0, precision="f16f8c", seed=SEED)
    comm = twd.Comm(eng, rank=0, world=1)
    with pytest.raises(RuntimeError, match="no device-resident collect result"):
        comm.gather_collected(0)
    spec = ("puzzle", 3, 3, 6, 2, 256)
    pol = _policy(spec, False)
    col = tw.collector.PPOCollector(500, GAMMA, LAM, 1, engine=eng)
    eng.set_collect_id(5)
    ref = col.collect(_env(spec), pol)
    eng.set_collect_id(5)
    own = col.collect_device(_env(spec), pol)
    c = comm.gather_collected(0)
    for f, _ in _lib.Collected._fields_:
        assert getattr(c, f) == getattr(own, f), f
    with pytest.raises(RuntimeError, match="root out of range"):
        comm.gather_collected(1)
    again = col.to_host(c)
    for k, a in _ppo_arrays(ref).items():
        assert np.array_equal(a, _ppo_arrays(again)[k]), k
    assert _lib.load().twr_gather_collected(eng._h, 0, C.byref(_lib.Collected())) == 0   # a second gather: still local
    pol.release()
    eng.close()
