"""GridWorld boards of 33..64 cells (6x6, 7x7, 8x8, 4x16) on the device.  The env state is the same 16 bytes at every
size; what changes is the policy's N*N-row table (1 296 to 4 096 rows).  GridWorld forwards run it as the compact table
of the 4N reachable rows: the pair kernel on tensor-core engines, the fp32 SIMT kernel's compact mode on fp32 engines.
Forwards that cannot use the compact table (rows given directly, twists that leave the reachable rows) run the generic
kernel.  Held to the oracle: env transitions bit-exact, fp32 forwards at 1e-5, tensor-core forwards to the CPU model of
the pair kernel's operand rounding (tc_emul), collects replayed record by record, searches under the near-tie rule on the
path the persistent kernel's footprint allows, the multi-GPU gather layout byte for byte."""
import ctypes as C
import re

import numpy as np
import pytest

from suite_loader import suite_precision

import tc_emul as te
from helpers import gridworld_transpose_twists, synth_state_dict
from oracle import orc

pytestmark = pytest.mark.gpu

PRECISION = suite_precision(globals())
TC = PRECISION != "fp32"
TOL = {"fp32": 1e-5, "f16x2": 1e-4}.get(PRECISION, 1e-3)          # collect replay bar of the engine's forward
EMUL_BAR = 2.5e-7                                                    # tensor-core forward against tc_emul (|d| / S)
NEAR_TIE = {"fp32": 2e-4, "f16x2": 2e-3, "f16x2w16": 2e-2, "f16f8c": 2e-2}[PRECISION]
SEED = 0x64_6464_6464
BOARDS = [(6, 6), (7, 7), (8, 8), (4, 16)]
DEBUG_LINE = re.compile(r"\[mcts\] persistent: (\d+) trees")
PM_CS, PM_TPC, SMEM_LIMIT = 8, 40, 227 * 1024


@pytest.fixture(scope="module")
def eng():
    import twisterl_b200 as tw
    e = tw.Engine(device=0, precision=PRECISION, seed=SEED)
    yield e
    e.close()


def _sd(w, h, E, H, seed):
    return synth_state_dict(seed, (w * h) ** 2, E, H, 4)


def _twists(w, h, twists):
    return gridworld_transpose_twists(w) if twists and w == h else ((), ())


def _policies(w, h, twists, E=256, H=256, seed=64, sd=None):
    from parity import make_policies
    N = w * h
    return make_policies(sd if sd is not None else _sd(w, h, E, H, seed), N * N, *_twists(w, h, twists))


def _batch(eng, w, h, n, base=11, cid=3, difficulty=None):
    from twisterl_b200.env import EnvBatch
    b = EnvBatch(orc.gridworld_spec(w, h, 100, difficulty or (w + h) // 2), n, eng)
    b.reset(env_id_base=base, collect_id=cid)
    return b


def _check_forward(w_, logits, values, obs, perm=None, twists=((), ()), opol=None, generic=False):
    """fp32 (and every forward that runs an fp32 kernel): 1e-5 of the oracle.  Tensor-core GridWorld forwards: the CPU
    model of the pair kernel."""
    if TC and not generic:
        ml, mv, _ = te.engine_forward(w_, PRECISION, obs, perm, *twists)
        sl, sv = te.magnitude(w_, obs, perm, *twists)
        m = max(te.rel_to_s(logits, ml, sl), te.rel_to_s(values, mv, sv))
        assert m <= EMUL_BAR, m
        return
    for i in range(len(obs)):
        rl, rv = opol.raw_predict(list(map(int, obs[i])), -1 if perm is None else int(perm[i]))
        assert te.rel_err(logits[i], rl) <= 1e-5 and abs(values[i] - rv) <= 1e-5 * max(1.0, abs(rv)), i


# ------------------------------------------------------------------------------------------------------- env ---
@pytest.mark.parametrize("w,h", BOARDS + [(1, 64), (6, 10)], ids=lambda v: str(v))
def test_env_reset_and_forced_steps_bit_exact(eng, w, h):
    """reset at several difficulties, then 50 random (often off-board) forced actions: state, observation, masks,
    reward, final flag, success and steps_left equal the oracle's at every step."""
    from twisterl_b200.env import EnvBatch
    n = 97
    for difficulty in (1, 4, w + h):
        ospec = orc.gridworld_spec(w, h, 30, difficulty)
        rng = np.random.default_rng(w * 100 + h + difficulty)
        b = EnvBatch(ospec, n, eng)
        b.reset(env_id_base=500, collect_id=2)
        envs = [orc.Env(ospec) for _ in range(n)]
        for i, e in enumerate(envs):
            e.reset(seed=eng.seed, env_id=500 + i, collect_id=2)

        def compare(tag):
            st, ob, mk = b.get_state(), b.observe(), b.masks()
            rw, fi, su, dp = b.reward(), b.is_final(), b.success(), b.depth()
            for i, e in enumerate(envs):
                assert st[i].tolist() == e.get_state(), (tag, i)
                assert ob[i].tolist() == e.observe(), (tag, i)
                assert mk[i].tolist() == e.masks(), (tag, i)
                assert rw[i] == np.float32(e.reward()), (tag, i)
                assert bool(fi[i]) == e.is_final() and bool(su[i]) == e.success(), (tag, i)
                assert dp[i] == e.depth, (tag, i)

        compare("reset")
        for t in range(50):
            acts = rng.integers(0, 4, size=n)
            b.step(acts)
            for e, a in zip(envs, acts):
                e.step(int(a))
            compare(t)


def test_env_set_state_round_trips_at_8x8(eng):
    from twisterl_b200.env import EnvBatch
    src = _batch(eng, 8, 8, 64)
    st = src.get_state()
    b = EnvBatch(orc.gridworld_spec(8, 8, 100, 7), 64, eng)
    b.set_state(st)
    assert np.array_equal(b.get_state(), st) and np.array_equal(b.observe(), src.observe())
    bad = st.copy(); bad[3, 63] = 4
    with pytest.raises(RuntimeError, match="GridWorld cell values"):
        b.set_state(bad)


# --------------------------------------------------------------------------------------------------- forward ---
@pytest.mark.parametrize("w,h,twists,E,H", [(6, 6, False, 256, 256), (6, 6, True, 512, 128), (7, 7, False, 256, 128),
                                            (7, 7, True, 256, 256), (8, 8, False, 512, 256), (8, 8, True, 256, 128),
                                            (4, 16, False, 256, 256)])
def test_forward_on_the_compact_table(eng, w, h, twists, E, H):
    from twisterl_b200.nn import forward_batch, forward_obs
    sd = _sd(w, h, E, H, E + H + w)
    pol, opol = _policies(w, h, twists, sd=sd)
    tws = _twists(w, h, twists)
    b = _batch(eng, w, h, 300)
    perm = np.random.default_rng(3).integers(0, 2, size=b.n).astype(np.int32) if tws[0] else None
    logits, values = forward_batch(eng, pol, b, perm_idx=perm)
    obs = b.observe().astype(np.int64)
    _check_forward(te.Weights(sd), logits, values, obs, perm, tws, opol)
    if not TC and w * h == 36:
        # a 6x6 table also fits the fp32 kernel whole, which is what twr_policy_forward_obs runs on the same rows: the
        # compact table sums the same rows in the same order, bit for bit
        rl, rv = forward_obs(eng, pol, obs, perm_idx=perm)
        assert np.array_equal(logits, rl) and np.array_equal(values, rv)
    pol.release()


def test_forward_obs_and_twists_off_the_compact_rows_run_the_generic_kernel(eng):
    """twr_policy_forward_obs on an 8x8 policy (64 indices per row, arbitrary rows included), and an env forward under a
    twist set that sends reachable rows to unreachable ones: the generic fp32 kernel, within 1e-5 of the oracle."""
    from twisterl_b200.nn import forward_batch, forward_obs
    sd = _sd(8, 8, 256, 256, 7)
    w_ = te.Weights(sd)
    pol, opol = _policies(8, 8, False, sd=sd)
    b = _batch(eng, 8, 8, 128)
    obs = b.observe().astype(np.int64)
    rng = np.random.default_rng(5)
    arb = rng.integers(0, 4096, size=(64, 64))
    for rows in (obs, arb, obs[:, :40]):
        l, v = forward_obs(eng, pol, rows)
        _check_forward(w_, l, v, rows, opol=opol, generic=True)
    with pytest.raises(RuntimeError, match="1..64"):
        forward_obs(eng, pol, np.zeros((2, 65), np.int64))
    pol.release()
    # a twist that swaps value 0 and value 5 of every cell: row i*64 + 0 leaves the reachable rows
    ob, ac = gridworld_transpose_twists(8)
    N = 64
    tw2 = [(i // N) * N + {0: 5, 5: 0}.get(i % N, i % N) for i in range(N * N)]
    twists = ([ob[0], tw2], [ac[0], [0, 1, 2, 3]])
    from parity import make_policies
    pol, opol = make_policies(sd, N * N, *twists)
    perm = rng.integers(0, 2, size=b.n).astype(np.int32)
    l, v = forward_batch(eng, pol, b, perm_idx=perm)
    _check_forward(w_, l, v, obs, perm, twists, opol, generic=True)
    pol.release()


# --------------------------------------------------------------------------------------------------- collect ---
@pytest.mark.parametrize("w,h,episodes,twists", [(6, 6, 400, False), (6, 6, 300, True), (8, 8, 400, False),
                                                 (8, 8, 300, True), (4, 16, 300, False)])
def test_collect_replays_through_oracle(eng, w, h, episodes, twists):
    import twisterl_b200 as tw
    from parity import check_collect_against_oracle
    pol, opol = _policies(w, h, twists, 256, 256, seed=w * h)
    ospec = orc.gridworld_spec(w, h, 64, w + h)
    env = tw.env.GridWorld(w, h, 64, w + h)
    col = tw.collector.PPOCollector(episodes, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(13)
    data = col.collect(env, pol)
    rep = check_collect_against_oracle(data, ospec, opol, seed=eng.seed, collect_id=13, gamma=0.995, lam=0.995, tol=TOL)
    assert rep["records"] == len(data.values_array) and data.stats["episodes"] == episodes
    assert data.obs_array.shape[1] == w * h
    eng.set_collect_id(13)
    t = col.collect_torch(env, pol, dense_obs=False)
    R = len(data.values_array)
    for k, a in (("values", data.values_array), ("logits", data.logits_array), ("rewards", data.rewards_array)):
        assert np.array_equal(t[k].cpu().numpy().reshape(a.shape), a), k
    assert np.array_equal(t["obs"].cpu().numpy().reshape(R, -1).astype(np.int64), data.obs_array.astype(np.int64))
    if w * h == 64:                                  # the dense one-hot the reference trainer consumes: R x 4096 floats
        eng.set_collect_id(13)
        dense = col.collect_torch(env, pol, dense_obs=True)["obs"].cpu().numpy().reshape(R, -1)
        assert dense.shape == (R, 4096) and (dense.sum(axis=1) == 64).all()
        rows = data.obs_array.astype(np.int64)
        assert (dense[np.arange(R)[:, None], rows] == 1).all()
    pol.release()


def test_collect_host_pipelined_and_fused_gae_match_plain(eng, monkeypatch):
    """twr_ppo_collect_host on 8x8 (sub-batches; u16 observation indices, obs_size 4096) holds exactly what the plain
    collect produces, and the collect's fused GAE equals twr_gae over its records."""
    import twisterl_b200 as tw
    from twisterl_b200 import _lib, collector as twc
    pol, _ = _policies(8, 8, True, 256, 128, seed=3)
    env = tw.env.GridWorld(8, 8, 64, 10)
    E = 1000
    col = tw.collector.PPOCollector(E, 0.97, 0.9, 32, engine=eng)
    eng.set_collect_id(21)
    ref = col.collect(env, pol)
    L = _lib.load()
    spec = tw.env.spec_from_env(env)
    cap = int(L.twr_max_records(C.byref(spec), E))
    for parts in ("334,333,333", "1000"):
        monkeypatch.setenv("TWISTERL_B200_E2E_PARTS", parts)
        hb, arr, _ = twc._host_buffers(cap, 64, 4, E, pinned=True)
        out = _lib.Collected()
        eng.set_collect_id(21)
        _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), pol.device_handle(eng), None, E, 0.97, 0.9,
                                          C.byref(hb), C.byref(out)))
        R = int(out.n_records)
        assert R == len(ref.values_array) and int(out.successes) == ref.stats["successes"]
        assert np.array_equal(arr["ep_len"], ref.ep_len)
        for k, a in (("obs", ref.obs_array), ("actions", ref.actions_array), ("logits", ref.logits_array),
                     ("values", ref.values_array), ("rewards", ref.rewards_array), ("perms", ref.perms_array),
                     ("advs", ref.additional_array("advs")), ("rets", ref.additional_array("rets"))):
            assert np.array_equal(arr[k][:R], a), k
    r, v = np.ascontiguousarray(ref.rewards_array, np.float32), np.ascontiguousarray(ref.values_array, np.float32)
    R = len(v)
    off = np.concatenate([[0], np.cumsum(ref.ep_len.astype(np.int64)[orc.merge_order(E)])]).astype(np.int64)
    assert off[-1] == R
    adv = np.zeros(R, np.float32); ret = np.zeros(R, np.float32)
    _lib.check(L.twr_gae(eng._h, _lib.ptr(r), _lib.ptr(v), _lib.ptr(off), E, 0.97, 0.9, _lib.ptr(adv), _lib.ptr(ret)))
    assert np.array_equal(adv, ref.additional_array("advs")) and np.array_equal(ret, ref.additional_array("rets"))
    assert set(np.unique(ref.perms_array)) == {0, 1}
    pol.release()


def test_gather_layout_on_one_gpu_8x8(eng):
    """three engines as ranks 0..2 collect E episodes each; their records placed head_2, tail_0, head_0, tail_1, head_1,
    tail_2 and their ep_len concatenated equal one engine's collect of 3E episodes, byte for byte."""
    import twisterl_b200 as tw
    W, E, cid = 3, 300, 77

    def arrays(d):
        return dict(obs=d.obs_array, logits=d.logits_array, values=d.values_array, rewards=d.rewards_array,
                    actions=d.actions_array, perms=d.perms_array, advs=d.additional_array("advs"),
                    rets=d.additional_array("rets"), ep_len=d.ep_len)

    def run(n, **kw):
        e = tw.Engine(device=0, precision=PRECISION, seed=SEED, **kw)
        pol, _ = _policies(8, 8, False, 256, 256, seed=8)
        e.set_collect_id(cid)
        out = arrays(tw.collector.PPOCollector(n, 0.99, 0.95, 1, engine=e).collect(tw.env.GridWorld(8, 8, 64, 10), pol))
        pol.release()
        e.close()
        return out

    ref = run(W * E)
    shards = [run(E, rank=r, world=W) for r in range(W)]
    heads = [int(s["ep_len"][E - 1]) for s in shards]
    for k, a in ref.items():
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


# ---------------------------------------------------------------------------------------------------- search ---
def pm_footprint(E, H, obs):
    """Shared memory of k_mcts_persistent: a copy of pm_layout (twr_mcts.cu), as in test_gpu_mcts_shapes.py."""
    EC, per = E // PM_CS, PM_TPC // PM_CS
    floats = EC * H + obs * EC + PM_TPC * EC + H + EC + 5 * (H + 8) + per * PM_CS * H + per * H + per * 8
    return (4 * floats + 16 * PM_TPC + 4 * PM_TPC + 15) & ~15


@pytest.mark.parametrize("w,h,E,H,twists", [(6, 6, 128, 128, False), (6, 6, 128, 128, True), (8, 8, 256, 256, False),
                                            (7, 7, 256, 128, True)])
def test_mcts_on_the_path_the_footprint_allows(eng, capfd, monkeypatch, w, h, E, H, twists):
    """The persistent search keeps the full N*N-row table slice in shared memory: a small-E 6x6 policy fits, 7x7 and
    8x8 do not and run the lockstep kernels.  The path that ran is the one the footprint predicts; the search is held to
    the oracle under the near-tie rule."""
    from twisterl_b200 import _lib
    N = w * h
    persistent = pm_footprint(E, H, N * N) <= SMEM_LIMIT
    assert persistent == (N == 36)
    pol, opol = _policies(w, h, twists, E, H, seed=E + H + N)
    b = _batch(eng, w, h, 40, base=70, difficulty=5)
    states = b.get_state()
    monkeypatch.setenv("TWISTERL_B200_MCTS_DEBUG", "1")
    n, sims = b.n, 16
    probs = np.zeros((n, 4), np.float32); visits = np.zeros((n, 4), np.int32)
    trace = np.zeros((sims, n, 2), np.int32)
    capfd.readouterr()
    n0 = eng.launch_count()
    _lib.check(_lib.load().twr_debug_mcts_trace(eng._h, pol.device_handle(eng), b._h, sims, 1.41, 1, 700, 5, 1,
                                                _lib.ptr(probs), _lib.ptr(visits), _lib.ptr(trace)))
    launches = eng.launch_count() - n0
    assert bool(DEBUG_LINE.findall(capfd.readouterr().err)) == persistent
    if not persistent:
        assert launches > sims
    same = 0
    for i in range(n):
        env = orc.Env(orc.gridworld_spec(w, h, 100, 5)); env.set_state(states[i].tolist())
        op, ov = orc.mcts_probs(env, opol, sims, 1.41, 1, seed=eng.seed, collect_id=5, stream_id=700 + i, t=1)
        assert visits[i].sum() == ov.sum()
        if np.array_equal(visits[i], ov):
            same += 1
            assert np.allclose(probs[i], op, atol=1e-6 if not TC or persistent else 1e-3)
            continue
        _, _, leaf, child, margin = orc.mcts_trace(env, opol, sims, 1.41, 1, seed=eng.seed, collect_id=5, stream_id=700 + i, t=1)
        div = next((s for s in range(sims) if trace[s, i, 0] != leaf[s] or trace[s, i, 1] != child[s]), None)
        assert div is not None and margin[div] < NEAR_TIE, (i, div)
    assert same >= n // 2
    pol.release()


@pytest.mark.parametrize("det,searches,mcts", [(True, 1, 0), (False, 4, 0), (False, 1, 8)])
def test_evaluate_matches_oracle_7x7(eng, det, searches, mcts):
    import twisterl_b200 as tw
    from twisterl_b200 import _lib
    pol, opol = _policies(7, 7, False, 256, 128, seed=8)
    ospec = orc.gridworld_spec(7, 7, 30, 6)
    spec = tw.env.spec_from_env(tw.env.GridWorld(7, 7, 30, 6))
    n = 48 if mcts else 160
    s, r = C.c_float(), C.c_float()
    bs, bt = np.zeros(n, np.float32), np.zeros(n, np.float32)
    eng.set_collect_id(7)
    _lib.check(_lib.load().twr_evaluate_episodes(eng._h, C.byref(spec), pol.device_handle(eng), n, int(det), searches,
                                                 mcts, 1.41, 1, C.byref(s), C.byref(r), _lib.ptr(bs), _lib.ptr(bt)))
    obs_, obt, mm = orc.evaluate_margins(ospec, opol, n, det, searches, seed=eng.seed, collect_id=7, num_mcts_searches=mcts,
                                         c_puct=1.41, max_expand_depth=1)
    diff = [i for i in range(n) if bs[i] != obs_[i] or abs(float(bt[i]) - float(obt[i])) > 1e-5]
    for i in diff:
        assert mm[i] < NEAR_TIE, f"episode {i} differs with smallest margin {mm[i]}"
    assert len(diff) <= n // 4
    assert abs(s.value - float(bs.mean())) < 1e-6
    pol.release()


def test_solve_and_az_collect_on_8x8(eng):
    import twisterl_b200 as tw
    tw.configure(device=0, precision=PRECISION, seed=SEED)
    pol, _ = _policies(8, 8, False, 256, 256)
    g = tw.env.GridWorld(8, 8, 40, 6)
    g.reset()
    start = g.get_state()
    for det, mcts in ((True, 0), (False, 0), (False, 6)):
        g.set_state(start)
        (succ, rew), acts = tw.collector.solve(g, pol, det, 4, mcts, 1.41, 1)
        o = orc.Env(orc.gridworld_spec(8, 8, 40, 6)); o.set_state(start)
        for a in acts:
            o.step(a)
        assert len(acts) <= 40 and succ in (0.0, 1.0) and bool(succ) == o.success()
    pol.release()
    pol, _ = _policies(8, 8, False, 256, 256)
    col = tw.collector.AZCollector(64, 12, 1.41, 1, 1, engine=eng)
    eng.set_collect_id(9)
    d = col.collect(tw.env.GridWorld(8, 8, 24, 5), pol)
    R = len(d.obs_array)
    assert R == int(d.ep_len.sum()) and np.allclose(d.logits_array.sum(axis=1), 1.0, atol=1e-5)
    vals = d.obs_array.astype(np.int64) - np.arange(64) * 64
    assert ((vals >= 0) & (vals <= 3)).all() and ((vals == 1).sum(axis=1) == 1).all()
    pol.release()


# ------------------------------------------------------------------------------------------------ weight refresh ---
def test_update_from_torch_on_8x8(eng):
    """After update_from_torch(W1) (on tensor-core engines it repacks the compact operand image on the device), a policy
    created from W0 computes bit for bit what a policy created from W1 computes: forwards and a PPO collect."""
    import torch

    import twisterl_b200 as tw
    from twisterl_b200.nn import forward_batch
    sd0, sd1 = _sd(8, 8, 256, 128, 91), _sd(8, 8, 256, 128, 92)
    pol, _ = _policies(8, 8, True, sd=sd0)
    fresh, _ = _policies(8, 8, True, sd=sd1)
    b = _batch(eng, 8, 8, 200)
    forward_batch(eng, pol, b)
    m = torch.nn.Module()
    m.embeddings = torch.nn.Linear(4096, 256)
    m.common = torch.nn.Sequential(torch.nn.Linear(256, 128), torch.nn.ReLU())
    m.action = torch.nn.Sequential(torch.nn.Linear(128, 4))
    m.value = torch.nn.Sequential(torch.nn.Linear(128, 1))
    m.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd1.items()})
    pol.update_from_torch(m.to(torch.device("cuda", eng.device)), eng)
    for x, y in zip(forward_batch(eng, pol, b), forward_batch(eng, fresh, b)):
        assert np.array_equal(x, y)
    env = tw.env.GridWorld(8, 8, 64, 10)
    outs = []
    for p in (pol, fresh):
        eng.set_collect_id(61)
        d = tw.collector.PPOCollector(256, 0.995, 0.995, 1, engine=eng).collect(env, p)
        outs.append([d.obs_array, d.logits_array, d.values_array, d.actions_array, d.perms_array, np.asarray(d.ep_len)])
    for x, y in zip(*outs):
        assert np.array_equal(x, y)
    pol.release(); fresh.release()
