"""Puzzle boards of 17..25 cells (the 24-puzzle, 5x5, among them) on the device.  Their state is the 5-bit encoding of
twr_common.cuh; their N*N >= 289-row tables run the fp32 SIMT forward on every engine (the pair kernel takes a table
above 256 rows only as GridWorld's compact image).  Held to the oracle: env transitions bit-exact, logits and values at
1e-5, collects replayed record by record, searches under the near-tie rule, the multi-GPU gather layout byte for byte."""
import ctypes as C
import re

import numpy as np
import pytest

from suite_loader import suite_precision

from helpers import scramble_states, synth_state_dict, transpose_twists
from oracle import orc

pytestmark = pytest.mark.gpu

PRECISION = suite_precision(globals())
TOL = 1e-5                                  # wide boards run the fp32 kernel on every engine
NEAR_TIE = 2e-4
SEED = 0x24_2424_2424
BOARDS = [(3, 6), (6, 3), (4, 5), (5, 4), (4, 6), (5, 5), (1, 25)]
DEBUG_LINE = re.compile(r"\[mcts\] persistent: (\d+) trees")


@pytest.fixture(scope="module")
def eng():
    import twisterl_b200 as tw
    e = tw.Engine(device=0, precision=PRECISION, seed=SEED)
    yield e
    e.close()


def _spec(o):
    """device spec of an oracle spec: a Puzzle above 16 cells is env kind TWR_ENV_PUZZLE_WIDE"""
    from twisterl_b200 import _lib
    kind = _lib.ENV_PUZZLE_WIDE if o.kind == _lib.ENV_PUZZLE and o.width * o.height > 16 else o.kind
    return _lib.EnvSpec(kind, o.width, o.height, o.difficulty, o.depth_slope, o.max_depth)


def _close(a, ref, tol):
    return float((np.abs(a - ref) / np.maximum(1.0, np.abs(ref))).max(initial=0.0)) <= tol


def _policies(w, h, twists, E=256, H=256, seed=25):
    from parity import make_policies
    N = w * h
    return make_policies(synth_state_dict(seed, N * N, E, H, 4), N * N, *(transpose_twists(w) if twists else ((), ())))


# ------------------------------------------------------------------------------------------------------- env ---
@pytest.mark.parametrize("w,h", BOARDS, ids=lambda v: str(v))
def test_env_reset_and_forced_steps_bit_exact(eng, w, h):
    """reset at several difficulties, then 40 random (often illegal) forced actions: state, observation, masks, reward,
    final flag, success and depth equal the oracle's at every compared step."""
    from twisterl_b200.env import EnvBatch
    n = 97
    for difficulty in (0, 3, 64, 300):
        ospec = orc.puzzle_spec(w, h, difficulty, 1, 256)
        rng = np.random.default_rng(w * 100 + h + difficulty)
        b = EnvBatch(_spec(ospec), n, eng)
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
        for t in range(40):
            acts = rng.integers(0, 4, size=n)
            b.step(acts)
            for e, a in zip(envs, acts):
                e.step(int(a))
            if t % 8 == 7 or t < 2:
                compare(t)


@pytest.mark.parametrize("w,h", [(5, 5), (4, 6), (1, 25), (3, 6)], ids=lambda v: str(v))
def test_env_set_state_and_position_round_trips(eng, w, h):
    import twisterl_b200 as tw
    from twisterl_b200.env import EnvBatch
    N = w * h
    states = scramble_states(np.random.default_rng(N), 64, w, h, 80).astype(np.int64)
    states[0] = np.arange(N)
    states[1] = np.arange(N)[::-1]                        # every 5-bit field rewritten, the blank in the last cell
    b = EnvBatch(_spec(orc.puzzle_spec(w, h, 5, 2, 256)), len(states), eng)
    b.set_state(states)
    assert np.array_equal(b.get_state(), states) and (b.depth() == 256).all()
    for i in (0, 1, 7, 63):
        o = orc.Env(orc.puzzle_spec(w, h, 5, 2, 256)); o.set_state(states[i].tolist())
        assert b.observe()[i].tolist() == o.observe() and b.masks()[i].tolist() == o.masks()
        assert bool(b.success()[i]) == o.success() and b.reward()[i] == np.float32(o.reward())
    assert b.success()[0] and not b.success()[1]
    tw.configure(device=0, precision=PRECISION)
    p = tw.env.Puzzle(w, h, 1, 2, 256)
    p.set_state(states[1].tolist())
    masks = p.masks()
    want = [int(t) for t in states[1]]
    for x, y, v in ((w - 1, 0, N - 1), (0, h - 1, 7), (w // 2, h // 2, N - 2), (0, h // 2, 1)):
        p.set_position(x, y, v)                           # one 5-bit field rewritten, blank and depth untouched
        want[y * w + x] = v
        assert p.get_position(x, y) == v and p.get_state() == want and p.masks() == masks
        assert p.observe() == [i * N + t for i, t in enumerate(want)]
    with pytest.raises(RuntimeError, match="tiles 0..cells-1"):
        p.set_position(0, 0, N)


def test_env_kinds_at_the_16_and_25_cell_limits(eng):
    """TWR_ENV_PUZZLE keeps its 16-cell limit; TWR_ENV_PUZZLE_WIDE takes boards of up to 25 cells (and smaller ones, in
    the byte encoding) and refuses 26 with a message naming its limit; Puzzle(w, h) picks the kind from the size."""
    import twisterl_b200 as tw
    from twisterl_b200 import _lib
    from twisterl_b200.env import EnvBatch
    TWR_ERR_UNSUPPORTED = -2
    L = _lib.load()
    for w, h in ((5, 5), (1, 25), (25, 1), (4, 4), (3, 3)):
        ok = EnvBatch(_lib.EnvSpec(_lib.ENV_PUZZLE_WIDE, w, h, 1, 1, 1), 2, eng)
        assert ok.get_state().tolist() == [list(range(w * h))] * 2 and ok.success().all()
        ok.set_state([[1, 0] + list(range(2, w * h))] * 2)
        x, y = 1 % w, 1 // w
        assert ok.masks().tolist() == [[x > 0, y > 0, x < w - 1, y < h - 1]] * 2 and not ok.success().any()
    for kind, w, h, msg in ((_lib.ENV_PUZZLE, 5, 5, "TWR_ENV_PUZZLE_WIDE"), (_lib.ENV_PUZZLE, 17, 1, "16 cells"),
                            (_lib.ENV_PUZZLE_WIDE, 2, 13, "25 cells"), (_lib.ENV_PUZZLE_WIDE, 6, 5, "25 cells")):
        with pytest.raises(RuntimeError, match=msg):
            EnvBatch(_lib.EnvSpec(kind, w, h, 1, 1, 1), 1, eng)
        assert L.twr_envs_create(eng._h, C.byref(_lib.EnvSpec(kind, w, h, 1, 1, 1)), 1, C.byref(C.c_void_p())) \
            == TWR_ERR_UNSUPPORTED
    tw.configure(device=0, precision=PRECISION)
    assert tw.env.spec_from_env(tw.env.Puzzle(5, 5, 3, 2, 64)).kind == _lib.ENV_PUZZLE_WIDE
    assert tw.env.spec_from_env(tw.env.Puzzle(4, 4, 3, 2, 64)).kind == _lib.ENV_PUZZLE


# --------------------------------------------------------------------------------------------------- forward ---
def _fp32_reference(pol, w, h, states, perm_idx=None):
    """the same forward on an fp32 engine: the kernel every engine must run for these tables"""
    import twisterl_b200 as tw
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import forward_batch
    ref = tw.Engine(device=0, precision="fp32", seed=SEED)
    try:
        b = EnvBatch(_spec(orc.puzzle_spec(w, h, 1, 2, 256)), len(states), ref)
        b.set_state(states)
        return forward_batch(ref, pol, b, perm_idx=perm_idx)
    finally:
        pol.release()
        ref.close()


@pytest.mark.parametrize("w,h,twists,E,H", [(5, 5, False, 512, 256), (5, 5, True, 512, 128), (4, 5, False, 512, 256),
                                            (3, 6, False, 256, 128), (4, 6, False, 512, 256), (5, 5, True, 256, 256)])
def test_forward_matches_oracle_on_the_fp32_kernel(eng, w, h, twists, E, H):
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import forward_batch
    pol, opol = _policies(w, h, twists, E, H)
    states = scramble_states(np.random.default_rng(E + H), 300, w, h, 120)
    perm = np.random.default_rng(3).integers(0, 2, size=len(states)).astype(np.int32) if twists else None
    b = EnvBatch(_spec(orc.puzzle_spec(w, h, 1, 2, 256)), len(states), eng)
    b.set_state(states)
    logits, values = forward_batch(eng, pol, b, perm_idx=perm)
    obs = b.observe()
    for i in range(len(states)):
        rl, rv = opol.raw_predict(obs[i].tolist(), -1 if perm is None else int(perm[i]))
        assert _close(logits[i], rl, TOL) and abs(values[i] - rv) <= TOL * max(1.0, abs(rv)), i
    rl, rv = _fp32_reference(pol, w, h, states, perm)
    assert np.array_equal(logits, rl) and np.array_equal(values, rv)        # the fp32 kernel ran, on every engine


def test_one_625_row_policy_runs_fp32_for_puzzle_and_pair_kernel_for_gridworld(eng):
    """On a tensor-core engine a 625-row policy is also packed as GridWorld 5x5's compact image; the launch-time guard
    keeps a 5x5 Puzzle off that operand (fp32 kernel, bit-identical to an fp32 engine) while a 5x5 GridWorld of the
    same policy still runs the pair kernel."""
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import forward_batch
    pol, opol = _policies(5, 5, False, 512, 128, seed=6)
    states = scramble_states(np.random.default_rng(1), 256, 5, 5, 200)
    b = EnvBatch(_spec(orc.puzzle_spec(5, 5, 1, 2, 256)), len(states), eng)
    b.set_state(states)
    pl, pv = forward_batch(eng, pol, b)
    g = EnvBatch(_spec(orc.gridworld_spec(5, 5, 64, 6)), 256, eng)
    g.reset(env_id_base=3, collect_id=1)
    gl, gv = forward_batch(eng, pol, g)
    gst = g.get_state()
    import twisterl_b200 as tw
    ref = tw.Engine(device=0, precision="fp32", seed=SEED)
    try:
        rb = EnvBatch(_spec(orc.puzzle_spec(5, 5, 1, 2, 256)), len(states), ref); rb.set_state(states)
        rl, rv = forward_batch(ref, pol, rb)
        rg = EnvBatch(_spec(orc.gridworld_spec(5, 5, 64, 6)), 256, ref); rg.set_state(gst)
        rgl, rgv = forward_batch(ref, pol, rg)
    finally:
        pol.release()
        ref.close()
    assert np.array_equal(pl, rl) and np.array_equal(pv, rv)
    obs = b.observe()
    for i in range(0, 256, 17):
        l, v = opol.raw_predict(obs[i].tolist())
        assert _close(pl[i], l, TOL) and abs(pv[i] - v) <= TOL * max(1.0, abs(v))
    if PRECISION == "fp32":
        assert np.array_equal(gl, rgl)
    else:                                                   # the pair kernel's rounding, not the fp32 kernel's
        assert not np.array_equal(gl, rgl) and _close(gl, rgl, 1e-3)


def test_full_predict_with_twists_on_5x5(eng):
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import full_predict_batch
    pol, opol = _policies(5, 5, True, 512, 256)
    states = scramble_states(np.random.default_rng(9), 200, 5, 5, 150)
    b = EnvBatch(_spec(orc.puzzle_spec(5, 5, 1, 2, 256)), len(states), eng)
    b.set_state(states)
    probs, values = full_predict_batch(eng, pol, b)
    obs, masks = b.observe(), b.masks()
    for i in range(len(states)):
        rp, rv = opol.full_predict(obs[i].tolist(), masks[i].tolist())
        assert np.allclose(probs[i], rp, atol=1e-5) and abs(values[i] - rv) <= 1e-5 * max(1.0, abs(rv)), i


# --------------------------------------------------------------------------------------------------- collect ---
@pytest.mark.parametrize("w,h,difficulty,episodes,twists", [(3, 6, 40, 300, False), (4, 5, 64, 300, False),
                                                             (5, 5, 64, 300, False), (5, 5, 128, 200, True)])
def test_collect_replays_through_oracle(eng, w, h, difficulty, episodes, twists):
    import twisterl_b200 as tw
    from parity import check_collect_against_oracle
    pol, opol = _policies(w, h, twists)
    ospec = orc.puzzle_spec(w, h, difficulty, 2, 256)
    env = tw.env.Puzzle(w, h, difficulty, 2, 256, add_perms=twists)
    col = tw.collector.PPOCollector(episodes, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(13)
    data = col.collect(env, pol)
    rep = check_collect_against_oracle(data, ospec, opol, seed=eng.seed, collect_id=13, gamma=0.995, lam=0.995, tol=TOL)
    assert rep["records"] == len(data.values_array) and data.stats["episodes"] == episodes
    assert set(np.unique(data.perms_array)) == ({0, 1} if twists else {-1})
    # collect_torch: the same collect handed off as CUDA tensors
    eng.set_collect_id(13)
    t = col.collect_torch(env, pol, dense_obs=False)
    R = len(data.values_array)
    for k, a in (("values", data.values_array), ("logits", data.logits_array), ("rewards", data.rewards_array)):
        assert np.array_equal(t[k].cpu().numpy().reshape(a.shape), a), k
    assert np.array_equal(t["obs"].cpu().numpy().reshape(R, -1).astype(np.int64), data.obs_array.astype(np.int64))
    pol.release()


def test_collect_full_size_properties_5x5(eng):
    """65 536 episodes of the 24-puzzle at difficulty 128: record count, ep_len, every observation an index set
    {25 i + v} over a permutation, legal moves between records, merge order, then replays spread over all tiles."""
    import twisterl_b200 as tw
    from parity import check_collect_against_oracle
    pol, opol = _policies(5, 5, False, 512, 256, seed=0)
    ospec = orc.puzzle_spec(5, 5, 128, 2, 256)
    env = tw.env.Puzzle(5, 5, 128, 2, 256)
    E = 65536
    col = tw.collector.PPOCollector(E, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(5)
    d = col.collect(env, pol)
    L, R = d.ep_len.astype(np.int64), len(d.values_array)
    assert L.min() >= 1 and L.max() <= 257 and L.sum() == R == d.stats["records"]
    tiles = d.obs_array.astype(np.int64) - np.arange(25) * 25
    assert (np.sort(tiles, axis=1) == np.arange(25)).all()
    order = orc.merge_order(E)
    starts = np.concatenate([[0], np.cumsum(L[order])])[:-1]
    ends = starts + L[order] - 1
    solved = (tiles == np.arange(25)).all(axis=1)
    rew = d.rewards_array
    inner = np.ones(R, bool); inner[ends] = False
    assert not solved[inner].any() and (rew[inner] == np.float32(-0.5 / 256)).all()
    assert (solved[ends] | (L[order] == 257)).all()
    assert int(solved[ends].sum()) == d.stats["successes"]
    blank = np.argmax(tiles == 0, axis=1)
    nxt = np.where(inner)[0]
    act = d.actions_array.astype(np.int64)[nxt]
    assert (blank[nxt + 1] - blank[nxt] == np.array([-1, -5, 1, 5])[act]).all()
    assert ((tiles[nxt + 1] != tiles[nxt]).sum(axis=1) == 2).all()
    masks = np.stack([blank % 5 > 0, blank // 5 > 0, blank % 5 < 4, blank // 5 < 4], 1)
    assert np.array_equal(d.logits_array == np.float32(-1e10), ~masks)
    adv, ret = d.additional_array("advs"), d.additional_array("rets")
    assert np.abs((ret - adv) - d.values_array).max() <= 1e-5 and np.array_equal(ret[ends], rew[ends])
    rep = check_collect_against_oracle(d, ospec, opol, seed=eng.seed, collect_id=5, gamma=0.995, lam=0.995, tol=TOL,
                                       max_episodes=16, stride=4093)
    assert rep["records"] > 16
    pol.release()


@pytest.mark.parametrize("twists", [False, True])
def test_collect_host_pipelined_matches_plain(eng, monkeypatch, twists):
    """twr_ppo_collect_host (sub-batches, packed action / twist / reward byte expanded by host threads) on the 24-puzzle:
    the host buffers hold exactly what the plain collect produces (u16 observation indices: obs_size 625)."""
    import twisterl_b200 as tw
    from twisterl_b200 import _lib, collector as twc
    pol, _ = _policies(5, 5, twists)
    env = tw.env.Puzzle(5, 5, 24, 2, 256, add_perms=twists)
    E = 1000
    col = tw.collector.PPOCollector(E, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(21)
    ref = col.collect(env, pol)
    L = _lib.load()
    spec = tw.env.spec_from_env(env)
    cap = int(L.twr_max_records(C.byref(spec), E))
    for parts in ("334,333,333", "1000"):
        monkeypatch.setenv("TWISTERL_B200_E2E_PARTS", parts)
        hb, arr, _ = twc._host_buffers(cap, 25, 4, E, pinned=True)
        out = _lib.Collected()
        eng.set_collect_id(21)
        _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), pol.device_handle(eng), None, E, 0.995, 0.995,
                                          C.byref(hb), C.byref(out)))
        R = int(out.n_records)
        assert R == len(ref.values_array) and int(out.successes) == ref.stats["successes"]
        assert np.array_equal(arr["ep_len"], ref.ep_len)
        for k, a in (("obs", ref.obs_array), ("actions", ref.actions_array), ("logits", ref.logits_array),
                     ("values", ref.values_array), ("rewards", ref.rewards_array), ("perms", ref.perms_array),
                     ("advs", ref.additional_array("advs")), ("rets", ref.additional_array("rets"))):
            assert np.array_equal(arr[k][:R], a), k
        hb_u8, _, _ = twc._host_buffers(cap, 25, 4, E, pinned=True, obs_u8=True)
        with pytest.raises(RuntimeError, match="obs_u8 needs obs_size <= 256"):
            _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), pol.device_handle(eng), None, E, 0.995, 0.995,
                                              C.byref(hb_u8), C.byref(out)))
    assert set(np.unique(ref.perms_array)) == ({0, 1} if twists else {-1})
    pol.release()


def test_collect_fused_gae_matches_twr_gae(eng):
    import twisterl_b200 as tw
    from twisterl_b200 import _lib
    pol, _ = _policies(4, 5, False, 256, 128, seed=5)
    E = 5000
    col = tw.collector.PPOCollector(E, 0.97, 0.9, 32, engine=eng)
    eng.set_collect_id(4)
    d = col.collect(tw.env.Puzzle(4, 5, 40, 2, 256), pol)
    r, v = np.ascontiguousarray(d.rewards_array, np.float32), np.ascontiguousarray(d.values_array, np.float32)
    R = len(v)
    L = d.ep_len.astype(np.int64)[orc.merge_order(E)]
    off = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    assert off[-1] == R > E
    adv = np.zeros(R, np.float32); ret = np.zeros(R, np.float32)
    _lib.check(_lib.load().twr_gae(eng._h, _lib.ptr(r), _lib.ptr(v), _lib.ptr(off), E, 0.97, 0.9, _lib.ptr(adv), _lib.ptr(ret)))
    assert np.array_equal(adv, d.additional_array("advs")) and np.array_equal(ret, d.additional_array("rets"))
    pol.release()


def test_gather_layout_on_one_gpu_5x5(eng):
    """The layout twr_gather_collected relies on: three engines as ranks 0..2 collect E episodes each; their records
    placed head_2, tail_0, head_0, tail_1, head_1, tail_2 and their ep_len concatenated equal one engine's collect of
    3E episodes, byte for byte."""
    import twisterl_b200 as tw
    W, E, cid = 3, 300, 77

    def arrays(d):
        return dict(obs=d.obs_array, logits=d.logits_array, values=d.values_array, rewards=d.rewards_array,
                    actions=d.actions_array, perms=d.perms_array, advs=d.additional_array("advs"),
                    rets=d.additional_array("rets"), ep_len=d.ep_len)

    def run(n, **kw):
        e = tw.Engine(device=0, precision=PRECISION, seed=SEED, **kw)
        pol, _ = _policies(5, 5, True)
        e.set_collect_id(cid)
        out = arrays(tw.collector.PPOCollector(n, 0.99, 0.95, 1, engine=e).collect(tw.env.Puzzle(5, 5, 32, 2, 256, add_perms=True), pol))
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
def _check_episodes(bs, bt, obs, obt, margins, what):
    diff = [i for i in range(len(bs)) if bs[i] != obs[i] or abs(float(bt[i]) - float(obt[i])) > 1e-5]
    for i in diff:
        assert margins[i] < NEAR_TIE, f"{what}: episode {i} differs with smallest margin {margins[i]}"
    assert len(diff) <= len(bs) // 4


@pytest.mark.parametrize("det,searches,mcts", [(True, 1, 0), (False, 4, 0), (False, 1, 8)])
def test_evaluate_matches_oracle_4x5(eng, det, searches, mcts):
    import twisterl_b200 as tw
    from twisterl_b200 import _lib
    pol, opol = _policies(4, 5, False, 256, 128, seed=8)
    ospec = orc.puzzle_spec(4, 5, 6, 2, 64)
    env = tw.env.Puzzle(4, 5, 6, 2, 64)
    n = 48 if mcts else 160
    spec = tw.env.spec_from_env(env)
    s, r = C.c_float(), C.c_float()
    bs, bt = np.zeros(n, np.float32), np.zeros(n, np.float32)
    eng.set_collect_id(7)
    _lib.check(_lib.load().twr_evaluate_episodes(eng._h, C.byref(spec), pol.device_handle(eng), n, int(det), searches,
                                                 mcts, 1.41, 1, C.byref(s), C.byref(r), _lib.ptr(bs), _lib.ptr(bt)))
    obs_, obt, mm = orc.evaluate_margins(ospec, opol, n, det, searches, seed=eng.seed, collect_id=7, num_mcts_searches=mcts,
                                         c_puct=1.41, max_expand_depth=1)
    _check_episodes(bs, bt, obs_, obt, mm, f"evaluate det={det} searches={searches} mcts={mcts}")
    assert abs(s.value - float(bs.mean())) < 1e-6
    pol.release()


def test_solve_and_az_collect_on_5x5(eng):
    import twisterl_b200 as tw
    tw.configure(device=0, precision=PRECISION, seed=SEED)
    pol, _ = _policies(5, 5, False, 256, 256)
    p = tw.env.Puzzle(5, 5, 3, 2, 64)
    p.reset()
    start = p.get_state()
    for det, mcts in ((True, 0), (False, 0), (False, 6)):
        p.set_state(start)
        (succ, rew), acts = tw.collector.solve(p, pol, det, 4, mcts, 1.41, 1)
        o = orc.Env(orc.puzzle_spec(5, 5, 3, 2, 64)); o.set_state(start)
        for a in acts:
            o.step(a)
        assert len(acts) <= 64 and succ in (0.0, 1.0) and bool(succ) == o.success()
    pol.release()
    pol, _ = _policies(5, 5, False, 256, 256)
    col = tw.collector.AZCollector(64, 12, 1.41, 1, 1, engine=eng)
    eng.set_collect_id(9)
    d = col.collect(tw.env.Puzzle(5, 5, 4, 2, 32), pol)
    R = len(d.obs_array)
    assert R == int(d.ep_len.sum()) and np.allclose(d.logits_array.sum(axis=1), 1.0, atol=1e-5)
    tiles = d.obs_array.astype(np.int64) - np.arange(25) * 25
    assert (np.sort(tiles, axis=1) == np.arange(25)).all()
    pol.release()


@pytest.mark.parametrize("E,H,twists,lockstep,persistent", [(256, 256, False, False, True), (256, 128, True, False, True),
                                                            (512, 128, False, False, True), (512, 256, False, False, False),
                                                            (256, 256, False, True, False)])
def test_mcts_paths_on_5x5(eng, capfd, monkeypatch, E, H, twists, lockstep, persistent):
    """pm_layout decides from the table size alone, so a 625-row Puzzle table takes the same paths as GridWorld 5x5's:
    persistent (table slice through shared memory, twist tables through the read-only path) up to E = 512 at H = 128;
    E = 512 at H = 256 needs 289 KB and runs the lockstep kernels, as does any search under TWISTERL_B200_MCTS_LOCKSTEP.
    Each case asserts which path ran and holds the search to the oracle under the near-tie rule."""
    from twisterl_b200 import _lib
    from twisterl_b200.env import EnvBatch
    pol, opol = _policies(5, 5, twists, E, H, seed=E + H)
    states = scramble_states(np.random.default_rng(E), 40, 5, 5, 10)
    monkeypatch.setenv("TWISTERL_B200_MCTS_DEBUG", "1")
    if lockstep:
        monkeypatch.setenv("TWISTERL_B200_MCTS_LOCKSTEP", "1")
    b = EnvBatch(_spec(orc.puzzle_spec(5, 5, 5, 2, 64)), len(states), eng)
    b.set_state(states)
    h = pol.device_handle(eng)
    n, sims = len(states), 16
    probs = np.zeros((n, 4), np.float32); visits = np.zeros((n, 4), np.int32)
    trace = np.zeros((sims, n, 2), np.int32)
    capfd.readouterr()
    n0 = eng.launch_count()
    _lib.check(_lib.load().twr_debug_mcts_trace(eng._h, h, b._h, sims, 1.41, 1, 700, 5, 1,
                                                _lib.ptr(probs), _lib.ptr(visits), _lib.ptr(trace)))
    launches = eng.launch_count() - n0
    ran_persistent = bool(DEBUG_LINE.findall(capfd.readouterr().err))
    assert ran_persistent == persistent, (ran_persistent, launches)
    if not persistent:
        assert launches > sims
    same = 0
    for i in range(n):
        env = orc.Env(orc.puzzle_spec(5, 5, 5, 2, 64)); env.set_state(states[i].tolist())
        op, ov = orc.mcts_probs(env, opol, sims, 1.41, 1, seed=eng.seed, collect_id=5, stream_id=700 + i, t=1)
        assert visits[i].sum() == ov.sum()
        if np.array_equal(visits[i], ov):
            same += 1
            assert np.allclose(probs[i], op, atol=1e-6)
            continue
        _, _, leaf, child, margin = orc.mcts_trace(env, opol, sims, 1.41, 1, seed=eng.seed, collect_id=5, stream_id=700 + i, t=1)
        div = next((s for s in range(sims) if trace[s, i, 0] != leaf[s] or trace[s, i, 1] != child[s]), None)
        assert div is not None and margin[div] < NEAR_TIE
    assert same >= n // 2
    pol.release()
