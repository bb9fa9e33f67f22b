"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs,
against the committed golden fixtures, and -- at BASELINE.json's full size -- through size-independent
properties.  Bars: bit-exact for env transitions / observations / masks / rewards / twists / episode
layout; |d| <= 1e-5 * max(1,|ref|) for fp32 logits and values (1e-4 for the f16x2
tensor-core forward, 1e-3 for f16x2w16 and f16f8c);
1e-5 for GAE (the kernel is in fact bit-exact); chi-square p > 0.001 for sampled actions."""
import os

import numpy as np
import pytest

from suite_loader import suite_precision

from helpers import (GOLDEN, gridworld_transpose_twists, obs_from_states, replays, scramble_states, synth_state_dict, trained15,
                     transpose_twists)
from oracle import orc

pytestmark = pytest.mark.gpu

PRECISION = suite_precision(globals())
TOL = {"fp32": 1e-5, "f16x2": 1e-4}.get(PRECISION, 1e-3)


@pytest.fixture(scope="module")
def eng():
    import twisterl_b200 as tw
    e = tw.Engine(device=0, precision=PRECISION, seed=0xABCDEF12345)
    yield e
    e.close()


def _spec(o):
    from twisterl_b200 import _lib
    return _lib.EnvSpec(o.kind, o.width, o.height, o.difficulty, o.depth_slope, o.max_depth)


def _close(a, ref, tol):
    return float((np.abs(a - ref) / np.maximum(1.0, np.abs(ref))).max(initial=0.0)) <= tol


# ------------------------------------------------------------------------ K1 ---
@pytest.mark.parametrize("key,w", [("puzzle8_35", 3), ("puzzle8_123", 3)])
def test_env_notebook_replays(eng, key, w):
    from twisterl_b200.env import EnvBatch
    r = replays()[key]
    b = EnvBatch(_spec(orc.puzzle_spec(w, w, 1, 2, 256)), 1, eng)
    b.set_state([r["start"]])
    assert b.depth()[0] == 256
    for a, board in zip(r["actions"], r["boards"][1:]):
        b.step([a])
        assert b.get_state()[0].tolist() == board
        assert b.observe()[0].tolist() == [i * 9 + v for i, v in enumerate(board)]
    assert b.success()[0] and b.is_final()[0] and b.reward()[0] == 1.0


def test_env_gridworld_notebook_replay(eng):
    from twisterl_b200.env import EnvBatch
    r = replays()["gridworld_4"]
    b = EnvBatch(_spec(orc.gridworld_spec(5, 5, 64, 1)), 1, eng)
    b.set_state([r["start"]])
    for a, board in zip(r["actions"], r["boards"][1:]):
        b.step([a])
        assert b.get_state()[0].tolist() == board
    assert b.success()[0] and b.reward()[0] == 1.0 and b.depth()[0] == 60


SPECS = [orc.puzzle_spec(4, 4, 128, 2, 256), orc.puzzle_spec(3, 3, 32, 2, 256), orc.puzzle_spec(2, 2, 3, 1, 10),
         orc.puzzle_spec(3, 2, 9, 3, 40), orc.puzzle_spec(4, 4, 0, 2, 256), orc.puzzle_spec(4, 4, 1, 2, 256),
         orc.gridworld_spec(5, 5, 64, 10), orc.gridworld_spec(4, 3, 7, 2), orc.gridworld_spec(5, 5, 64, 1)]


@pytest.mark.parametrize("ospec", SPECS, ids=lambda s: f"k{s.kind}_{s.width}x{s.height}_d{s.difficulty}")
def test_env_reset_and_forced_steps_bit_exact(eng, ospec):
    """reset from the shared Philox stream, then 40 forced (random, often illegal) actions: state,
    observation, masks, reward, final flag, success and depth must equal the oracle's at every step."""
    from twisterl_b200.env import EnvBatch
    n, steps = 257, 40
    rng = np.random.default_rng(ospec.width * 100 + ospec.difficulty)
    b = EnvBatch(_spec(ospec), n, eng)
    b.reset(env_id_base=1000, collect_id=3)
    envs = [orc.Env(ospec) for _ in range(n)]
    for i, e in enumerate(envs):
        e.reset(seed=eng.seed, env_id=1000 + i, collect_id=3)

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
    for t in range(steps):
        acts = rng.integers(0, 4, size=n)
        b.step(acts)
        for e, a in zip(envs, acts):
            e.step(int(a))
        if t % 4 == 3 or t < 3:
            compare(t)


def test_env_set_state_edge_cases(eng):
    from twisterl_b200.env import EnvBatch
    b = EnvBatch(_spec(orc.puzzle_spec(4, 4, 5, 2, 256)), 3, eng)
    states = [list(range(16)), [1, 0] + list(range(2, 16)), [5, 1, 2, 3, 4, 0] + list(range(6, 16))]
    b.set_state(states)
    assert b.get_state().tolist() == states and b.depth().tolist() == [256] * 3
    assert b.success().tolist() == [True, False, False]
    assert b.masks().tolist() == [[False, False, True, True], [True, False, True, True], [True, True, True, True]]
    with pytest.raises(RuntimeError, match="blank"):
        b.set_state([[1] * 16] * 3)
    # a tile label >= cells would index past the embedding table (the reference panics there): rejected, state untouched
    with pytest.raises(RuntimeError, match="tiles 0..cells-1"):
        b.set_state([[200] + list(range(1, 16))] + states[1:])
    with pytest.raises(RuntimeError, match="tiles 0..cells-1"):
        b.set_state([[16, 0] + list(range(2, 16))] + states[1:])
    assert b.get_state().tolist() == states
    g = EnvBatch(_spec(orc.gridworld_spec(5, 5, 64, 3)), 1, eng)
    with pytest.raises(RuntimeError, match="GridWorld cell values"):
        g.set_state([[4] + [0] * 24])
    with pytest.raises(RuntimeError, match="depth budget"):
        b.set_difficulty(1 << 24)
    # Puzzle.set_position (puzzle.rs:71-73): one cell poked, blank location / depth / masks as before
    import twisterl_b200 as tw
    tw.configure(device=0, precision=PRECISION)
    p = tw.env.Puzzle(3, 3, 1, 2, 256)
    p.set_state([1, 0, 2, 3, 4, 5, 6, 7, 8])
    masks = p.masks()
    p.set_position(2, 1, 7)
    o = orc.Env(orc.puzzle_spec(3, 3, 1, 2, 256)); o.set_state([1, 0, 2, 3, 4, 7, 6, 7, 8])
    assert p.get_position(2, 1) == 7 and p.get_state() == [1, 0, 2, 3, 4, 7, 6, 7, 8] and p.masks() == masks
    assert p.observe() == o.observe()
    with pytest.raises(RuntimeError, match="tiles 0..cells-1"):
        p.set_position(0, 0, 9)
    with pytest.raises(IndexError):
        p.set_position(3, 0, 1)
    empty = EnvBatch(_spec(orc.puzzle_spec(4, 4, 5, 2, 256)), 0, eng)
    assert empty.get_state().shape == (0, 16)
    empty.reset(); empty.step([])
    from twisterl_b200 import _lib
    with pytest.raises(RuntimeError, match="16 cells"):
        EnvBatch(_lib.EnvSpec(0, 5, 5, 1, 1, 1), 1, eng)
    with pytest.raises(RuntimeError, match="unknown env kind"):
        EnvBatch(_lib.EnvSpec(7, 2, 2, 1, 1, 1), 1, eng)


# ------------------------------------------------------------------------ K2 ---
def test_forward_matches_reference_torch_golden(eng):
    """logits/values of the reference's own torch BasicPolicy on the shipped ppo_puzzle15_v1.pt weights."""
    from parity import make_policies
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import forward_batch
    z, sd = trained15()
    pol, opol = make_policies(sd, 256)
    st = z["states"]
    b = EnvBatch(_spec(orc.puzzle_spec(4, 4, 1, 2, 256)), len(st), eng)
    b.set_state(st)
    logits, values = forward_batch(eng, pol, b)
    assert _close(logits, z["logits"], TOL) and _close(values, z["values"], TOL)
    # the split-operand tensor-core path is held to its measured margin too (1.1e-5 on these trained weights), not only
    # to the 1e-3 bar of a bf16 path
    if PRECISION not in ("f16x2w16", "f16f8c"):
        assert _close(logits, z["logits"], 1e-4) and _close(values, z["values"], 1e-4)
    assert _close(logits[0], np.array([-4.4116335, -5.16946, -2.0670972, 0.8337202], np.float32), TOL)
    # and against the oracle, element by element
    ref = np.array([np.append(*opol.raw_predict(o)) for o in obs_from_states(st[:128])])
    assert _close(logits[:128], ref[:, :4], TOL) and _close(values[:128], ref[:, 4], TOL)
    # masked variant = forward_with_perm
    ml, _ = forward_batch(eng, pol, b, apply_masks=True)
    mk = b.masks()
    assert np.array_equal(ml == np.float32(-1e10), ~mk)
    assert np.array_equal(ml[mk], logits[mk])


def test_forward_twists_match_reference_torch_golden(eng):
    from parity import make_policies
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import forward_batch, forward_obs
    z, sd = trained15()
    obs_perms, act_perms = transpose_twists(4)
    pol, opol = make_policies(sd, 256, obs_perms, act_perms)
    st = z["states"]
    b = EnvBatch(_spec(orc.puzzle_spec(4, 4, 1, 2, 256)), len(st), eng)
    b.set_state(st)
    logits, values = forward_batch(eng, pol, b, perm_idx=z["twist_perm_idx"])
    assert _close(logits, z["twist_logits"], TOL) and _close(values, z["twist_values"], TOL)
    # the direct-observation entry point gives the same numbers
    l2, v2 = forward_obs(eng, pol, obs_from_states(st), z["twist_perm_idx"])
    assert np.array_equal(l2, logits) and np.array_equal(v2, values)
    # twist consistency: value is invariant, logits permute (transpose symmetry of the puzzle)
    with pytest.raises(RuntimeError, match="perm_idx"):
        forward_batch(eng, pol, b, perm_idx=np.full(len(st), 2))


@pytest.mark.parametrize("name,N,kind", [("puzzle8", 9, 0), ("gridworld", 25, 1)])
def test_forward_other_config_shapes(eng, name, N, kind):
    from parity import make_policies
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import forward_batch
    z = np.load(GOLDEN / "policy_synth.npz")
    sd = synth_state_dict(int(z[f"{name}.seed"]), N * N, 512, int(z[f"{name}.hidden"]), 4)
    pol, _ = make_policies(sd, N * N)
    st = z[f"{name}.states"]
    spec = orc.puzzle_spec(3, 3, 1, 2, 256) if kind == 0 else orc.gridworld_spec(5, 5, 64, 3)
    b = EnvBatch(_spec(spec), len(st), eng)
    b.set_state(st)
    logits, values = forward_batch(eng, pol, b)
    assert _close(logits, z[f"{name}.logits"], TOL) and _close(values, z[f"{name}.values"], TOL)


def test_forward_ragged_batch_sizes(eng):
    """batch sizes around the 128-env tile: 1, 127, 128, 129, 1000."""
    from parity import make_policies
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import forward_batch
    z, sd = trained15()
    pol, _ = make_policies(sd, 256)
    for n in (1, 127, 128, 129, 1000):
        st = np.tile(z["states"], (2, 1))[:n]
        b = EnvBatch(_spec(orc.puzzle_spec(4, 4, 1, 2, 256)), n, eng)
        b.set_state(st)
        logits, values = forward_batch(eng, pol, b)
        ref_l, ref_v = np.tile(z["logits"], (2, 1))[:n], np.tile(z["values"], 2)[:n]
        assert _close(logits, ref_l, TOL) and _close(values, ref_v, TOL), n


def test_policy_scalar_api_and_unsupported_shapes(eng):
    import twisterl_b200 as tw
    from parity import make_policies
    z, sd = trained15()
    obs_perms, act_perms = transpose_twists(4)
    pol, opol = make_policies(sd, 256, obs_perms, act_perms)
    tw.configure(device=0, precision=PRECISION)
    o = obs_from_states(z["states"])[5].tolist()
    masks = [True, False, True, True]
    probs, value = pol.full_predict(o, masks)
    rp, rv = opol.full_predict(o, masks)
    assert np.allclose(probs, rp, atol=max(TOL, 1e-5)) and abs(value - rv) <= max(TOL, 1e-5) * max(1, abs(rv))
    ml, v = pol.forward(o, masks)
    assert ml[1] == -1e10 and len(ml) == 4
    deep = tw.nn.Policy(pol.embeddings, tw.nn.Sequential(pol.common.layers * 2), pol.action_net, pol.value_net, [], [])
    with pytest.raises(RuntimeError, match="do not chain"):                   # Linear(512,256) twice: sizes do not chain
        deep.device_handle(eng)
    conv = tw.nn.Policy(tw.nn.EmbeddingBag(np.zeros((15, 32)), np.zeros(512), True, [16, 16], 0), pol.common,
                        pol.action_net, pol.value_net, [], [])
    with pytest.raises(RuntimeError, match="obs_shape\\[conv_dim\\] vectors"):     # Conv1d table with a missing row
        conv.device_handle(eng)


# ------------------------------------------------------------------------ K3 ---
def _sample(eng, logits, env_id_base, step, cid):
    import ctypes as C
    from twisterl_b200 import _lib
    l = np.ascontiguousarray(logits, dtype=np.float32)
    n, A = l.shape
    acts = np.zeros(n, np.int32); u = np.zeros((n, A), np.float32)
    _lib.check(_lib.load().twr_sample(eng._h, _lib.ptr(l), n, A, env_id_base, step, cid, _lib.ptr(acts), _lib.ptr(u)))
    return acts, u


def test_sample_uses_shared_philox_stream_and_matches_oracle(eng):
    rng = np.random.default_rng(3)
    n = 4096
    logits = rng.normal(0, 2, size=(n, 4)).astype(np.float32)
    logits[rng.random((n, 4)) < 0.2] = -1e10
    logits[:, 0][np.all(logits == -1e10, axis=1)] = 0.0
    acts, u = _sample(eng, logits, 77, 9, 4)
    key = [eng.seed & 0xFFFFFFFF, eng.seed >> 32]
    mism = 0
    for i in range(n):
        w = orc.philox([77 + i, 9, orc.RNG_SAMPLE, 4], key)
        ref_u = [orc.u32_to_unit_f32(int(x)) for x in w]
        assert u[i].tolist() == ref_u                                  # uniforms bit-exact
        with np.errstate(divide="ignore"):
            g = np.sort(logits[i].astype(np.float64) - np.log(np.abs(np.log(u[i].astype(np.float64)))))
        if g[-1] - g[-2] > 1e-4:                                       # libm vs CUDA logf: <= 1 ulp apart
            mism += orc.sample_from_logits(logits[i], ref_u) != acts[i]
        assert logits[i, acts[i]] != np.float32(-1e10)                 # a masked action is never sampled
    assert mism == 0


def test_sample_distribution_chi_square(eng):
    logits = np.tile(np.array([[0.3, -1e10, 1.2, -0.8]], np.float32), (1_000_000, 1))
    acts, _ = _sample(eng, logits, 0, 0, 0)
    cnt = np.bincount(acts, minlength=4).astype(np.float64)
    p = np.exp(np.array([0.3, -np.inf, 1.2, -0.8])); p /= p.sum()
    assert cnt[1] == 0
    keep = [0, 2, 3]
    chi2 = (((cnt[keep] - 1e6 * p[keep]) ** 2) / (1e6 * p[keep])).sum()
    assert chi2 < 13.82, chi2                                           # p > 0.001 at 2 degrees of freedom


# ------------------------------------------------------------------------ K4 ---
def test_gae_matches_oracle(eng):
    from twisterl_b200 import _lib
    rng = np.random.default_rng(5)
    lens = np.concatenate([[1, 2, 257, 1, 3], rng.integers(1, 258, size=300)])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    R = int(off[-1])
    r = rng.normal(0, 1, R).astype(np.float32); v = rng.normal(0, 1, R).astype(np.float32)
    adv = np.zeros(R, np.float32); ret = np.zeros(R, np.float32)
    _lib.check(_lib.load().twr_gae(eng._h, _lib.ptr(r), _lib.ptr(v), _lib.ptr(off), len(lens), 0.995, 0.995,
                                   _lib.ptr(adv), _lib.ptr(ret)))
    for i in range(len(lens)):
        a, g = orc.gae(r[off[i]:off[i + 1]], v[off[i]:off[i + 1]], 0.995, 0.995)
        assert np.abs(a - adv[off[i]:off[i + 1]]).max() <= 1e-5 and np.abs(g - ret[off[i]:off[i + 1]]).max() <= 1e-5
        assert np.array_equal(a, adv[off[i]:off[i + 1]]) and np.array_equal(g, ret[off[i]:off[i + 1]])
    # known answer derived from collector/ppo.rs:82-92 with r=v=1, gamma=.9, lambda=.95
    o2 = np.array([0, 2], np.int64); one = np.ones(2, np.float32); a2 = np.zeros(2, np.float32); g2 = np.zeros(2, np.float32)
    _lib.check(_lib.load().twr_gae(eng._h, _lib.ptr(one), _lib.ptr(one), _lib.ptr(o2), 1, 0.9, 0.95, _lib.ptr(a2), _lib.ptr(g2)))
    assert np.allclose(g2, [1.9, 1.0], atol=1e-7) and np.allclose(a2, [0.9, 0.0], atol=1e-7)


# ------------------------------------------------------------------- collect ---
CASES = [
    ("puzzle8", orc.puzzle_spec(3, 3, 6, 2, 256), 81, 256, 700, False),
    ("puzzle15_d1", orc.puzzle_spec(4, 4, 1, 2, 256), 256, 256, 300, False),
    ("puzzle15_d32_twists", orc.puzzle_spec(4, 4, 32, 2, 256), 256, 256, 130, True),
    ("gridworld", orc.gridworld_spec(5, 5, 64, 10), 625, 128, 400, False),
    ("gridworld_twists", orc.gridworld_spec(5, 5, 64, 10), 625, 128, 300, True),
    ("one_episode", orc.puzzle_spec(4, 4, 4, 2, 256), 256, 256, 1, False),
]


@pytest.mark.parametrize("name,ospec,obs_size,hidden,episodes,twists", CASES, ids=[c[0] for c in CASES])
def test_collect_replays_through_oracle(eng, name, ospec, obs_size, hidden, episodes, twists):
    import twisterl_b200 as tw
    from parity import check_collect_against_oracle, make_policies
    if obs_size == 256:
        _, sd = trained15()
    else:
        sd = synth_state_dict(21, obs_size, 512, hidden, 4)
    perms = (gridworld_transpose_twists(5) if ospec.kind == 1 else transpose_twists(4)) if twists else ((), ())
    pol, opol = make_policies(sd, obs_size, *perms)
    env = (tw.env.Puzzle(ospec.width, ospec.height, ospec.difficulty, ospec.depth_slope, ospec.max_depth)
           if ospec.kind == 0 else tw.env.GridWorld(ospec.width, ospec.height, ospec.max_depth, ospec.difficulty))
    col = tw.collector.PPOCollector(episodes, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(11)
    data = col.collect(env, pol)
    rep = check_collect_against_oracle(data, ospec, opol, seed=eng.seed, collect_id=11, gamma=0.995, lam=0.995, tol=TOL)
    assert rep["records"] == len(data.values_array)
    assert data.stats["episodes"] == episodes and data.stats["records"] == rep["records"]
    if twists:
        assert set(np.unique(data.perms_array)) == {0, 1}
    else:
        assert (data.perms_array == -1).all()
    # same call again: collect_id advanced -> different rollouts; pinned id -> identical rollouts
    eng.set_collect_id(11)
    again = col.collect(env, pol)
    assert np.array_equal(again.obs_array, data.obs_array) and np.array_equal(again.actions_array, data.actions_array)
    assert np.array_equal(again.additional_array("rets"), data.additional_array("rets"))
    # whole-collect comparison with the oracle collector on the same streams (actions can differ only
    # where ulp-level logit differences flip a Gumbel near-tie)
    oc = orc.ppo_collect(ospec, opol, episodes, 0.995, 0.995, seed=eng.seed, collect_id=11)
    same = sum(int(a == b) for a, b in zip(oc["ep_len"], data.ep_len))
    assert same >= 0.98 * episodes
    if oc["n_records"] == rep["records"] and np.array_equal(oc["actions"], data.actions_array):
        assert np.array_equal(oc["obs"], data.obs_array) and np.array_equal(oc["rewards"], data.rewards_array)
        assert _close(data.logits_array, oc["logits"], TOL) and np.abs(oc["rets"] - data.additional_array("rets")).max() <= 1e-4


def test_collect_reference_semantics(eng):
    """terminal state recorded, merge order [last, 0..n-2], list-valued drop-in properties."""
    import twisterl_b200 as tw
    from parity import make_policies
    sd = synth_state_dict(2, 4, 512, 128, 4)
    pol, _ = make_policies(sd, 4)
    env = tw.env.Puzzle(2, 1, 1, 1, 10)                                # 1 or 2 records per episode
    col = tw.collector.PPOCollector(num_episodes=64, gamma=0.9, num_cores=1, **{"lambda": 0.95})
    col._engine = eng
    d = col.collect(env, pol)
    assert set(d.ep_len.tolist()) == {1, 2}
    assert isinstance(d.obs, list) and isinstance(d.obs[0], list) and len(d.obs) == int(d.ep_len.sum())
    assert set(d.additional_data) == {"advs", "rets"} and len(d.additional_data["rets"]) == len(d.obs)
    assert d.get_additional_data_item("advs") is not None
    order = orc.merge_order(64)
    off = 0
    for ep in order:                                                   # first chunk is the LAST episode
        n = int(d.ep_len[ep])
        last = d.obs_array[off + n - 1].tolist()
        if n == 2:
            assert d.rewards_array[off] == np.float32(-0.5 / 10) and last in ([0, 3], [1, 2])
            assert d.rewards_array[off + 1] in (np.float32(1.0), np.float32(-0.5))
        else:
            assert last == [0, 3] and d.rewards_array[off] == 1.0       # scramble no-op: solved at reset
        off += n
    with pytest.raises(RuntimeError, match="No data in collected data chunks to merge"):
        tw.collector.PPOCollector(0, 0.9, 0.9, 1, engine=eng).collect(env, pol)
    big, _ = make_policies(synth_state_dict(2, 256, 512, 256, 4), 256)
    with pytest.raises(RuntimeError, match="obs_size"):
        col.collect(env, big)


def test_collect_full_size_properties(eng):
    """BASELINE config 2 size (65 536 envs, puzzle15, difficulty 128): size-independent properties."""
    import twisterl_b200 as tw
    from parity import check_collect_against_oracle, make_policies
    sd = synth_state_dict(0, 256, 512, 256, 4)
    pol, opol = make_policies(sd, 256)
    ospec = orc.puzzle_spec(4, 4, 128, 2, 256)
    env = tw.env.Puzzle(4, 4, 128, 2, 256)
    E = 65536
    col = tw.collector.PPOCollector(E, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(5)
    d = col.collect(env, pol)
    L, R = d.ep_len.astype(np.int64), len(d.values_array)
    assert L.min() >= 1 and L.max() <= 257 and L.sum() == R == d.stats["records"]
    obs = d.obs_array.astype(np.int64)
    tiles = obs - np.arange(16) * 16
    assert tiles.min() >= 0 and tiles.max() <= 15
    assert (np.sort(tiles, axis=1) == np.arange(16)).all()              # every record is a permutation board
    order = orc.merge_order(E)
    starts = np.concatenate([[0], np.cumsum(L[order])])[:-1]
    ends = starts + L[order] - 1
    solved = (tiles == np.arange(16)).all(axis=1)
    rew = d.rewards_array
    assert set(np.unique(rew)) <= {np.float32(1.0), np.float32(-0.5), np.float32(-0.5 / 256)}
    inner = np.ones(R, bool); inner[ends] = False
    assert not solved[inner].any() and (rew[inner] == np.float32(-0.5 / 256)).all()
    assert (solved[ends] | (L[order] == 257)).all()                     # episodes end solved or out of budget
    assert (rew[ends] == np.where(solved[ends], np.float32(1.0), np.float32(-0.5))).all()
    assert int(solved[ends].sum()) == d.stats["successes"]
    # consecutive records inside an episode differ by one legal blank move matching the recorded action
    blank = np.argmax(tiles == 0, axis=1)
    nxt = np.where(inner)[0]
    delta = blank[nxt + 1] - blank[nxt]
    act = d.actions_array.astype(np.int64)[nxt]
    exp = np.array([-1, -4, 1, 4])[act]
    legal = np.stack([blank[nxt] % 4 > 0, blank[nxt] // 4 > 0, blank[nxt] % 4 < 3, blank[nxt] // 4 < 3], 1)[np.arange(len(nxt)), act]
    assert (legal).all(), "a masked (illegal) action was sampled"
    assert (delta == exp).all()
    changed = (tiles[nxt + 1] != tiles[nxt]).sum(axis=1)
    assert (changed == 2).all()
    # masked logits exactly where the move is illegal
    bl = blank
    masks = np.stack([bl % 4 > 0, bl // 4 > 0, bl % 4 < 3, bl // 4 < 3], 1)
    assert np.array_equal(d.logits_array == np.float32(-1e10), ~masks)
    # GAE identity on every record: rets - advs == values ; terminal rets == rewards
    adv, ret = d.additional_array("advs"), d.additional_array("rets")
    assert np.abs((ret - adv) - d.values_array).max() <= 1e-5
    assert np.array_equal(ret[ends], rew[ends])
    # and the full replay check on the first 24 episodes in merge order, then on 40 episodes spread over all tiles
    # (own and time-split groups of the balanced schedule alike)
    rep = check_collect_against_oracle(d, ospec, opol, seed=eng.seed, collect_id=5, gamma=0.995, lam=0.995, tol=TOL,
                                       max_episodes=24)
    assert rep["records"] > 24
    rep = check_collect_against_oracle(d, ospec, opol, seed=eng.seed, collect_id=5, gamma=0.995, lam=0.995, tol=TOL,
                                       max_episodes=40, stride=1637)
    assert rep["records"] > 40


@pytest.mark.parametrize("twists", [False, True])
def test_collect_host_pipelined_matches_plain(eng, monkeypatch, twists):
    """twr_ppo_collect_host splits large collects into sub-batches whose D2H overlaps the next rollout, and moves action /
    twist index / reward as one packed byte (advantages not at all) that host threads expand; the host buffers must hold
    exactly what the plain collect + to_host path produces."""
    import ctypes as C
    import twisterl_b200 as tw
    from parity import make_policies
    from twisterl_b200 import _lib, collector as twc
    _, sd = trained15()
    pol, _ = make_policies(sd, 256, *(transpose_twists(4) if twists else ((), ())))
    env = tw.env.Puzzle(4, 4, 12, 2, 256)
    E = 1000
    col = tw.collector.PPOCollector(E, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(21)
    ref = col.collect(env, pol)
    L = _lib.load()
    spec = tw.env.spec_from_env(env)
    cap = int(L.twr_max_records(C.byref(spec), E))
    # "1000" with u8 still runs the pipelined body (one sub-batch); the last split is unequal
    for parts, u8 in (("334,333,333", False), ("143,143,143,143,143,143,142", True), ("1000", True), ("600,300,100", True)):
        monkeypatch.setenv("TWISTERL_B200_E2E_PARTS", parts)
        hb, arr, _ = twc._host_buffers(cap, 16, 4, E, pinned=True, obs_u8=u8)   # u8: one-byte observation indices
        out = _lib.Collected()
        eng.set_collect_id(21)
        _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), pol.device_handle(eng), None, E, 0.995, 0.995,
                                          C.byref(hb), C.byref(out)))
        R = int(out.n_records)
        assert R == len(ref.values_array) and int(out.successes) == ref.stats["successes"]
        assert abs(out.reward_sum - ref.stats["reward_sum"]) < 1e-6
        assert np.array_equal(arr["ep_len"], ref.ep_len)
        assert np.array_equal(arr["obs"][:R], ref.obs_array) and np.array_equal(arr["actions"][:R], ref.actions_array)
        assert np.array_equal(arr["logits"][:R], ref.logits_array) and np.array_equal(arr["values"][:R], ref.values_array)
        assert np.array_equal(arr["rewards"][:R], ref.rewards_array) and np.array_equal(arr["perms"][:R], ref.perms_array)
        assert np.array_equal(arr["advs"][:R], ref.additional_array("advs"))
        assert np.array_equal(arr["rets"][:R], ref.additional_array("rets"))
    assert set(np.unique(ref.perms_array)) == ({0, 1} if twists else {-1})
    assert len(set(np.unique(ref.rewards_array))) >= 2            # step reward and solved (and, for some seeds, out-of-budget) all cross as codes


@pytest.mark.parametrize("E,difficulty", [(5000, 40), (33, 3), (20000, 128)])
def test_collect_fused_gae_matches_twr_gae(eng, E, difficulty):
    """The PPO collect computes advantages and returns inside the compaction pass (k_compact<true>: reverse walk over the
    time tiles, collector/ppo.rs:82-92 per episode).  twr_gae, the stand-alone GAE held to the oracle by
    test_gae_matches_oracle, run on the same collect's rewards and values must give the same arrays, bit for bit."""
    import twisterl_b200 as tw
    from parity import make_policies
    from twisterl_b200 import _lib
    pol, _ = make_policies(synth_state_dict(5, 256, 512, 256, 4), 256)
    env = tw.env.Puzzle(4, 4, difficulty, 2, 256)
    col = tw.collector.PPOCollector(E, 0.97, 0.9, 32, engine=eng)
    eng.set_collect_id(4)
    d = col.collect(env, pol)
    r, v = np.ascontiguousarray(d.rewards_array, np.float32), np.ascontiguousarray(d.values_array, np.float32)
    R = len(v)
    assert R > E
    L = d.ep_len.astype(np.int64)[orc.merge_order(E)]
    off = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    assert off[-1] == R
    adv = np.zeros(R, np.float32); ret = np.zeros(R, np.float32)
    _lib.check(_lib.load().twr_gae(eng._h, _lib.ptr(r), _lib.ptr(v), _lib.ptr(off), E, 0.97, 0.9, _lib.ptr(adv), _lib.ptr(ret)))
    assert np.array_equal(d.additional_array("advs"), adv)
    assert np.array_equal(d.additional_array("rets"), ret)
    pol.release()


@pytest.mark.parametrize("E,difficulty,chunk,trained", [(65536, 128, None, False), (60000, 6, "8", True), (57100, 20, "5", False),
                                                        (45000, 40, None, False), (38400, 24, "6", True)])     # the last two: two own groups per pair
def test_collect_balanced_schedule_matches_plain(eng, monkeypatch, E, difficulty, chunk, trained):
    """The persistent pair kernel cuts left-over tile groups along time and hands them from CTA pair to CTA pair
    (Sched in twr_forward_tc2.cu).  Scheduling must not change a single byte: the same collect with the balanced
    schedule off (TWISTERL_B200_BALANCE=0, oracle-checked by the replay tests) gives identical records."""
    if PRECISION == "fp32":
        pytest.skip("the fused persistent kernel is the tensor-core path")
    import twisterl_b200 as tw
    from parity import make_policies
    sd = trained15()[1] if trained else synth_state_dict(3, 256, 512, 256, 4)
    pol, _ = make_policies(sd, 256, *(transpose_twists(4) if trained else ((), ())))
    env = tw.env.Puzzle(4, 4, difficulty, 2, 256)
    col = tw.collector.PPOCollector(E, 0.995, 0.995, 32, engine=eng)
    if chunk:
        monkeypatch.setenv("TWISTERL_B200_CHUNK", chunk)
    out = []
    for bal in ("0", "2", "3", "6"):
        monkeypatch.setenv("TWISTERL_B200_BALANCE", bal)
        eng.set_collect_id(9)
        d = col.collect(env, pol)
        out.append(d)
    ref = out[0]
    for d in out[1:]:
        assert np.array_equal(d.ep_len, ref.ep_len) and d.stats == ref.stats
        assert np.array_equal(d.obs_array, ref.obs_array) and np.array_equal(d.actions_array, ref.actions_array)
        assert np.array_equal(d.logits_array, ref.logits_array) and np.array_equal(d.values_array, ref.values_array)
        assert np.array_equal(d.rewards_array, ref.rewards_array) and np.array_equal(d.perms_array, ref.perms_array)
        assert np.array_equal(d.additional_array("advs"), ref.additional_array("advs"))
        assert np.array_equal(d.additional_array("rets"), ref.additional_array("rets"))


@pytest.mark.parametrize("conv_dim", [0, 1])
def test_conv1d_policy_forward_and_collect(eng, conv_dim):
    """SURVEY 8f row f4: Conv1dPolicy (2-D EmbeddingBag path, nn/layers.rs:63-77) on the device -- forward against
    the reference's own torch Conv1dPolicy (golden fixture), +/- twists, then a collect replayed through the oracle."""
    import twisterl_b200 as tw
    from helpers import synth_conv_state_dict
    from parity import check_collect_against_oracle, make_conv1d_policies
    from twisterl_b200.nn import forward_obs
    g = np.load(GOLDEN / "policy_conv1d.npz")
    sd = synth_conv_state_dict(int(g[f"dim{conv_dim}.seed"]), 16, 32, 512, 256, 4)
    obs = obs_from_states(g["states"])
    pol, opol = make_conv1d_policies(sd, [16, 16], conv_dim)
    l, v = forward_obs(eng, pol, obs, None)
    assert _close(l, g[f"dim{conv_dim}.plain.logits"], TOL) and _close(v, g[f"dim{conv_dim}.plain.values"], TOL)
    tpol, topol = make_conv1d_policies(sd, [16, 16], conv_dim, *transpose_twists(4))
    l, v = forward_obs(eng, tpol, obs, g["twist_perm_idx"])
    assert _close(l, g[f"dim{conv_dim}.twist.logits"], TOL) and _close(v, g[f"dim{conv_dim}.twist.values"], TOL)
    ospec = orc.puzzle_spec(4, 4, 5, 2, 256)
    env = tw.env.Puzzle(4, 4, 5, 2, 256)
    col = tw.collector.PPOCollector(200, 0.995, 0.995, 1, engine=eng)
    eng.set_collect_id(31)
    data = col.collect(env, tpol)
    rep = check_collect_against_oracle(data, ospec, topol, seed=eng.seed, collect_id=31, gamma=0.995, lam=0.995, tol=TOL)
    assert rep["records"] == len(data.values_array)
    # weight refresh keeps working on the expanded table (twr_policy_update re-expands)
    sd2 = synth_conv_state_dict(77, 16, 32, 512, 256, 4)
    pol2, opol2 = make_conv1d_policies(sd2, [16, 16], conv_dim)
    l2, _ = forward_obs(eng, pol2, obs[:8], None)
    ref = np.array([opol2.raw_predict(o)[0] for o in obs[:8]])
    assert _close(l2, ref, TOL)


def test_forward_obs_multiset_and_wide_tables_use_the_fp32_kernel(eng):
    """EmbeddingBag sums repeated indices (layers.rs:58-62); the one-hot tensor-core operand cannot, so such calls --
    and tables wider than 256 rows -- must run the fp32 kernel on an f16x2 engine instead of failing."""
    from parity import make_policies
    from twisterl_b200.nn import forward_obs
    _, sd = trained15()
    pol, opol = make_policies(sd, 256)
    obs = np.array([[3, 3, 17, 40, 41, 42, 43, 44, 45, 46, 47, 48, 49, 50, 51, 255],
                    [0, 17, 34, 51, 68, 85, 102, 119, 136, 153, 170, 187, 204, 221, 238, 255]], np.int32)
    l, v = forward_obs(eng, pol, obs, None)
    for k in range(2):
        rl, rv = opol.raw_predict(obs[k].tolist())
        assert _close(l[k], rl, TOL) and abs(v[k] - rv) <= TOL * max(1.0, abs(rv))


@pytest.mark.parametrize("E", [30000, 20000])
def test_collect_mid_size_sampled_replay(eng, E):
    """Between one and two tiles per CTA pair (two with the deferred fused step, and pairs with one and two tiles in
    the same launch): every 211th episode, spread over all tiles, is replayed record by record through the oracle."""
    import twisterl_b200 as tw
    from parity import check_collect_against_oracle, make_policies
    _, sd = trained15()
    pol, opol = make_policies(sd, 256, *transpose_twists(4))
    ospec = orc.puzzle_spec(4, 4, 18, 2, 256)
    env = tw.env.Puzzle(4, 4, 18, 2, 256)
    col = tw.collector.PPOCollector(E, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(17)
    d = col.collect(env, pol)
    rep = check_collect_against_oracle(d, ospec, opol, seed=eng.seed, collect_id=17, gamma=0.995, lam=0.995, tol=TOL, stride=211)
    assert rep["records"] > 200


def test_deep_stack_policy_forward_and_collect(eng):
    """SURVEY 8f row f4, second half: general layer stacks run k_forward_generic -- forward against the reference's own
    torch BasicPolicy with deeper stacks (golden fixture), +/- twists, a collect replayed through the oracle, evaluate,
    a head-only policy (no common layer), and the in-place weight refresh."""
    import twisterl_b200 as tw
    from helpers import synth_deep_state_dict
    from parity import check_collect_against_oracle, make_policies_general
    from twisterl_b200.nn import forward_obs
    g = np.load(GOLDEN / "policy_deep.npz")
    sd = synth_deep_state_dict(int(g["seed"]), 256, 512, (256, 128), (64,), (32,), 4)
    obs = obs_from_states(g["states"])
    pol, opol = make_policies_general(sd, 256)
    l, v = forward_obs(eng, pol, obs, None)
    assert _close(l, g["plain.logits"], 1e-5) and _close(v, g["plain.values"], 1e-5)       # fp32 kernel on either engine
    tpol, topol = make_policies_general(sd, 256, *transpose_twists(4))
    l, v = forward_obs(eng, tpol, obs, g["twist_perm_idx"])
    assert _close(l, g["twist.logits"], 1e-5) and _close(v, g["twist.values"], 1e-5)
    ospec = orc.puzzle_spec(4, 4, 6, 2, 256)
    env = tw.env.Puzzle(4, 4, 6, 2, 256)
    eng.set_collect_id(41)
    data = tw.collector.PPOCollector(150, 0.995, 0.995, 1, engine=eng).collect(env, tpol)
    rep = check_collect_against_oracle(data, ospec, topol, seed=eng.seed, collect_id=41, gamma=0.995, lam=0.995, tol=1e-5)
    assert rep["records"] == len(data.values_array)
    s, r = tw.collector.evaluate(env, pol, 32, True, 1, 0, 0, 1.4, 1, 1) if eng is tw.default_engine() else (0.0, 0.0)
    assert 0.0 <= s <= 1.0
    # no common layer at all: heads read the embedding directly
    hsd = synth_deep_state_dict(9, 256, 128, (), (), (), 4)
    hpol, hopol = make_policies_general(hsd, 256)
    l, v = forward_obs(eng, hpol, obs[:16], None)
    ref = [hopol.raw_predict(o) for o in obs[:16]]
    assert _close(l, np.array([x[0] for x in ref]), 1e-5) and _close(v, np.array([x[1] for x in ref]), 1e-5)
    # twr_policy_update keeps the layer layout
    sd2 = synth_deep_state_dict(77, 256, 512, (256, 128), (64,), (32,), 4)
    pol2, opol2 = make_policies_general(sd2, 256)
    l2, _ = forward_obs(eng, pol2, obs[:8], None)
    assert _close(l2, np.array([opol2.raw_predict(o)[0] for o in obs[:8]]), 1e-5)


def test_collect_schedule_sweep_matches_plain(eng, monkeypatch):
    """Batch sizes around every regime boundary of the persistent kernel's schedule (one / two / three tiles per CTA pair,
    whole and ragged tile counts, left-over groups from 1 to P-1): balanced == plain, byte for byte."""
    if PRECISION == "fp32":
        pytest.skip("the fused persistent kernel is the tensor-core path")
    import twisterl_b200 as tw
    from parity import make_policies
    pol, _ = make_policies(synth_state_dict(5, 256, 512, 256, 4), 256)
    env = tw.env.Puzzle(4, 4, 16, 2, 256)                      # horizon 33 -> 4-step launches (the shortest balanced ones)
    for E in (1, 255, 257, 18944, 18945, 37887, 37889, 38000, 47000, 56831, 56833, 57088, 65535, 70001, 75776):
        col = tw.collector.PPOCollector(E, 0.995, 0.995, 32, engine=eng)
        out = []
        for bal in ("0", "2"):
            monkeypatch.setenv("TWISTERL_B200_BALANCE", bal)
            eng.set_collect_id(3)
            out.append(col.collect(env, pol))
        a, b = out
        assert np.array_equal(a.ep_len, b.ep_len) and a.stats == b.stats, E
        assert np.array_equal(a.obs_array, b.obs_array) and np.array_equal(a.actions_array, b.actions_array), E
        assert np.array_equal(a.logits_array, b.logits_array) and np.array_equal(a.values_array, b.values_array), E
        assert np.array_equal(a.additional_array("rets"), b.additional_array("rets")), E


def test_native_safetensors_reader(eng, tmp_path):
    """twr_policy_create_from_safetensors: checkpoints of the reference's state dicts (BasicPolicy with the shipped trained
    weights, a deeper-stack BasicPolicy, a Conv1dPolicy) loaded natively give the same logits as the to_rust() route."""
    st = pytest.importorskip("safetensors.numpy")
    import twisterl_b200 as tw
    from helpers import synth_conv_state_dict, synth_deep_state_dict
    from parity import make_conv1d_policies, make_policies, make_policies_general
    from twisterl_b200.nn import forward_obs
    z, sd = trained15()
    obs = obs_from_states(z["states"][:64])
    twists = transpose_twists(4)
    cases = [("basic", sd, make_policies(sd, 256, *twists)[0], dict(obs_perms=twists[0], act_perms=twists[1]))]
    dsd = synth_deep_state_dict(5, 256, 512, (256, 128), (64,), (32,), 4)
    cases.append(("deep", dsd, make_policies_general(dsd, 256)[0], {}))
    csd = synth_conv_state_dict(6, 16, 32, 512, 256, 4)
    cases.append(("conv", csd, make_conv1d_policies(csd, [16, 16], 1)[0], dict(obs_shape=[16, 16], conv_dim=1)))
    for name, state, ref_pol, kw in cases:
        path = tmp_path / f"{name}.safetensors"
        st.save_file({k: np.ascontiguousarray(v, dtype=np.float32) for k, v in state.items()}, str(path), metadata={"format": "pt"})
        pol = tw.nn.Policy.from_safetensors(path, engine=eng, **kw)
        perm = (np.arange(len(obs)) % 2).astype(np.int32) if "obs_perms" in kw else None
        l, v = forward_obs(eng, pol, obs, perm)
        rl, rv = forward_obs(eng, ref_pol, obs, perm)
        assert np.array_equal(l, rl) and np.array_equal(v, rv), name
        pol.release()
    # a collect runs on the natively loaded policy like on any other
    path = tmp_path / "basic.safetensors"
    pol = tw.nn.Policy.from_safetensors(path, engine=eng)
    d = tw.collector.PPOCollector(64, 0.995, 0.995, 1, engine=eng).collect(tw.env.Puzzle(4, 4, 5, 2, 256), pol)
    assert len(d.values_array) >= 64
    bad = tmp_path / "bad.safetensors"
    bad.write_bytes(b"\\x10\\x00\\x00\\x00\\x00\\x00\\x00\\x00{not json at all}")
    with pytest.raises(RuntimeError, match="safetensors"):
        tw.nn.Policy.from_safetensors(bad, engine=eng)
    with pytest.raises(RuntimeError, match="cannot open"):
        tw.nn.Policy.from_safetensors(tmp_path / "missing.safetensors", engine=eng)


def test_collect_host_large_uses_round_sized_sub_batches(eng):
    """Above four kernel rounds twr_ppo_collect_host cuts the collect into two-round sub-batches (37 888 envs on a
    148-SM device) plus a halved tail; the host buffers must equal the plain collect + to_host path."""
    import ctypes as C
    import twisterl_b200 as tw
    from parity import make_policies
    from twisterl_b200 import _lib, collector as twc
    _, sd = trained15()
    pol, _ = make_policies(sd, 256)
    env = tw.env.Puzzle(4, 4, 3, 2, 256)
    E = 120000
    col = tw.collector.PPOCollector(E, 0.995, 0.995, 32, engine=eng)
    eng.set_collect_id(23)
    ref = col.collect(env, pol)
    L = _lib.load()
    spec = tw.env.spec_from_env(env)
    cap = int(L.twr_max_records(C.byref(spec), E))
    hb, arr, _ = twc._host_buffers(cap, 16, 4, E, pinned=True, obs_u8=True)
    out = _lib.Collected()
    eng.set_collect_id(23)
    _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), pol.device_handle(eng), None, E, 0.995, 0.995, C.byref(hb), C.byref(out)))
    R = int(out.n_records)
    assert R == len(ref.values_array) and int(out.successes) == ref.stats["successes"]
    assert np.array_equal(arr["ep_len"], ref.ep_len)
    assert np.array_equal(arr["obs"][:R], ref.obs_array.astype(np.uint8)) and np.array_equal(arr["actions"][:R], ref.actions_array)
    assert np.array_equal(arr["logits"][:R], ref.logits_array) and np.array_equal(arr["rets"][:R], ref.additional_array("rets"))


def test_two_engines_on_two_devices_in_one_process():
    """Launch state (SM count, cluster residency, tensor maps of the operand images) is kept per device: two engines on two
    GPUs of one process, used alternately, must each produce exactly what a lone engine produces."""
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import twisterl_b200 as tw
    from parity import check_collect_against_oracle, make_policies
    _, sd = trained15()
    ospec = orc.puzzle_spec(4, 4, 6, 2, 256)
    env = tw.env.Puzzle(4, 4, 6, 2, 256)
    engs = [tw.Engine(device=d, precision=PRECISION, seed=77) for d in (0, 1)]
    pols = [make_policies(sd, 256) for _ in engs]
    outs = []
    for rnd in range(2):                                             # alternate between the devices
        for eng, (pol, opol) in zip(engs, pols):
            eng.set_collect_id(5)
            d = tw.collector.PPOCollector(3000, 0.995, 0.995, 1, engine=eng).collect(env, pol)
            check_collect_against_oracle(d, ospec, opol, seed=77, collect_id=5, gamma=0.995, lam=0.995, tol=TOL, stride=37)
            outs.append(d)
    for d in outs[1:]:
        assert np.array_equal(d.obs_array, outs[0].obs_array) and np.array_equal(d.logits_array, outs[0].logits_array)
        assert np.array_equal(d.actions_array, outs[0].actions_array)
    for (pol, _), eng in zip(pols, engs):
        pol.release(); eng.close()


@pytest.mark.parametrize("E,H", [(256, 256), (768, 256), (1024, 128), (256, 128), (128, 256), (384, 256), (640, 128), (896, 128)])
def test_forward_and_collect_other_layer_widths(eng, E, H):
    """Embedding widths of 1 to 8 chunks of 128 features (an odd count runs zero-padded to the next chunk pair) and both
    common widths of the pair kernel (the shipped configs are all E = 512): forward against the oracle on scrambled states,
    and a collect replayed record by record."""
    import twisterl_b200 as tw
    from parity import check_collect_against_oracle, make_policies
    from twisterl_b200.env import EnvBatch
    from twisterl_b200.nn import forward_batch
    sd = synth_state_dict(13 + E + H, 256, E, H, 4)
    pol, opol = make_policies(sd, 256, *transpose_twists(4))
    st = scramble_states(np.random.default_rng(E), 300, 4, 4, 60)
    b = EnvBatch(_spec(orc.puzzle_spec(4, 4, 1, 2, 256)), len(st), eng)
    b.set_state(st)
    perm = np.arange(len(st)) % 3 - 1                               # -1 (no twist), 0, 1
    logits, values = forward_batch(eng, pol, b, perm_idx=perm)
    ref = [opol.raw_predict(o, int(p)) for o, p in zip(obs_from_states(st).tolist(), perm)]
    assert _close(logits, np.array([r[0] for r in ref]), TOL) and _close(values, np.array([r[1] for r in ref]), TOL)
    ospec = orc.puzzle_spec(4, 4, 10, 2, 256)
    eng.set_collect_id(3)
    d = tw.collector.PPOCollector(700, 0.995, 0.995, 1, engine=eng).collect(tw.env.Puzzle(4, 4, 10, 2, 256), pol)
    rep = check_collect_against_oracle(d, ospec, opol, seed=eng.seed, collect_id=3, gamma=0.995, lam=0.995, tol=TOL, stride=7)
    assert rep["records"] > 500
