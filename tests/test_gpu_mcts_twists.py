"""GPU parity of MCTS with a twisted policy: the searches evaluate every leaf with Policy::full_predict (rl/search.rs:113,150;
nn/policy.rs:102-126), the average over all twists, on both device paths (the persistent whole-search kernel and the lockstep
kernels) and through evaluate / solve, against the oracle's restatement on the shared Philox streams."""
import ctypes as C

import numpy as np
import pytest

from suite_loader import suite_precision

from helpers import gridworld_transpose_twists, scramble_states, synth_state_dict, trained15, transpose_twists
from oracle import orc

pytestmark = pytest.mark.gpu
PRECISION = suite_precision(globals())

# first-divergence near-tie rule of test_gpu_az.py / test_gpu_eval.py, and the per-precision bar of one leaf evaluation
NEAR_TIE = {"fp32": 2e-4, "f16x2": 2e-3, "f16x2w16": 2e-2, "f16f8c": 2e-2}[PRECISION]
LEAF_BAR = {"fp32": 1e-5, "f16x2": 1e-4, "f16x2w16": 1e-3, "f16f8c": 1e-3}[PRECISION]
P15 = (0, 4, 4, 5, 2, 256)
G5 = (1, 5, 5, 6, 0, 64)


@pytest.fixture(scope="module")
def eng():
    import twisterl_b200 as tw
    tw.configure(device=0, precision=PRECISION, seed=0x7A157)
    return tw.default_engine()


def _identity_twists(obs_size):
    ident = list(range(obs_size))
    return [ident, ident], [[0, 1, 2, 3], [0, 1, 2, 3]]


def _batch(eng, spec, states=None, reset=None):
    from twisterl_b200 import _lib
    from twisterl_b200.env import EnvBatch
    n = len(states) if states is not None else reset[1]
    b = EnvBatch(_lib.EnvSpec(*spec), n, eng)
    if states is not None:
        b.set_state(states)
    else:
        b.reset(env_id_base=reset[0], collect_id=reset[2])
    return b


def _oracle_env(spec, state):
    kind, w, h, diff, slope, md = spec
    env = orc.Env(orc.puzzle_spec(w, h, diff, slope, md) if kind == 0 else orc.gridworld_spec(w, h, md, diff))
    env.set_state([int(x) for x in state])
    return env


def _mcts(eng, pol, batch, n_sims, c, med, base, cid, t):
    """(probs [n][A], visits [n][A], trace [n_sims][n][2]) of twr_debug_mcts_trace."""
    from twisterl_b200 import _lib
    n = batch.n
    probs = np.zeros((n, 4), np.float32); visits = np.zeros((n, 4), np.int32)
    trace = np.zeros((max(n_sims, 1), n, 2), np.int32)
    _lib.check(_lib.load().twr_debug_mcts_trace(eng._h, pol.device_handle(eng), batch._h, n_sims, c, med, base, cid, t,
                                                _lib.ptr(probs), _lib.ptr(visits), _lib.ptr(trace)))
    return probs, visits, trace[:n_sims]


def _check_searches(eng, pol, opol, spec, states, n_sims, med, base, cid, t):
    """Every search reproduces the oracle's visit counts, or parts from it first where the oracle met a near-tie."""
    b = _batch(eng, spec, states)
    probs, visits, trace = _mcts(eng, pol, b, n_sims, 1.41, med, base, cid, t)
    same = 0
    for i, st in enumerate(states):
        env = _oracle_env(spec, st)
        op, ov = orc.mcts_probs(env, opol, n_sims, 1.41, med, seed=eng.seed, collect_id=cid, stream_id=base + i, t=t)
        assert visits[i].sum() == ov.sum()
        if np.array_equal(visits[i], ov):
            same += 1
            assert np.allclose(probs[i], op, atol=1e-6)
            continue
        _, _, leaf, child, margin = orc.mcts_trace(env, opol, n_sims, 1.41, med, seed=eng.seed, collect_id=cid,
                                                   stream_id=base + i, t=t)
        div = next((s for s in range(n_sims) if trace[s, i, 0] != leaf[s] or trace[s, i, 1] != child[s]), None)
        assert div is not None, f"env {i}: visit counts differ but every simulation took the oracle's path"
        assert margin[div] < NEAR_TIE, f"env {i}: first divergence at simulation {div} where the oracle's margin was {margin[div]}"
    print(f"[twisted mcts n_sims={n_sims} med={med}] identical {same}/{len(states)}")
    assert same >= len(states) // 2


def _puzzle15_states(seed, n):
    return scramble_states(np.random.default_rng(seed), n, 4, 4, 12)


def _gridworld_states(eng, n, base, cid):
    return _batch(eng, G5, reset=(base, n, cid)).get_state()


# ---------------------------------------------------------------------------------------------- leaf evaluation ---
@pytest.mark.parametrize("which", ["puzzle15", "gridworld5"])
def test_full_predict_matches_oracle(eng, which):
    from parity import make_policies
    from twisterl_b200.nn import forward_batch, full_predict_batch
    if which == "puzzle15":
        sd, obs_size, twists, spec = trained15()[1], 256, transpose_twists(4), P15
        states = _puzzle15_states(5, 512)
    else:
        sd, obs_size, twists, spec = synth_state_dict(6, 625, 512, 128, 4), 625, gridworld_transpose_twists(5), G5
        states = _gridworld_states(eng, 512, 40, 2)
    pol, opol = make_policies(sd, obs_size, *twists)
    probs, values = full_predict_batch(eng, pol, _batch(eng, spec, states))
    worst_p = worst_v = 0.0
    for i, st in enumerate(states):
        env = _oracle_env(spec, st)
        op, ov = opol.full_predict(env.observe(), env.masks())
        worst_p = max(worst_p, float(np.abs(probs[i] - op).max()))
        worst_v = max(worst_v, abs(float(values[i]) - float(ov)) / max(1.0, abs(float(ov))))
    print(f"[full_predict {which}] max |dprob| {worst_p:.2e}, max value error {worst_v:.2e}")
    assert worst_p <= LEAF_BAR and worst_v <= LEAF_BAR
    # without twists full_predict is predict: the forward's own value, the masked exp / (sum + 1e-6) of its logits
    plain, _ = make_policies(sd, obs_size)
    b = _batch(eng, spec, states)
    p0, v0 = full_predict_batch(eng, plain, b)
    logits, values = forward_batch(eng, plain, b)
    assert np.array_equal(v0, values)
    masks = b.masks().astype(bool)
    e = np.where(masks, np.exp(logits), np.float32(0)).astype(np.float32)
    assert np.allclose(p0, e / (e.sum(axis=1, keepdims=True, dtype=np.float32) + np.float32(1e-6)), rtol=1e-6, atol=1e-7)


# ------------------------------------------------------------------------------------------ identity twist set ---
@pytest.mark.parametrize("lockstep", [False, True])
def test_identity_twists_reproduce_the_untwisted_search_bit_for_bit(eng, monkeypatch, lockstep):
    """{identity, identity}: raw/2 + raw/2 == raw exactly, so the averaged leaf evaluation and every search decision equal
    the untwisted policy's."""
    from parity import make_policies
    from twisterl_b200.nn import full_predict_batch
    if lockstep:
        monkeypatch.setenv("TWISTERL_B200_MCTS_LOCKSTEP", "1")
    for sd, obs_size, spec, states in ((trained15()[1], 256, P15, _puzzle15_states(9, 96)),
                                       (synth_state_dict(6, 625, 512, 128, 4), 625, G5, _gridworld_states(eng, 64, 900, 4))):
        plain, _ = make_policies(sd, obs_size)
        twin, _ = make_policies(sd, obs_size, *_identity_twists(obs_size))
        b = _batch(eng, spec, states)
        pa, va = full_predict_batch(eng, plain, b)
        pb, vb = full_predict_batch(eng, twin, b)
        assert np.array_equal(pa, pb) and np.array_equal(va, vb)
        for sims, med in ((40, 1), (24, 2)):
            ra = _mcts(eng, plain, b, sims, 1.41, med, 300, 6, 1)
            rb = _mcts(eng, twin, b, sims, 1.41, med, 300, 6, 1)
            for x, y in zip(ra, rb):
                assert np.array_equal(x, y)


# -------------------------------------------------------------------------------------- searches vs the oracle ---
@pytest.mark.parametrize("n_sims,med,lockstep", [(24, 1, False), (24, 1, True), (200, 1, False), (200, 1, True), (40, 2, True)])
def test_twisted_mcts_matches_oracle_puzzle15(eng, monkeypatch, n_sims, med, lockstep):
    from parity import make_policies
    if lockstep:
        monkeypatch.setenv("TWISTERL_B200_MCTS_LOCKSTEP", "1")
    pol, opol = make_policies(trained15()[1], 256, *transpose_twists(4))
    _check_searches(eng, pol, opol, P15, _puzzle15_states(n_sims + med, 96), n_sims, med, 500, 3, 2)


@pytest.mark.parametrize("lockstep", [False, True])
def test_twisted_mcts_matches_oracle_gridworld(eng, monkeypatch, lockstep):
    from parity import make_policies
    if lockstep:
        monkeypatch.setenv("TWISTERL_B200_MCTS_LOCKSTEP", "1")
    pol, opol = make_policies(synth_state_dict(6, 625, 512, 128, 4), 625, *gridworld_transpose_twists(5))
    _check_searches(eng, pol, opol, G5, _gridworld_states(eng, 64, 900, 4), 60, 1, 900, 4, 0)


# ------------------------------------------------------------------------------------------------ path choice ---
def test_small_twisted_batch_runs_one_persistent_launch_and_many_twists_fall_back(eng):
    from parity import make_policies
    from twisterl_b200 import _lib
    sd = trained15()[1]
    states = _puzzle15_states(21, 64)
    b = _batch(eng, P15, states)
    probs = np.zeros((64, 4), np.float32); visits = np.zeros((64, 4), np.int32)

    def launches(pol, sims):
        h = pol.device_handle(eng)                    # creating the device policy launches its operand packing
        n0 = eng.launch_count()
        _lib.check(_lib.load().twr_mcts_probs(eng._h, h, b._h, sims, 1.41, 1, 500, 3, 2,
                                              _lib.ptr(probs), _lib.ptr(visits)))
        return eng.launch_count() - n0

    pol, _ = make_policies(sd, 256, *transpose_twists(4))
    assert launches(pol, 50) == 2                     # the whole search, then the root read-out
    # six twists leave less than one tree per CTA of the persistent kernel: the lockstep path (T forwards per simulation)
    ob, ac = transpose_twists(4)
    many, omany = make_policies(sd, 256, ob * 3, ac * 3)
    assert launches(many, 50) > 50 * 6
    _check_searches(eng, many, omany, P15, states, 50, 1, 500, 3, 2)


# ---------------------------------------------------------------------------------------- evaluate and solve ---
def _check_episodes(bs, bt, obs_, obt, margins, what):
    """per-episode best (success, reward): equal to the oracle's, or the oracle met a near-tie in that episode"""
    diff = [i for i in range(len(bs)) if bs[i] != obs_[i] or abs(float(bt[i]) - float(obt[i])) > 1e-5]
    for i in diff:
        assert margins[i] < NEAR_TIE, f"{what}: episode {i} differs ({bs[i]}, {bt[i]}) vs ({obs_[i]}, {obt[i]}) with smallest margin {margins[i]}"
    print(f"[{what}] {len(bs) - len(diff)}/{len(bs)} episodes identical, {len(diff)} explained by near-ties")
    assert len(diff) <= len(bs) // 4


@pytest.mark.parametrize("det,searches,sims", [(True, 1, 24), (False, 2, 10)])
def test_evaluate_with_mcts_on_twisted_policy_matches_oracle(eng, det, searches, sims):
    import twisterl_b200 as tw
    from parity import make_policies
    from twisterl_b200 import _lib
    pol, opol = make_policies(synth_state_dict(8, 81, 512, 256, 4), 81, *transpose_twists(3))
    env = tw.env.Puzzle(3, 3, 4, 2, 256)
    n = 96
    spec = tw.env.spec_from_env(env)
    s, r = C.c_float(), C.c_float()
    bs, bt = np.zeros(n, np.float32), np.zeros(n, np.float32)
    eng.set_collect_id(13)
    _lib.check(_lib.load().twr_evaluate_episodes(eng._h, C.byref(spec), pol.device_handle(eng), n, int(det), searches, sims, 1.41,
                                                 1, C.byref(s), C.byref(r), _lib.ptr(bs), _lib.ptr(bt)))
    obs_, obt, mm = orc.evaluate_margins(orc.puzzle_spec(3, 3, 4, 2, 256), opol, n, det, searches, seed=eng.seed, collect_id=13,
                                         num_mcts_searches=sims, c_puct=1.41, max_expand_depth=1)
    _check_episodes(bs, bt, obs_, obt, mm, f"twisted evaluate+mcts det={det} searches={searches} sims={sims}")
    assert abs(s.value - float(bs.mean())) < 1e-6


def test_collector_evaluate_and_solve_with_mcts_on_add_perms_puzzle(eng):
    """The user path: a policy built with Puzzle(..., add_perms=True).twists(), evaluated and solved with MCTS through
    the collector module."""
    import twisterl_b200 as tw
    from parity import make_policies
    _, sd = trained15()
    env = tw.env.Puzzle(4, 4, 6, 2, 256, add_perms=True)
    obs_perms, act_perms = env.twists()
    assert len(obs_perms) == 2
    pol, opol = make_policies(sd, 256, obs_perms, act_perms)
    n = 64
    eng.set_collect_id(21)
    s, r = tw.collector.evaluate(env, pol, n, True, 1, 16, 0, 1.41, 1, 1)
    obs_, obt, mm = orc.evaluate_margins(orc.puzzle_spec(4, 4, 6, 2, 256), opol, n, True, 1, seed=eng.seed, collect_id=21,
                                         num_mcts_searches=16, c_puct=1.41, max_expand_depth=1)
    if not (abs(s - float(np.mean(obs_))) < 1e-6 and abs(r - float(np.mean(obt))) < 1e-4):
        assert float(np.min(mm)) < NEAR_TIE, (s, r, float(np.mean(obs_)), float(np.mean(obt)))
    assert s >= 0.9                                   # the trained policy solves shallow scrambles
    start = [1, 5, 2, 3, 4, 0, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15]         # two moves from solved
    env.set_state(start)
    eng.set_collect_id(22)
    (succ, rew), acts = tw.collector.solve(env, pol, True, 1, 16, 1.41, 1)
    oenv = orc.Env(orc.puzzle_spec(4, 4, 6, 2, 256)); oenv.set_state(start)
    (os_, or_), oacts = orc.solve(oenv, opol, True, 1, seed=eng.seed, collect_id=22, id0=0x50000000, num_mcts_searches=16,
                                  c_puct=1.41, max_expand_depth=1)       # twr_solve's search streams
    assert succ == 1.0 and os_ == 1.0
    assert acts == oacts and abs(rew - or_) < 1e-6
