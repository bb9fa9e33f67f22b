"""Pins the oracle's AlphaZero path (rust/src/rl/search.rs, tree.rs, collector/az.rs restated in
oracle/twr_oracle.c) through properties the reference code guarantees."""
import numpy as np

from helpers import synth_state_dict, trained15
from oracle import orc


def test_mcts_probs_properties():                     # rl/search.rs:104-189
    _, sd = trained15()
    p = orc.Policy.from_torch_state_dict(sd)
    spec = orc.puzzle_spec(4, 4, 6, 2, 256)
    env = orc.Env(spec)
    env.set_state([1, 0, 2, 3] + list(range(4, 16)))   # blank in the top row: action 1 (up) is illegal
    probs, visits = orc.mcts_probs(env, p, 64, 1.41, 1, seed=1)
    # one backup per simulation passes through exactly one root child; masked actions get no child
    assert visits.sum() == 64 and visits[1] == 0
    assert np.allclose(probs, visits / 64.0) and abs(probs.sum() - 1.0) < 1e-6
    assert probs.argmax() == 0                         # the solving move (blank left) dominates
    # zero simulations: no visits -> uniform (search.rs:183-186)
    p0, v0 = orc.mcts_probs(env, p, 0, 1.41, 1)
    assert v0.sum() == 0 and np.allclose(p0, 0.25)
    # max_expand_depth 0: value 0 is backed up from the selected root child, visits still add up
    p1, v1 = orc.mcts_probs(env, p, 10, 1.41, 0)
    assert v1.sum() == 10
    # deterministic given the stream, different streams differ somewhere in general
    a = orc.mcts_probs(env, p, 200, 1.41, 2, seed=5, stream_id=3)[1]
    b = orc.mcts_probs(env, p, 200, 1.41, 2, seed=5, stream_id=3)[1]
    assert (a == b).all() and a.sum() == 200


def test_az_collect_structure():                      # collector/az.rs:51-130
    sd = synth_state_dict(4, 81, 64, 32, 4)
    p = orc.Policy.from_torch_state_dict(sd)
    spec = orc.puzzle_spec(3, 3, 3, 2, 256)
    d = orc.az_collect(spec, p, 9, 12, 1.41, 1, seed=2, collect_id=1)
    assert d["n_records"] == d["ep_len"].sum() == len(d["remaining_values"])
    assert np.allclose(d["probs"].sum(axis=1), 1.0, atol=1e-6)
    order = orc.merge_order(9)
    off = 0
    for ep in order:
        n = int(d["ep_len"][ep])
        env = orc.Env(spec); env.reset(seed=2, env_id=int(ep), collect_id=1)
        tot = np.float32(0); prefix = []
        for t in range(n):
            assert env.observe() == d["obs"][off + t].tolist()
            assert np.float32(env.reward()) == d["rewards"][off + t]
            assert env.is_final() == (t == n - 1)        # terminal state recorded (az.rs:84-86)
            prefix.append(tot); tot = np.float32(tot + d["rewards"][off + t])
            masks = env.masks()
            assert all(d["probs"][off + t][a] == 0 for a in range(4) if not masks[a])
            env.step(int(d["actions"][off + t]))
        want = np.array([np.float32(tot - q) for q in prefix], dtype=np.float32)   # az.rs:93
        assert np.array_equal(want, d["remaining_values"][off:off + n])
        off += n


def test_solve_with_mcts_searches():
    """rl/solve.rs:37-48 with num_mcts_searches > 0: the per-step distribution is the MCTS visit distribution."""
    from helpers import trained15
    _, sd = trained15()
    pol = orc.Policy.from_torch_state_dict(sd)
    env = orc.Env(orc.puzzle_spec(4, 4, 1, 2, 256))
    start = [1, 5, 2, 3, 4, 0, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15]
    env.set_state(start)
    (s, r), acts = orc.solve(env, pol, True, 1, seed=3, num_mcts_searches=16)
    assert s == 1.0 and len(acts) >= 2
    for a in acts:
        env.step(a)
    assert env.success()
    # evaluation of a scrambled batch: MCTS guidance never lowers the success rate of this trained policy
    spec = orc.puzzle_spec(4, 4, 3, 2, 256)
    s0, _, _, _ = orc.evaluate(spec, pol, 24, True, 1, seed=5)
    s1, _, _, _ = orc.evaluate(spec, pol, 24, True, 1, seed=5, num_mcts_searches=12)
    assert s1 >= s0 - 1e-6


def test_trace_and_margin_instrumentation_leave_results_unchanged():
    """orc_mcts_trace / orc_evaluate_margins (used by the GPU near-tie rule) return exactly what the plain calls return;
    the trace is consistent with the search (each simulation backs up from the leaf or one of its new children)."""
    from helpers import synth_state_dict
    pol = orc.Policy.from_torch_state_dict(synth_state_dict(8, 81, 512, 256, 4))
    env = orc.Env(orc.puzzle_spec(3, 3, 4, 2, 256)); env.reset(seed=3, env_id=5, collect_id=1)
    for sims, med in ((20, 1), (12, 2), (8, 0)):
        p0, v0 = orc.mcts_probs(env, pol, sims, 1.41, med, seed=3, collect_id=1, stream_id=5, t=0)
        p1, v1, leaf, child, margin = orc.mcts_trace(env, pol, sims, 1.41, med, seed=3, collect_id=1, stream_id=5, t=0)
        assert np.array_equal(p0, p1) and np.array_equal(v0, v1)
        assert len(leaf) == sims and (margin >= 0).all()
        assert leaf[0] in (1, 2, 3, 4) and all(c >= l for l, c in zip(leaf, child))      # children are allocated after their parent
        if med == 0:
            assert np.array_equal(leaf, child)
    spec = orc.puzzle_spec(3, 3, 4, 2, 256)
    for det, mcts in ((True, 0), (False, 0), (False, 6)):
        s, r, bs, bt = orc.evaluate(spec, pol, 12, det, 2, seed=9, collect_id=2, num_mcts_searches=mcts)
        bs2, bt2, mm = orc.evaluate_margins(spec, pol, 12, det, 2, seed=9, collect_id=2, num_mcts_searches=mcts)
        assert np.array_equal(bs, bs2) and np.array_equal(bt, bt2)
        assert (mm >= 0).all() and np.isfinite(mm).any()


def test_trace_reports_backup_path_lengths_of_a_known_chain():
    """A policy whose logits are its action biases alone (all weights zero): the prior is one-hot, up to e^-20, on the
    first legal move in the order left, up, right, down, and the value is 0.  Every simulation then descends the one chain
    to its end, expands it and backs up from the new child, so simulation s updates s + 3 nodes (root, s + 1 chain nodes,
    the child) until the chain meets the depth-budget terminal at depth D, whose backups update D + 1 nodes."""
    D, E, H = 120, 16, 16
    sd = synth_state_dict(1, 256, E, H, 4)
    sd = {k: np.zeros_like(v) for k, v in sd.items()}
    sd["action.0.bias"] = np.array([60.0, 40.0, 20.0, 0.0], np.float32)
    pol = orc.Policy.from_torch_state_dict(sd)
    spec = orc.puzzle_spec(4, 4, 5, 2, D)               # set_state gives the board D moves
    start = list(range(1, 16)) + [0]                     # blank bottom right: left x3, up x3, then right / left forever
    env = orc.Env(spec); env.set_state(start)
    chain = []
    for _ in range(D):
        m = env.masks()
        chain.append(next(a for a in range(4) if m[a]))
        env.step(chain[-1])
        assert not env.success()
    assert chain[:8] == [0, 0, 0, 1, 1, 1, 2, 0] and env.is_final()
    env = orc.Env(spec); env.set_state(start)
    probs, visits, leaf, child, margin, plen = orc.mcts_trace(env, pol, D + 4, 1.41, 1, seed=3, collect_id=1, stream_id=5,
                                                              path_lengths=True)
    assert all(np.array_equal(x, y) for x, y in zip((probs, visits, leaf, child, margin),
                                                     orc.mcts_trace(env, pol, D + 4, 1.41, 1, seed=3, collect_id=1, stream_id=5)))
    assert plen.tolist()[:D] == list(range(3, D + 2)) + [D + 1]
    assert leaf[D - 1] == child[D - 1]                  # the terminal leaf backs up its own reward
    assert visits.tolist() == [D + 4, 0, 0, 0]          # blank bottom right: left (0) and up (1) are the legal moves
    assert plen.max() == D + 1 > 96                     # deeper than the device's recorded descent path (TWR_MCTS_PATH)
