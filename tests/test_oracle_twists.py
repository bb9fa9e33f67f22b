"""Pins the oracle's Policy::full_predict (nn/policy.rs:102-126), which the MCTS searches of twisted policies evaluate at
every leaf (rl/search.rs:113,150): a numpy float32 restatement of the average, and the identity twist set as a no-op."""
import numpy as np

from helpers import scramble_states, synth_state_dict, trained15, transpose_twists
from oracle import orc


def _identity_twists(obs_size, n_actions):
    ident = list(range(obs_size))
    return [ident, ident], [list(range(n_actions))] * 2


def _masked_exp_normalise(acc, masks):
    e = np.where(np.asarray(masks, bool), np.exp(acc.astype(np.float32)), np.float32(0)).astype(np.float32)
    s = np.float32(0)
    for x in e:                                       # the oracle's sum, in action order
        s = np.float32(s + x)
    return (e / np.float32(s + np.float32(1e-6))).astype(np.float32)


def test_full_predict_matches_numpy_restatement():
    _, sd = trained15()
    obs_perms, act_perms = transpose_twists(4)
    p = orc.Policy.from_torch_state_dict(sd, obs_perms, act_perms)
    W = {k: np.asarray(v, np.float32) for k, v in sd.items()}
    rng = np.random.default_rng(11)
    env = orc.Env(orc.puzzle_spec(4, 4, 5, 2, 256))
    np_ = np.float32(len(obs_perms))
    for state in scramble_states(rng, 48, 4, 4, 14):
        env.set_state(state.tolist())
        obs, masks = env.observe(), env.masks()
        acc, val = np.zeros(4, np.float32), np.float32(0)
        for pi in range(len(obs_perms)):
            raw, v = p.raw_predict(obs, pi)
            # _raw_predict: observation indices through obs_perms[pi], heads through act_perms[pi]
            rows = [obs_perms[pi][i] for i in obs]
            h1 = np.maximum(W["embeddings.bias"] + W["embeddings.weight"][:, rows].sum(axis=1, dtype=np.float64), 0)
            h2 = np.maximum(W["common.0.weight"].astype(np.float64) @ h1 + W["common.0.bias"], 0)
            head = W["action.0.weight"].astype(np.float64) @ h2 + W["action.0.bias"]
            want = np.array([head[act_perms[pi][i]] for i in range(4)])
            assert np.allclose(raw, want, rtol=1e-5, atol=1e-5)
            assert abs(float(v) - float(W["value.0.weight"][0] @ h2 + W["value.0.bias"][0])) < 1e-5
            # the contract: each term divided by n_perms, then added, in twist order (f32)
            acc = (acc + (raw / np_).astype(np.float32)).astype(np.float32)
            val = np.float32(val + np.float32(v / np_))
        probs, value = p.full_predict(obs, masks)
        assert value == val
        assert np.allclose(probs, _masked_exp_normalise(acc, masks), rtol=2e-7, atol=1e-8)


def test_identity_twists_are_exact_noop_for_full_predict_and_search():
    """{identity, identity}: raw/2 + raw/2 == raw exactly, so full_predict and both MCTS entry points reproduce the
    untwisted policy bit for bit."""
    for spec, sd, obs_size in ((orc.puzzle_spec(4, 4, 6, 2, 256), trained15()[1], 256),
                               (orc.gridworld_spec(5, 5, 64, 6), synth_state_dict(6, 625, 64, 32, 4), 625)):
        plain = orc.Policy.from_torch_state_dict(sd)
        twin = orc.Policy.from_torch_state_dict(sd, *_identity_twists(obs_size, 4))
        for i in range(12):
            env = orc.Env(spec); env.reset(seed=3, env_id=i, collect_id=1)
            a = plain.full_predict(env.observe(), env.masks())
            b = twin.full_predict(env.observe(), env.masks())
            assert np.array_equal(a[0], b[0]) and a[1] == b[1]
            for sims, med in ((24, 1), (16, 2)):
                pa, va = orc.mcts_probs(env, plain, sims, 1.41, med, seed=3, stream_id=i)
                pb, vb = orc.mcts_probs(env, twin, sims, 1.41, med, seed=3, stream_id=i)
                assert np.array_equal(va, vb) and np.array_equal(pa, pb)
                ta = orc.mcts_trace(env, plain, sims, 1.41, med, seed=3, stream_id=i)
                tb = orc.mcts_trace(env, twin, sims, 1.41, med, seed=3, stream_id=i)
                for x, y in zip(ta, tb):
                    assert np.array_equal(x, y)
