"""Puzzle boards of 17..25 cells (the 24-puzzle among them) without a device: the oracle against a plain Python model of
envs/puzzle.rs on every wide board shape, the 5x5 transpose twist set as a symmetry of the env, and the C ABI's spec
validation at the 25-cell limit of the 5-bit device state."""
import ctypes as C

import numpy as np
import pytest

from oracle import orc

BOARDS = [(3, 6), (6, 3), (4, 5), (5, 4), (4, 6), (5, 5)]
SEED = 0x1234_5678_9ABC


def _step(s, z, w, h, a):
    """puzzle.rs:135-160 on a list board: blank moves 0 left, 1 up, 2 right, 3 down; an illegal move is a no-op."""
    x, y = z % w, z // w
    t = {0: z - 1 if x > 0 else -1, 1: z - w if y > 0 else -1, 2: z + 1 if x < w - 1 else -1,
         3: z + w if y < h - 1 else -1}[a]
    if t >= 0:
        s[z], s[t], z = s[t], 0, t
    return z


def _reset_model(w, h, difficulty, seed, env_id, cid):
    """puzzle.rs:119-133 with the shared stream: draw j is the 2-bit field j % 16 of stream word j / 16."""
    s, z = list(range(w * h)), 0
    for j in range(difficulty):
        k = j // 16
        word = int(orc.philox([env_id, k // 4, orc.RNG_RESET, cid], [seed & 0xFFFFFFFF, seed >> 32])[k % 4])
        z = _step(s, z, w, h, (word >> (2 * (j % 16))) & 3)
    return s, z


@pytest.mark.parametrize("w,h", BOARDS, ids=lambda v: str(v))
def test_oracle_reset_reachability_and_budget(w, h):
    for difficulty in (0, 1, 17, 64, 200):
        env = orc.Env(orc.puzzle_spec(w, h, difficulty, 2, 256))
        for env_id in range(24):
            env.reset(seed=SEED, env_id=env_id, collect_id=5)
            s, z = _reset_model(w, h, difficulty, SEED, env_id, 5)
            st = env.get_state()
            assert st == s and sorted(st) == list(range(w * h))
            assert env.zero_location == (z % w, z // w)
            assert env.depth == 2 * difficulty
            assert env.observe() == [i * w * h + v for i, v in enumerate(s)]


@pytest.mark.parametrize("w,h", BOARDS, ids=lambda v: str(v))
def test_oracle_forced_actions_illegal_no_ops_and_depth_saturation(w, h):
    N, rng = w * h, np.random.default_rng(w * 10 + h)
    depth = 30
    env = orc.Env(orc.puzzle_spec(w, h, 3, 10, depth))
    env.reset(seed=SEED, env_id=7, collect_id=1)
    env.set_state(list(range(N)))                 # set_state: depth = max_depth, blank = first zero (puzzle.rs:107-117)
    s, z, d = list(range(N)), 0, depth
    assert env.success() and env.is_final() and env.reward() == 1.0
    illegal = 0
    for t in range(60):                           # past the budget: depth saturates at 0
        a = int(rng.integers(0, 4))
        before = list(s)
        x, y = z % w, z // w
        legal = [x > 0, y > 0, x < w - 1, y < h - 1]
        assert env.masks() == legal
        z = _step(s, z, w, h, a)
        illegal += s == before and not legal[a]
        d = max(0, d - 1)
        env.step(a)
        assert env.get_state() == s and env.depth == d and env.zero_location == (z % w, z // w)
        solved = s == list(range(N))
        assert env.success() == solved and env.is_final() == (solved or d == 0)
        want = 1.0 if solved else (-0.5 if d == 0 else np.float32(-0.5) / np.float32(depth))
        assert np.float32(env.reward()) == np.float32(want)
    assert illegal > 0 and d == 0


def test_puzzle_5x5_obs_shape_and_transpose_twists_are_a_symmetry():
    """Puzzle(5, 5, add_perms=True).twists(): {identity, transpose}; for the transpose T with action map A,
    twist(observe(step(s, a))) == observe(step(twist(s), A(a))) and the solved board is a fixed point."""
    import twisterl_b200 as tw
    from helpers import transpose_twists
    p = tw.env.Puzzle(5, 5, 3, 2, 256, add_perms=True)
    assert p.obs_shape() == [25, 25] and p.num_actions() == 4
    assert tw.env.Puzzle(5, 5, 3, 2, 256).twists() == ([], [])
    assert tw.env.Puzzle(4, 5, 3, 2, 256, add_perms=True).twists() == ([], [])     # not square: no transpose
    obs_perms, act_perms = p.twists()
    assert (obs_perms, act_perms) == transpose_twists(5)
    op, ap = obs_perms[1], act_perms[1]
    N, T = 25, [(i % 5) * 5 + i // 5 for i in range(25)]
    rng = np.random.default_rng(25)
    a_env, b_env = orc.Env(orc.puzzle_spec(5, 5, 3, 2, 256)), orc.Env(orc.puzzle_spec(5, 5, 3, 2, 256))
    for k in range(40):
        a_env.reset(seed=SEED, env_id=k, collect_id=2)
        s = a_env.get_state()
        twisted = [0] * N
        for i, v in enumerate(s):
            twisted[T[i]] = T[v]
        b_env.set_state(twisted)
        assert sorted(op[o] for o in a_env.observe()) == sorted(b_env.observe())
        for a in rng.integers(0, 4, size=12):
            a_env.step(int(a)); b_env.step(ap[int(a)])
            assert sorted(op[o] for o in a_env.observe()) == sorted(b_env.observe())
            assert a_env.success() == b_env.success()
    assert sorted(op[i * N + i] for i in range(N)) == [i * N + i for i in range(N)]   # the solved board is a fixed point


def test_max_records_at_the_16_and_25_cell_limits():
    """twr_max_records validates the spec as twr_envs_create does: TWR_ENV_PUZZLE_WIDE takes Puzzle boards of up to 25
    cells and refuses 26 with a message naming that limit; TWR_ENV_PUZZLE keeps its 16-cell limit and names the wide
    kind; Puzzle(w, h) and the C++ helper pick the kind from the board size."""
    import twisterl_b200 as tw
    from twisterl_b200 import _lib
    L = _lib.load()
    for w, h in BOARDS + [(1, 25), (25, 1), (4, 4)]:
        wide = _lib.EnvSpec(_lib.ENV_PUZZLE_WIDE, w, h, 64, 2, 256)
        assert L.twr_max_records(C.byref(wide), 100) == 100 * 129, (w, h)
    for kind, w, h, msg in ((_lib.ENV_PUZZLE_WIDE, 2, 13, b"25 cells"), (_lib.ENV_PUZZLE_WIDE, 6, 5, b"25 cells"),
                            (_lib.ENV_PUZZLE, 5, 5, b"TWR_ENV_PUZZLE_WIDE"), (_lib.ENV_PUZZLE, 3, 6, b"16 cells")):
        assert L.twr_max_records(C.byref(_lib.EnvSpec(kind, w, h, 1, 1, 1)), 1) == -1
        assert msg in L.twr_last_error(), (kind, w, h)
    for w, h in BOARDS:
        assert tw.env.spec_from_env(tw.env.Puzzle(w, h, 3, 2, 64)).kind == _lib.ENV_PUZZLE_WIDE
    assert tw.env.spec_from_env(tw.env.Puzzle(4, 4, 3, 2, 64)).kind == _lib.ENV_PUZZLE
