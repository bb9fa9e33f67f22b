"""GridWorld boards of 33..64 cells (6x6, 7x7, 8x8, 4x16, 6x10, 1x64) without a device: the oracle against a plain
Python model of examples/grid_world/src/lib.rs on every such board, the 8x8 transpose twists as a symmetry of the env,
and the C ABI's spec validation at the 64-cell limit."""
import ctypes as C

import numpy as np
import pytest

from oracle import orc

BOARDS = [(6, 6), (7, 7), (8, 8), (4, 16), (6, 10), (1, 64)]
SEED = 0x6464_6464_6464


def _draw(seed, env_id, cid, k):
    """word k of the reset stream: philox(env_id, k / 4, RNG_RESET, cid)[k % 4]"""
    return int(orc.philox([env_id, k // 4, orc.RNG_RESET, cid], [seed & 0xFFFFFFFF, seed >> 32])[k % 4])


def _mulhi(w, n):
    return (w * n) >> 32


def _reset_model(w, h, difficulty, seed, env_id, cid):
    """lib.rs:114-125: agent uniform; goal uniform among the cells within Manhattan `difficulty` of it, candidates listed
    x-outer / y-inner (random_pos_near, lib.rs:50-65), redrawn while it is the agent cell; trap uniform, redrawn while it
    is the agent or the goal cell.  Returns (agent, goal, trap) as (x, y)."""
    k, n = 0, w * h

    def draw():
        nonlocal k
        k += 1
        return _draw(seed, env_id, cid, k - 1)

    a = _mulhi(draw(), n)
    ax, ay = a % w, a // w
    cand = [(x, y) for x in range(w) for y in range(h) if abs(x - ax) + abs(y - ay) <= difficulty]
    while True:
        g = cand[_mulhi(draw(), len(cand))]
        if g != (ax, ay):
            break
    while True:
        t = _mulhi(draw(), n)
        if (t % w, t // w) not in ((ax, ay), g):
            break
    return (ax, ay), g, (t % w, t // w)


def _board(w, h, agent, goal, trap):
    """lib.rs:74-81: goal 2, trap 3, agent 1 written last"""
    b = [0] * (w * h)
    b[goal[1] * w + goal[0]] = 2
    b[trap[1] * w + trap[0]] = 3
    b[agent[1] * w + agent[0]] = 1
    return b


def _step(w, h, agent, a):
    """lib.rs:127-136: 0 up, 1 down, 2 left, 3 right; a move off the board is a no-op"""
    x, y = agent
    if a == 0 and y > 0: y -= 1
    elif a == 1 and y + 1 < h: y += 1
    elif a == 2 and x > 0: x -= 1
    elif a == 3 and x + 1 < w: x += 1
    return (x, y)


@pytest.mark.parametrize("w,h", BOARDS, ids=lambda v: str(v))
def test_oracle_reset_matches_the_model(w, h):
    for difficulty in (1, 2, 5, w + h):
        env = orc.Env(orc.gridworld_spec(w, h, 100, difficulty))
        for env_id in range(30):
            env.reset(seed=SEED, env_id=env_id, collect_id=3)
            agent, goal, trap = _reset_model(w, h, difficulty, SEED, env_id, 3)
            assert abs(goal[0] - agent[0]) + abs(goal[1] - agent[1]) <= difficulty
            assert goal != agent and trap not in (agent, goal)
            board = _board(w, h, agent, goal, trap)
            assert env.get_state() == board, (difficulty, env_id)
            assert env.observe() == [i * w * h + v for i, v in enumerate(board)]
            assert env.depth == 100 and not env.is_final()


@pytest.mark.parametrize("w,h", BOARDS, ids=lambda v: str(v))
def test_oracle_forced_steps_saturation_reward_and_final(w, h):
    """random forced actions (many of them off the board on thin boards): agent moves or stays as the model says,
    steps_left saturates at 0, reward and final follow lib.rs:147-155 until the episode ends, then 40 more steps."""
    rng = np.random.default_rng(w * 100 + h)
    max_steps, noop = 25, 0
    for env_id in range(12):
        env = orc.Env(orc.gridworld_spec(w, h, max_steps, 4))
        env.reset(seed=SEED, env_id=env_id, collect_id=9)
        agent, goal, trap = _reset_model(w, h, 4, SEED, env_id, 9)
        left = max_steps
        for t in range(max_steps + 40):
            x, y = agent
            legal = [y > 0, y + 1 < h, x > 0, x + 1 < w]
            assert env.masks() == legal
            a = int(rng.integers(0, 4))
            moved = _step(w, h, agent, a)
            noop += moved == agent
            agent, left = moved, max(0, left - 1)
            env.step(a)
            assert env.get_state() == _board(w, h, agent, goal, trap) and env.depth == left, (env_id, t)
            at_goal, at_trap = agent == goal, agent == trap
            assert env.success() == at_goal and env.is_final() == (at_goal or at_trap or left == 0)
            want = 1.0 if at_goal else -0.5 if (at_trap or left == 0) else np.float32(-0.5) / np.float32(left)
            assert np.float32(env.reward()) == np.float32(want)
        assert left == 0
    assert noop > 0


def test_gridworld_8x8_transpose_twists_are_a_symmetry():
    """helpers.gridworld_transpose_twists(8): for the transpose T with action map A (up<->left, down<->right),
    twist(observe(step(s, a))) == observe(step(twist(s), A(a))), and reward / final / success are unchanged.  Every
    twisted row keeps its cell value, so the twist keeps the 4 * 64 reachable rows of the compact table."""
    from helpers import gridworld_transpose_twists
    (ident, op), (_, ap) = gridworld_transpose_twists(8)
    N = 64
    assert ident == list(range(N * N)) and ap == [2, 3, 0, 1]
    assert all(op[i * N + v] % N == v for i in range(N) for v in range(N))
    T = [(i % 8) * 8 + i // 8 for i in range(N)]
    rng = np.random.default_rng(88)
    a_env, b_env = orc.Env(orc.gridworld_spec(8, 8, 64, 6)), orc.Env(orc.gridworld_spec(8, 8, 64, 6))
    for k in range(30):
        a_env.reset(seed=SEED, env_id=k, collect_id=2)
        s = a_env.get_state()
        twisted = [0] * N
        for i, v in enumerate(s):
            twisted[T[i]] = v
        b_env.set_state(twisted)
        assert sorted(op[o] for o in a_env.observe()) == sorted(b_env.observe())
        for a in rng.integers(0, 4, size=16):
            a_env.step(int(a)); b_env.step(ap[int(a)])
            assert sorted(op[o] for o in a_env.observe()) == sorted(b_env.observe())
            assert (a_env.success(), a_env.is_final(), a_env.reward()) == (b_env.success(), b_env.is_final(), b_env.reward())


def test_max_records_at_the_64_cell_limit():
    """twr_max_records validates the spec as twr_envs_create does: GridWorld takes every board of 3..64 cells and
    refuses 65 (5x13) with a message naming 64."""
    from twisterl_b200 import _lib
    L = _lib.load()
    for w, h in BOARDS + [(5, 5), (8, 4), (64, 1), (2, 32), (3, 1)]:
        spec = _lib.EnvSpec(_lib.ENV_GRIDWORLD, w, h, 6, 0, 100)
        assert L.twr_max_records(C.byref(spec), 10) == 10 * 101, (w, h)
    for w, h in ((5, 13), (13, 5), (9, 9), (1, 65), (2, 1)):
        assert L.twr_max_records(C.byref(_lib.EnvSpec(_lib.ENV_GRIDWORLD, w, h, 6, 0, 100)), 1) == -1, (w, h)
        assert b"3..64 cells" in L.twr_last_error(), (w, h)
