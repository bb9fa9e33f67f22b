"""Both MCTS device paths held to the oracle across the policy shapes, twist counts, batch sizes and tree depths they
accept: the persistent whole-search kernel (k_mcts_persistent, its own fp32 forward split over the 8 CTAs of a cluster) and
the lockstep kernels (the regular forward kernels), plus the weight refresh that every search, forward and collect reads.

Every case asserts which path ran -- a persistent search costs its launches plus one root read-out, a lockstep search
more launches than it has simulations -- and, where the slicing matters, the TWISTERL_B200_MCTS_DEBUG line of
launch_mcts_persistent (trees, twists, resident clusters, shared-memory footprint, launches)."""
import re

import numpy as np
import pytest

from suite_loader import suite_precision

from helpers import (gridworld_transpose_twists, scramble_states, synth_conv_state_dict, synth_deep_state_dict,
                     synth_state_dict, transpose_twists)
from oracle import orc

pytestmark = pytest.mark.gpu
PRECISION = suite_precision(globals())

# first-divergence near-tie rule of test_gpu_az.py / test_gpu_mcts_twists.py
NEAR_TIE = {"fp32": 2e-4, "f16x2": 2e-3, "f16x2w16": 2e-2, "f16f8c": 2e-2}[PRECISION]
MCTS_PATH = 96                         # TWR_MCTS_PATH: recorded descent entries; deeper backups walk parent links
PM_CS, PM_TPC, PM_MAX_EC = 8, 40, 64   # cluster size, leaf slots per cluster, feature slice bound of k_mcts_persistent
SMEM_LIMIT = 227 * 1024
P16 = (0, 4, 4, 5, 2, 256)             # EnvSpec fields: kind, width, height, difficulty, depth_slope, max_depth
G5 = (1, 5, 5, 6, 0, 64)
DEBUG_LINE = re.compile(r"\[mcts\] persistent: (\d+) trees, (-?\d+) twist\(s\), (\d+) resident clusters of (\d+) CTAs "
                        r"\((\d+) B shared memory\), (\d+) launch\(es\) of <= (\d+) trees")


@pytest.fixture(scope="module")
def eng():
    import twisterl_b200 as tw
    e = tw.Engine(device=0, precision=PRECISION, seed=0x5A4E5)
    yield e
    e.close()


def pm_footprint(E, H, obs):
    """Shared memory of k_mcts_persistent: a copy of pm_layout (twr_mcts.cu)."""
    EC, per = E // PM_CS, PM_TPC // PM_CS
    floats = EC * H + obs * EC + PM_TPC * EC + H + EC + 5 * (H + 8) + per * PM_CS * H + per * H + per * 8
    return (4 * floats + 16 * PM_TPC + 4 * PM_TPC + 15) & ~15


def persistent_accepts(E, H, obs, T=0):
    """The shape checks of launch_mcts_persistent for a standard-shape policy at max_expand_depth 1."""
    return (E % (PM_CS * 4) == 0 and E <= PM_CS * PM_MAX_EC and H in (128, 256)
            and PM_CS * (PM_TPC // PM_CS // max(T, 1)) >= PM_CS and pm_footprint(E, H, obs) <= SMEM_LIMIT)


def _batch(eng, spec, states):
    from twisterl_b200 import _lib
    from twisterl_b200.env import EnvBatch
    b = EnvBatch(_lib.EnvSpec(*spec), len(states), eng)
    b.set_state(states)
    return b


def _oracle_env(spec, state):
    kind, w, h, diff, slope, md = spec
    env = orc.Env(orc.puzzle_spec(w, h, diff, slope, md) if kind == 0 else orc.gridworld_spec(w, h, md, diff))
    env.set_state([int(x) for x in state])
    return env


def _puzzle_states(seed, n, w, h, moves=12):
    return scramble_states(np.random.default_rng(seed), n, w, h, moves)


def _gridworld_states(eng, spec, n, base, cid):
    from twisterl_b200 import _lib
    from twisterl_b200.env import EnvBatch
    b = EnvBatch(_lib.EnvSpec(*spec), n, eng)
    b.reset(env_id_base=base, collect_id=cid)
    return b.get_state()


def _ident_transpose_twists(kind, w, T):
    """T twists alternating transpose, identity, transpose, ... (the pair set of _identity_twists / transpose_twists)."""
    ob, ac = (transpose_twists if kind == 0 else gridworld_transpose_twists)(w)
    order = [1, 0] * 3
    return [ob[i] for i in order[:T]], [ac[i] for i in order[:T]]


def _search(eng, pol, spec, states, n_sims, capfd, monkeypatch, med=1, base=700, cid=5, t=1, lockstep=False):
    """One twr_debug_mcts_trace call: (probs, visits, trace, launches, debug) where debug is the parsed line of
    launch_mcts_persistent (None: the lockstep path ran)."""
    from twisterl_b200 import _lib
    monkeypatch.setenv("TWISTERL_B200_MCTS_DEBUG", "1")
    if lockstep:
        monkeypatch.setenv("TWISTERL_B200_MCTS_LOCKSTEP", "1")
    b = _batch(eng, spec, states)
    h = pol.device_handle(eng)                            # creating the device policy launches its operand packing
    n = len(states)
    probs = np.zeros((n, 4), np.float32); visits = np.zeros((n, 4), np.int32)
    trace = np.zeros((max(n_sims, 1), n, 2), np.int32)
    earlier = capfd.readouterr().out
    n0 = eng.launch_count()
    _lib.check(_lib.load().twr_debug_mcts_trace(eng._h, h, b._h, n_sims, 1.41, med, base, cid, t,
                                                _lib.ptr(probs), _lib.ptr(visits), _lib.ptr(trace)))
    launches = eng.launch_count() - n0
    lines = DEBUG_LINE.findall(capfd.readouterr().err)
    print(earlier, end="")                                # the case's report lines so far stay in its captured output
    monkeypatch.delenv("TWISTERL_B200_MCTS_DEBUG")
    monkeypatch.delenv("TWISTERL_B200_MCTS_LOCKSTEP", raising=False)
    assert len(lines) <= 1
    dbg = None
    if lines:
        trees, twists, nc, cs, smem, n_launch, slice_ = (int(x) for x in lines[0])
        dbg = dict(trees=trees, twists=twists, nc=nc, cs=cs, smem=smem, n_launch=n_launch, slice=slice_)
        assert trees == n and cs == PM_CS and 1 <= n_launch <= 4 and 1 <= nc <= 148 // PM_CS
        assert launches == n_launch + 1, f"persistent search took {launches} launches, the line says {n_launch} + read-out"
    return probs, visits, trace[:n_sims], launches, dbg


def _expect_path(dbg, launches, n_sims, persistent):
    if persistent:
        assert dbg is not None, "the search fell back to the lockstep path"
    else:
        assert dbg is None, f"the search ran persistent: {dbg}"
        assert launches > n_sims, f"a lockstep search of {n_sims} simulations took only {launches} launches"


def _check(eng, opol, spec, states, res, n_sims, label, med=1, base=700, cid=5, t=1):
    """test_gpu_mcts_twists.py::_check_searches on one result: equal visit sums; equal visit counts with probabilities
    within 1e-6, or a first divergence where the oracle's margin was below NEAR_TIE; at least half identical."""
    probs, visits, trace, launches, dbg = res
    same = checked = 0
    for i in range(len(states)):
        env = _oracle_env(spec, states[i])
        op, ov = orc.mcts_probs(env, opol, n_sims, 1.41, med, seed=eng.seed, collect_id=cid, stream_id=base + i, t=t)
        checked += 1
        assert visits[i].sum() == ov.sum(), f"tree {i}: {visits[i]} vs oracle {ov}"
        if np.array_equal(visits[i], ov):
            same += 1
            assert np.allclose(probs[i], op, atol=1e-6)
            continue
        _, _, leaf, child, margin = orc.mcts_trace(env, opol, n_sims, 1.41, med, seed=eng.seed, collect_id=cid,
                                                   stream_id=base + i, t=t)
        div = next((s for s in range(n_sims) if trace[s, i, 0] != leaf[s] or trace[s, i, 1] != child[s]), None)
        assert div is not None, f"tree {i}: visit counts differ but every simulation took the oracle's path"
        assert margin[div] < NEAR_TIE, f"tree {i}: first divergence at simulation {div} where the oracle's margin was {margin[div]}"
    path = "lockstep" if dbg is None else f"persistent ({dbg['nc']} clusters, {dbg['smem']} B, {dbg['n_launch']} launch(es))"
    print(f"[{label}] {path}: identical {same}/{checked}, near-tie {checked - same}")
    assert same >= checked // 2


def _run_case(eng, capfd, monkeypatch, pol, opol, spec, states, n_sims, persistent, label, med=1, lockstep=False,
              footprint=None):
    res = _search(eng, pol, spec, states, n_sims, capfd, monkeypatch, med=med, lockstep=lockstep)
    _expect_path(res[4], res[3], n_sims, persistent)
    if footprint is not None and res[4] is not None:
        assert res[4]["smem"] == footprint
    _check(eng, opol, spec, states, res, n_sims, label, med=med)
    return res


# ---------------------------------------------------------------------------- 1. embedding and common widths ---
@pytest.mark.parametrize("H", [128, 256])
@pytest.mark.parametrize("E", [32, 96, 128, 256, 384, 512])
def test_widths_run_persistent_and_match_oracle(eng, capfd, monkeypatch, E, H):
    """EC = E/8 from 4 to PM_MAX_EC: every register-cache bound of phase B, one and two leaf groups (H = 256 / 128)."""
    from parity import make_policies
    assert persistent_accepts(E, H, 256)
    pol, opol = make_policies(synth_state_dict(E + H, 256, E, H, 4), 256)
    _run_case(eng, capfd, monkeypatch, pol, opol, P16, _puzzle_states(E * H, 64, 4, 4), 24, True, f"E{E} H{H}",
              footprint=pm_footprint(E, H, 256))


@pytest.mark.parametrize("shape", ["E1024-H256", "E528-H128", "E256-H64", "E256-H192"])
def test_refused_widths_fall_back_to_lockstep_and_match_oracle(eng, capfd, monkeypatch, shape):
    """E beyond PM_CS * PM_MAX_EC (the tensor-core forward on its precisions), E not a multiple of 32 (the fp32 forward),
    H outside {128, 256}."""
    from parity import make_policies
    E, H = (int(x[1:]) for x in shape.split("-"))
    assert not persistent_accepts(E, H, 256)
    pol, opol = make_policies(synth_state_dict(E + H, 256, E, H, 4), 256)
    _run_case(eng, capfd, monkeypatch, pol, opol, P16, _puzzle_states(E + 3 * H, 48, 4, 4), 16, False, shape)


def test_deep_stack_policy_falls_back_to_lockstep_and_matches_oracle(eng, capfd, monkeypatch):
    from parity import make_policies_general
    pol, opol = make_policies_general(synth_deep_state_dict(12, 256, 256, (128, 128), (64,), (32,), 4), 256)
    _run_case(eng, capfd, monkeypatch, pol, opol, P16, _puzzle_states(12, 48, 4, 4), 16, False, "deep stack")


@pytest.mark.parametrize("conv_dim", [0, 1])
def test_conv1d_policy_runs_persistent_on_its_expanded_table_and_matches_oracle(eng, capfd, monkeypatch, conv_dim):
    """A Conv1dPolicy reaches the engine as its expanded [N*N][v*N] EmbeddingBag table (twr_policy_create), a plain
    standard-shape policy: with v*N = 256 it takes the persistent kernel like any other."""
    from parity import make_conv1d_policies
    pol, opol = make_conv1d_policies(synth_conv_state_dict(13 + conv_dim, 16, 16, 256, 128, 4), [16, 16], conv_dim)
    _run_case(eng, capfd, monkeypatch, pol, opol, P16, _puzzle_states(13 + conv_dim, 48, 4, 4), 16, True,
              f"conv1d dim {conv_dim}", footprint=pm_footprint(256, 128, 256))


@pytest.mark.parametrize("med", [0, 2])
def test_max_expand_depth_other_than_one_runs_lockstep_and_matches_oracle(eng, capfd, monkeypatch, med):
    from parity import make_policies
    pol, opol = make_policies(synth_state_dict(96, 256, 96, 256, 4), 256)
    _run_case(eng, capfd, monkeypatch, pol, opol, P16, _puzzle_states(96 + med, 48, 4, 4), 20, False,
              f"E96 H256 max_expand_depth {med}", med=med)


# -------------------------------------------------------------------------------------------- 2. geometries ---
GEOMETRIES = {
    # name: (spec, E, H, persistent)
    "puzzle2x2": ((0, 2, 2, 3, 2, 16), 128, 128, True),
    "puzzle3x2": ((0, 3, 2, 4, 2, 32), 128, 128, True),
    "puzzle3x3": ((0, 3, 3, 5, 2, 64), 128, 256, True),
    "gridworld4x3": ((1, 4, 3, 3, 0, 32), 128, 128, True),
    "gridworld5x5-E512-H128": ((1, 5, 5, 6, 0, 64), 512, 128, True),      # 1952 B under the limit
    "gridworld5x5-E512-H256": ((1, 5, 5, 6, 0, 64), 512, 256, False),     # 289 KB
    "gridworld6x5-E128-H128": ((1, 6, 5, 5, 0, 64), 128, 128, True),
    "gridworld6x5-E352-H128": ((1, 6, 5, 5, 0, 64), 352, 128, True),      # the largest E under the limit
    "gridworld6x5-E384-H128": ((1, 6, 5, 5, 0, 64), 384, 128, False),     # 32 B over it
    "gridworld8x4-E128-H128": ((1, 8, 4, 5, 0, 64), 128, 128, True),
    "gridworld8x4-E320-H128": ((1, 8, 4, 5, 0, 64), 320, 128, True),
    "gridworld8x4-E352-H128": ((1, 8, 4, 5, 0, 64), 352, 128, False),
}


@pytest.mark.parametrize("name", list(GEOMETRIES))
def test_geometries_match_oracle_on_the_path_their_footprint_allows(eng, capfd, monkeypatch, name):
    from parity import make_policies
    spec, E, H, persistent = GEOMETRIES[name]
    kind, w, h = spec[:3]
    N = w * h
    obs = N * N
    assert persistent_accepts(E, H, obs) == persistent, (name, pm_footprint(E, H, obs) - SMEM_LIMIT)
    seed = sum(map(ord, name))
    try:
        pol, opol = make_policies(synth_state_dict(seed, obs, E, H, 4), obs)
        pol.device_handle(eng)
    except RuntimeError as exc:                      # a precision that has no forward kernel for this shape says so
        assert "policy shape not supported on the device" in str(exc), str(exc)
        print(f"[{name}] refused on {PRECISION}: {exc}")
        return
    states = _puzzle_states(seed, 64, w, h) if kind == 0 else _gridworld_states(eng, spec, 64, seed, 3)
    res = _run_case(eng, capfd, monkeypatch, pol, opol, spec, states, 24, persistent, name,
                    footprint=pm_footprint(E, H, obs))
    if persistent:
        print(f"[{name}] footprint {res[4]['smem']} B, {SMEM_LIMIT - res[4]['smem']} B under the limit")
    else:
        print(f"[{name}] footprint {pm_footprint(E, H, obs)} B, {pm_footprint(E, H, obs) - SMEM_LIMIT} B over the limit")


# --------------------------------------------------------------------------- 3. twist counts, persistent kernel ---
@pytest.mark.parametrize("T", [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("which", ["puzzle4x4", "gridworld5x5"])
def test_twist_counts_match_oracle(eng, capfd, monkeypatch, which, T):
    """T = 1..5 leave 8 * floor(5 / T) trees per cluster (T = 3, 4 leave leaf slots idle, T = 5 fills all 40); T = 6 leaves
    none and falls back.  Twists alternate transpose and identity."""
    from parity import make_policies
    if which == "puzzle4x4":
        spec, obs, E, H = P16, 256, 256, 256
        states = _puzzle_states(40 + T, 64, 4, 4)
    else:
        spec, obs, E, H = G5, 625, 512, 128
        states = _gridworld_states(eng, spec, 64, 40 + T, 2)
    persistent = T <= 5
    assert persistent_accepts(E, H, obs, T) == persistent
    pol, opol = make_policies(synth_state_dict(50 + T, obs, E, H, 4), obs, *_ident_transpose_twists(spec[0], spec[1], T))
    res = _run_case(eng, capfd, monkeypatch, pol, opol, spec, states, 20, persistent, f"{which} T={T}")
    if persistent:
        assert res[4]["twists"] == T
    else:
        assert res[3] > 20 * T                        # T forwards per simulation


# ---------------------------------------------------------------------------- 4. batch sizes, launch splitting ---
@pytest.mark.parametrize("T", [0, 2])
def test_batch_sizes_and_launch_splitting_match_oracle(eng, capfd, monkeypatch, T):
    """Batches of 1 tree, fewer trees than resident clusters, k * room +- 1 for 1 to 4 launches (room = resident clusters x
    trees per cluster, read from the debug line, not assumed), and the first size that falls back."""
    from parity import make_policies
    twists = _ident_transpose_twists(0, 4, T) if T else ()
    pol, opol = make_policies(synth_state_dict(60 + T, 256, 128, 128, 4), 256, *twists)
    n_sims = 10
    all_states = _puzzle_states(61 + T, 4 * 720 + 8, 4, 4)

    def run(n, expect_launches):
        states = all_states[:n]
        res = _search(eng, pol, P16, states, n_sims, capfd, monkeypatch)
        _expect_path(res[4], res[3], n_sims, expect_launches > 0)
        if expect_launches:
            assert res[4]["n_launch"] == expect_launches and res[4]["slice"] == -(-n // expect_launches)
            assert res[4]["twists"] == T
        _check(eng, opol, P16, states, res, n_sims, f"T={T} batch {n}")
        return res[4]

    dbg = run(1, 1)
    nc = dbg["nc"]
    room = nc * PM_CS * (PM_TPC // PM_CS // max(T, 1))
    print(f"[T={T}] {nc} resident clusters, {room} trees per launch")
    assert len(all_states) > 4 * room
    if nc > 2:
        run(nc - 1, 1)                                 # one tree per cluster, fewer clusters than resident
    for n in sorted({room - 1, room, room + 1, 2 * room - 1, 2 * room + 1, 3 * room + 1, 4 * room}):
        run(n, -(-n // room))
    run(4 * room + 1, 0)                               # five launches' worth: the lockstep path


# ------------------------------------------------------------------------------------------------ 5. deep trees ---
def _chain_policy(seed, E, H):
    """A policy whose prior is nearly one-hot on the first legal move in the order left, up, right, down (action biases
    60, 40, 20, 0 dwarf the trained part of the logits), with a zero value head: each simulation extends one chain by a
    node until it reaches the depth-budget terminal."""
    sd = synth_state_dict(seed, 256, E, H, 4)
    sd["action.0.bias"] = np.array([60.0, 40.0, 20.0, 0.0], np.float32)
    sd["value.0.weight"] = np.zeros_like(sd["value.0.weight"])
    sd["value.0.bias"] = np.zeros_like(sd["value.0.bias"])
    return sd


@pytest.mark.parametrize("lockstep", [False, True])
def test_deep_trees_back_up_past_the_recorded_path(eng, capfd, monkeypatch, lockstep):
    """Descents deeper than TWR_MCTS_PATH: both kernels switch from the recorded path to the parent walk."""
    from parity import make_policies
    depth_budget, n_sims, n = 150, 300, 48
    spec = (0, 4, 4, 5, 2, depth_budget)               # set_state gives every board depth_budget moves
    rng = np.random.default_rng(77)
    states = np.array([rng.permutation(16) for _ in range(n)])
    pol, opol = make_policies(_chain_policy(78, 128, 128), 256)
    _run_case(eng, capfd, monkeypatch, pol, opol, spec, states, n_sims, not lockstep,
              f"deep trees {'lockstep' if lockstep else 'persistent'}", lockstep=lockstep)
    deepest = []
    for i in range(n):
        _, _, _, _, _, plen = orc.mcts_trace(_oracle_env(spec, states[i]), opol, n_sims, 1.41, 1, seed=eng.seed,
                                             collect_id=5, stream_id=700 + i, t=1, path_lengths=True)
        deepest.append(int(plen.max()))
    print(f"[deep trees] longest backup path {max(deepest)} nodes, {sum(d > MCTS_PATH for d in deepest)}/{n} trees past {MCTS_PATH}")
    assert max(deepest) > MCTS_PATH
    assert sum(d > MCTS_PATH for d in deepest) >= n // 2
    assert max(deepest) == depth_budget + 1            # the chain reached the depth-budget terminal


# -------------------------------------------------------------------------------------------- 6. weight refresh ---
def _torch_basic(sd, device):
    """A torch module shaped like the reference's BasicPolicy holding the weights of state dict `sd`."""
    import torch
    obs, E = sd["embeddings.weight"].shape[1], sd["embeddings.weight"].shape[0]
    H, A = sd["common.0.weight"].shape[0], sd["action.0.weight"].shape[0]
    m = torch.nn.Module()
    m.embeddings = torch.nn.Linear(obs, E)
    m.common = torch.nn.Sequential(torch.nn.Linear(E, H), torch.nn.ReLU())
    m.action = torch.nn.Sequential(torch.nn.Linear(H, A))
    m.value = torch.nn.Sequential(torch.nn.Linear(H, 1))
    m.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()})
    return m.to(device)


def _collect(eng, env, pol, n, cid):
    import twisterl_b200 as tw
    eng.set_collect_id(cid)
    d = tw.collector.PPOCollector(n, 0.995, 0.995, 1, engine=eng).collect(env, pol)
    return [d.obs_array, d.logits_array, d.values_array, d.rewards_array, d.actions_array, d.perms_array,
            d.additional_array("advs"), d.additional_array("rets"), np.asarray(d.ep_len)]


@pytest.mark.parametrize("which", ["puzzle4x4", "puzzle4x4-twisted", "gridworld5x5"])
def test_update_from_torch_reaches_every_consumer(eng, capfd, monkeypatch, which):
    """After update_from_torch(W1), a policy created from W0 and already used by both search kernels and the operand image
    computes bit for bit what a policy created from W1 computes: forwards, searches on both paths and a PPO collect."""
    import torch

    import twisterl_b200 as tw
    from parity import make_policies
    from twisterl_b200.nn import forward_batch
    if which.startswith("puzzle"):
        spec, obs, E, H = P16, 256, 256, 128
        twists = transpose_twists(4) if which.endswith("twisted") else ()
        states = _puzzle_states(90, 64, 4, 4)
        env = tw.env.Puzzle(4, 4, 5, 2, 256)
    else:
        spec, obs, E, H = G5, 625, 512, 128
        twists = gridworld_transpose_twists(5)
        states = _gridworld_states(eng, spec, 64, 90, 1)
        env = tw.env.GridWorld(5, 5, 64, 6)
    sd0, sd1 = synth_state_dict(91, obs, E, H, 4), synth_state_dict(92, obs, E, H, 4)
    pol, _ = make_policies(sd0, obs, *twists)
    fresh, ofresh = make_policies(sd1, obs, *twists)
    b = _batch(eng, spec, states)
    for lockstep in (False, True):                      # both kernels (and the operand image) have read W0
        _search(eng, pol, spec, states, 12, capfd, monkeypatch, lockstep=lockstep)
    forward_batch(eng, pol, b)
    pol.update_from_torch(_torch_basic(sd1, torch.device("cuda", eng.device)), eng)
    for x, y in zip(forward_batch(eng, pol, b), forward_batch(eng, fresh, b)):
        assert np.array_equal(x, y)
    for lockstep in (False, True):
        ra = _search(eng, pol, spec, states, 24, capfd, monkeypatch, lockstep=lockstep)
        rb = _search(eng, fresh, spec, states, 24, capfd, monkeypatch, lockstep=lockstep)
        _expect_path(ra[4], ra[3], 24, not lockstep)
        for x, y in zip(ra[:3], rb[:3]):
            assert np.array_equal(x, y)
        if not lockstep:                                # and W1 is what the oracle evaluates
            _check(eng, ofresh, spec, states, ra, 24, f"{which} refreshed")
    for x, y in zip(_collect(eng, env, pol, 256, 61), _collect(eng, env, fresh, 256, 61)):
        assert np.array_equal(x, y)


def test_update_from_torch_refusals(eng):
    import torch

    from parity import make_conv1d_policies, make_policies
    dev = torch.device("cuda", eng.device)
    sd = synth_state_dict(93, 256, 256, 128, 4)
    conv, _ = make_conv1d_policies(synth_conv_state_dict(94, 16, 16, 256, 128, 4), [16, 16], 0)
    with pytest.raises(NotImplementedError):
        conv.update_from_torch(_torch_basic(sd, dev), eng)
    pol, _ = make_policies(sd, 256)
    with pytest.raises(ValueError, match="different architectures"):
        pol.update_from_torch(_torch_basic(synth_state_dict(95, 256, 256, 256, 4), dev), eng)
    with pytest.raises(ValueError, match="lives on cpu"):
        pol.update_from_torch(_torch_basic(sd, torch.device("cpu")), eng)
