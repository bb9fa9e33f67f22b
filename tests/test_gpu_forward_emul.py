"""The tensor-core forward (k_forward_tc2) against tests/tc_emul.py, the exact CPU model of its operand rounding.

Main measure, per output: |kernel - model| / S, S = the sum of the magnitudes of everything the output is built from
(tc_emul.magnitude).  The model reproduces every rounding of the kernel's operands, so what remains is the order and
precision of fp32 accumulation; a dropped, misplaced or wrongly scaled term is much larger.  Measured over this file on
a B200 (1000 W power limit):

    precision   kernel vs model / S   BAR       a mutant of the kernel, same measure
    fp32        1.7e-8                1e-7      --
    f16x2       2.2e-8                1e-7      lo term of the last 128-feature chunk dropped in k_tc2_pack: 1.7e-6
    f16x2w16    2.2e-8                1e-7      (same mutant)
    f16f8c      9.7e-8                2.5e-7    TABLE8_SCALE 512 instead of 1024: 9.3e-7

Every rung of the ladder (set_tc_terms) is held to the bar of its kind, except rungs 1 and 5 (table lo term, h1 rounded
to nearest with no residue): there a pre-activation that the fp32 accumulator and the float64 model put on the two sides
of an fp16 rounding boundary moves h1 by one fp16 ulp (2^-10), 3.3e-7 S measured, BAR_RN_FLIP.  The kernel run at
one rung is >= 3.2e-7 S away from the model of every other rung at every width (MUTANT_MIN): well above the bars, so
the measure tells which terms ran.  f16x2w16 and f16f8c differ by less (~5e-8 S); where the choice between them
depends on the rows (forward_obs), the kernel is asserted to sit closer to the model of the variant that should run.

The suite's usual measure |d| / max(1, |ref|) against the float64 forward is asserted too, at the graded bars of
the README: fp32 1e-5, f16x2 1e-4, f16x2w16 and f16f8c 1e-3, on weights that give logits of order 1-5 (the embedding of
synth_state_dict x 8; measured 1.5e-6, 1.2e-5, 9.8e-4, 9.6e-4).  test_weight_scales prints where each precision leaves
its grade; DESIGN.md section 3 keeps the table."""
import os
from collections import defaultdict

import numpy as np
import pytest

import tc_emul as te
from helpers import synth_state_dict
from oracle import orc

pytestmark = pytest.mark.gpu

PRECISIONS = ("fp32", "f16x2", "f16x2w16", "f16f8c")
GRADE = {"fp32": 1e-5, "f16x2": 1e-4, "f16x2w16": 1e-3, "f16f8c": 1e-3}
BAR = {"fp32": 1e-7, "f16x2": 1e-7, "f16x2w16": 1e-7, "f16f8c": 2.5e-7}
BAR_RN_FLIP = 1e-6
MUTANT_MIN = 3e-7
RUNGS = list(range(8)) + [16 | 3]
WIDTHS = [(E, H) for E in range(128, 1025, 128) for H in (128, 256)]

MEASURED = defaultdict(float)          # precision -> max kernel-vs-model / S seen
WORST = {}                             # precision -> the test (and rung) where it was seen
MUTANT = {}                            # (E, H) -> smallest kernel(rung) vs model(other rung) / S
RUNGM = {}                             # (E, H, rung) -> kernel at that rung vs its model / S
DISPATCH = []                          # forward_obs on f16f8c: (n_obs, twists, fp8 ran, measure, measure vs the other variant)
GRADED = defaultdict(float)            # precision -> max |d| / max(1, |ref|) against float64 (normal scales)
SCALES = {}                            # (emb, w1) -> precision -> error against float64


@pytest.fixture(scope="module")
def engines():
    import twisterl_b200 as tw
    e = {p: tw.Engine(device=0, precision=p, seed=0x7C2) for p in PRECISIONS}
    yield e
    rows = ["\nkernel vs model, max |d| / S:  " + "  ".join(f"{p} {MEASURED[p]:.2e}" for p in PRECISIONS),
            "against float64, max |d| / max(1,|ref|):  " + "  ".join(f"{p} {GRADED[p]:.2e}" for p in PRECISIONS)]
    rows += [f"  worst {p}: {WORST.get(p)}" for p in PRECISIONS]
    for t in RUNGS:
        if RUNGM:
            rows.append(f"rung {t:2d} vs its model, max over widths: {max(v for k, v in RUNGM.items() if k[2] == t):.2e}")
    for d in DISPATCH:
        rows.append("f16f8c forward_obs n_obs %d %s fp8=%s: %.2e (other variant %.2e)" % d)
    if MUTANT:
        rows.append("smallest mutant gap / S: " + " ".join(f"{k}:{v:.1e}" for k, v in sorted(MUTANT.items())))
    for k, v in sorted(SCALES.items()):
        rows.append(f"scale emb x{k[0]} W1 x{k[1]}: " + "  ".join(f"{p} {v[p]:.2e}" for p in PRECISIONS))
    print("\n".join(rows))
    for x in e.values():
        x.close()


def _sd(E, H, A=4, obs_size=256, seed=0, emb_scale=8.0, w_scale=1.0):
    sd = synth_state_dict(seed + 7 * E + H, obs_size, E, H, A)
    sd["embeddings.weight"] = (sd["embeddings.weight"] * np.float32(emb_scale)).astype(np.float32)
    sd["common.0.weight"] = (sd["common.0.weight"] * np.float32(w_scale)).astype(np.float32)
    return sd


def _pol(sd, obs_size, twists=((), ())):
    from parity import make_policies
    return make_policies(sd, obs_size, *twists)[0]


def _spec(kind, w, h):
    from twisterl_b200 import _lib
    o = orc.puzzle_spec(w, h, 60, 2, 256) if kind == 0 else orc.gridworld_spec(w, h, 64, 10)
    return _lib.EnvSpec(o.kind, o.width, o.height, o.difficulty, o.depth_slope, o.max_depth)


def _batch(engines, kind, w, h, n, seed=1):
    """The same n envs (reset from the engines' shared seed) on every engine: (batches, their observations)."""
    from twisterl_b200.env import EnvBatch
    bs = {}
    for p, eng in engines.items():
        bs[p] = EnvBatch(_spec(kind, w, h), n, eng)
        bs[p].reset(env_id_base=1000 * seed, collect_id=seed)
    obs = bs["f16x2"].observe()
    assert all(np.array_equal(b.observe(), obs) for b in bs.values())
    return bs, obs


def _measure(w, prec, l, v, obs, perm=None, twists=((), ()), tc_terms=None, obs_rows=False, graded=True):
    """kernel (l, v) vs the model of what `prec` runs: returns the measure / S, records it, and checks the grade."""
    ml, mv, _ = te.engine_forward(w, prec, obs, perm, *twists, tc_terms=tc_terms, obs_rows=obs_rows)
    sl, sv = te.magnitude(w, obs, perm, *twists)
    m = max(te.rel_to_s(l, ml, sl), te.rel_to_s(v, mv, sv))
    _record(prec, m)
    if graded and tc_terms is None:
        rl, rv = te.forward64(w, obs, perm, *twists)
        g = max(te.rel_err(l, rl), te.rel_err(v, rv))
        GRADED[prec] = max(GRADED[prec], g)
        assert g <= GRADE[prec], (prec, g)
    assert m <= BAR[prec], (prec, tc_terms, m)
    return m


def _record(prec, m, what=""):
    if m > MEASURED[prec]:
        MEASURED[prec] = m
        WORST[prec] = os.environ.get("PYTEST_CURRENT_TEST", "").split(" ")[0] + what


def _fwd_batch(engines, pols, bs, perm=None):
    from twisterl_b200.nn import forward_batch
    return {p: forward_batch(engines[p], pols[p], bs[p], perm_idx=perm) for p in PRECISIONS}


# ----------------------------------------------------------------------------------------------- twist sets ---
def block_twists(rng, N, count, A=4, values=None):
    """`count` twists that map each block of N rows (one cell) onto another block: a cell permutation and, per cell, a
    permutation of the values below `values` (GridWorld: 4, so the compact table keeps its rows).  tc_fold = N."""
    values = values or N
    op, ap = [], []
    for _ in range(count):
        cells = rng.permutation(N)
        pm = np.zeros(N * N, np.int64)
        for i in range(N):
            v = np.concatenate([rng.permutation(values), np.arange(values, N)])
            pm[i * N:(i + 1) * N] = cells[i] * N + v
        op.append(pm.tolist()); ap.append(rng.permutation(A).tolist())
    return op, ap


def row_twists(rng, N, count, A=4, values=None):
    """`count` arbitrary row permutations (tc_fold = 0); with `values`, rows of a value below it stay among themselves
    (GridWorld's compact table)."""
    values = values or N
    op, ap = [], []
    for _ in range(count):
        rows = np.arange(N * N)
        reach = rows[rows % N < values]
        pm = rows.copy()
        pm[reach] = rng.permutation(reach)
        rest = rows[rows % N >= values]
        pm[rest] = rng.permutation(rest)
        op.append(pm.tolist()); ap.append(rng.permutation(A).tolist())
    return op, ap


def _perm(n, count):
    return None if count == 0 else (np.arange(n) % (count + 1) - 1).astype(np.int32)        # -1 and every twist


# ------------------------------------------------------------------------------------------------------ tests ---
@pytest.mark.parametrize("E,H", WIDTHS, ids=[f"E{e}_H{h}" for e, h in WIDTHS])
def test_widths_every_precision_and_rung(engines, E, H):
    """Puzzle15 with block-preserving twists at every width of the pair kernel: each engine against its model, then
    every rung of the ladder (set_tc_terms: the run-time-terms instantiation) against the model of THAT rung and,
    as mutants, against the model of every other rung."""
    from twisterl_b200.nn import forward_batch
    rng = np.random.default_rng(E + H)
    sd, tw = _sd(E, H), block_twists(rng, 16, 2)
    w = te.Weights(sd)
    pols = {p: _pol(sd, 256, tw) for p in PRECISIONS}
    b, obs = _batch(engines, 0, 4, 4, 257, seed=E)
    perm = _perm(257, 2)
    out = _fwd_batch(engines, pols, b, perm)
    for p in PRECISIONS:
        _measure(w, p, *out[p], obs, perm, tw)
    eng, pol = engines["f16x2"], pols["f16x2"]
    runs = {}
    try:
        for t in RUNGS:
            eng.set_tc_terms(t)
            runs[t] = forward_batch(eng, pol, b["f16x2"], perm_idx=perm)
    finally:
        eng.set_tc_terms(-1)
    sl, sv = te.magnitude(w, obs, perm, *tw)
    fold = te.fold_block(256, tw[0])
    models = {t: te.tc_forward(w, obs, perm, *tw, *te.dispatch(8 | t, fold, True)) for t in RUNGS}
    gap = np.inf
    for t, (l, v) in runs.items():
        ml, mv = models[t]
        m = max(te.rel_to_s(l, ml, sl), te.rel_to_s(v, mv, sv))
        RUNGM[(E, H, t)] = m
        assert m <= (BAR_RN_FLIP if t in (1, 5) else BAR["f16f8c"] if t & 16 else BAR["f16x2"]), (t, m)
        for u, (ml2, mv2) in models.items():
            if u != t and {u, t} != {3, 16 | 3}:       # fp8 and fp16 corrections of the same terms: close by design
                gap = min(gap, max(te.rel_to_s(l, ml2, sl), te.rel_to_s(v, mv2, sv)))
    MUTANT[(E, H)] = gap
    assert gap >= MUTANT_MIN, gap
    for p in PRECISIONS:
        pols[p].release()


CHUNKS = [(E, H, c) for E in (384, 640, 1024) for H in (128, 256) for c in range(E // 128)]


@pytest.mark.parametrize("E,H,chunk", CHUNKS, ids=[f"E{e}_H{h}_c{c}" for e, h, c in CHUNKS])
def test_chunk_isolation(engines, E, H, chunk):
    """Weights non-zero in one 128-feature chunk only (table columns, embedding bias, W1 rows): a term missing from that
    chunk shows at full size instead of being diluted by the others."""
    sd = _sd(E, H, seed=chunk)
    off = np.ones(E, bool)
    off[chunk * 128:(chunk + 1) * 128] = False
    sd["embeddings.weight"][off, :] = 0
    sd["embeddings.bias"][off] = 0
    sd["common.0.weight"][:, off] = 0
    tw = transpose_pair(4)
    w = te.Weights(sd)
    pols = {p: _pol(sd, 256, tw) for p in PRECISIONS}
    b, obs = _batch(engines, 0, 4, 4, 129, seed=chunk + 3)
    perm = _perm(129, 2)
    out = _fwd_batch(engines, pols, b, perm)
    for p in PRECISIONS:
        _measure(w, p, *out[p], obs, perm, tw)
        pols[p].release()


def transpose_pair(w):
    from helpers import transpose_twists
    return transpose_twists(w)


GEOMS = [(0, 2, 2), (0, 3, 2), (0, 3, 3), (0, 4, 3), (0, 4, 4), (1, 4, 3), (1, 5, 5), (1, 6, 5), (1, 8, 4)]
GEOM_CASES = [(k, gw, gh, E, H, tk) for (k, gw, gh) in GEOMS for (E, H) in ((512, 256), (384, 128)) for tk in ("none", "block", "rows")]


@pytest.mark.parametrize("kind,gw,gh,E,H,twk", GEOM_CASES, ids=[f"{'pz' if c[0] == 0 else 'gw'}{c[1]}x{c[2]}_E{c[3]}_H{c[4]}_{c[5]}" for c in GEOM_CASES])
def test_geometries(engines, kind, gw, gh, E, H, twk):
    """Tables of 16 to 256 rows (1 to 4 k-blocks of GEMM1, 3 with puzzle / GridWorld 4x3), the compact GridWorld table
    (5x5, 6x5, 8x4), without twists, with block-preserving twists (tc_fold > 0) and with arbitrary row permutations
    (tc_fold = 0: f16f8c runs its non-folded fp8 image with twists)."""
    N = gw * gh
    rng = np.random.default_rng(N + E)
    vals = 4 if kind == 1 else None
    tw = {"none": ((), ()), "block": block_twists(rng, N, 3, values=vals), "rows": row_twists(rng, N, 3, values=vals)}[twk]
    sd = _sd(E, H, obs_size=N * N, seed=N)
    w = te.Weights(sd)
    pols = {p: _pol(sd, N * N, tw) for p in PRECISIONS}
    b, obs = _batch(engines, kind, gw, gh, 300, seed=N)
    perm = _perm(300, 0 if twk == "none" else 3)
    out = _fwd_batch(engines, pols, b, perm)
    for p in PRECISIONS:
        _measure(w, p, *out[p], obs, perm, tw)
        pols[p].release()


TWIST_CASES = [(c, k, g) for c in (2, 8, 9, 32, 33, 127) for k in ("block", "rows") for g in ("pz4x4", "pz3x3")]


@pytest.mark.parametrize("count,twk,geom", TWIST_CASES, ids=[f"{c}_{k}_{g}" for c, k, g in TWIST_CASES])
def test_twist_counts(engines, count, twk, geom):
    """2 to 127 twists: the twist tables in shared memory (obs: <= 2048 entries, actions: <= 32 twists) and in global
    memory, with perm_idx rows mixing -1 and every twist; forward_obs on the same rows gives the same bits."""
    from twisterl_b200.nn import forward_obs
    gw, gh, E, H = (4, 4, 512, 256) if geom == "pz4x4" else (3, 3, 384, 128)
    N = gw * gh
    rng = np.random.default_rng(count * 7 + N)
    tw = (block_twists if twk == "block" else row_twists)(rng, N, count)
    sd = _sd(E, H, obs_size=N * N, seed=count)
    w = te.Weights(sd)
    pols = {p: _pol(sd, N * N, tw) for p in PRECISIONS}
    n = 2 * (count + 1) + 3
    b, obs = _batch(engines, 0, gw, gh, n, seed=count)
    perm = _perm(n, count)
    out = _fwd_batch(engines, pols, b, perm)
    for p in PRECISIONS:
        _measure(w, p, *out[p], obs, perm, tw)
        l2, v2 = forward_obs(engines[p], pols[p], obs, perm)
        assert np.array_equal(l2, out[p][0]) and np.array_equal(v2, out[p][1]), p
        pols[p].release()


@pytest.mark.parametrize("small,geom", [(8, "pz4x4"), (32, "pz4x4"), (25, "pz3x3"), (32, "pz3x3")])
def test_twist_tables_shared_and_global_agree(engines, small, geom):
    """A set of small + 1 twists whose first `small` are the small set: same bits on perm_idx -1..small-1, though one more
    twist moves the observation (4x4: 8 -> 9, 3x3: 25 -> 26) or action (32 -> 33) table to global memory."""
    gw, E, H = (4, 512, 256) if geom == "pz4x4" else (3, 384, 128)
    N = gw * gw
    rng = np.random.default_rng(small)
    op, ap = block_twists(rng, N, small + 1)
    sd = _sd(E, H, obs_size=N * N, seed=small)
    n = 3 * (small + 1)
    b, _ = _batch(engines, 0, gw, gw, n, seed=small)
    perm = _perm(n, small)
    from twisterl_b200.nn import forward_batch
    for p in PRECISIONS:
        a = _pol(sd, N * N, (op[:small], ap[:small]))
        c = _pol(sd, N * N, (op, ap))
        la, va = forward_batch(engines[p], a, b[p], perm_idx=perm)
        lc, vc = forward_batch(engines[p], c, b[p], perm_idx=perm)
        assert np.array_equal(la, lc) and np.array_equal(va, vc), p
        a.release(); c.release()


@pytest.mark.parametrize("twk", ["plain", "block", "rows"])
def test_forward_obs_rows(engines, twk):
    """Rows given directly: one index per block (the folded f16f8c image applies), and rows of 1 to 32 distinct indices
    that are not one per block, where f16f8c must fall back to fp16 corrections (and the model says so)."""
    from twisterl_b200.nn import forward_obs
    rng = np.random.default_rng(5)
    tw = {"plain": ((), ()), "block": block_twists(rng, 16, 2), "rows": row_twists(rng, 16, 2)}[twk]
    sd = _sd(512, 256, seed=11)
    w = te.Weights(sd)
    pols = {p: _pol(sd, 256, tw) for p in PRECISIONS}
    fold = te.fold_block(256, tw[0])
    _, obs0 = _batch(engines, 0, 4, 4, 200, seed=9)
    cases = [obs0] + [np.array([rng.choice(256, k, replace=False) for _ in range(129)]) for k in range(1, 33)]
    for obs in cases:
        perm = _perm(len(obs), 0 if twk == "plain" else 2)
        blocks = te.one_per_block(obs, fold)
        for p in PRECISIONS:
            l, v = forward_obs(engines[p], pols[p], obs, perm)
            m = _measure(w, p, l, v, obs, perm, tw, obs_rows=True)
            if p == "f16f8c":
                # which corrections ran: the kernel sits closer to the model of the dispatched variant than to the other
                f8 = fold == 0 or blocks
                ml, mv = te.tc_forward(w, obs, perm, *tw, terms=3, f8=not f8)
                sl, sv = te.magnitude(w, obs, perm, *tw)
                alt = max(te.rel_to_s(l, ml, sl), te.rel_to_s(v, mv, sv))
                DISPATCH.append((len(obs[0]), twk, f8, m, alt))
                assert m < alt, (len(obs[0]), twk, f8, m, alt)
    for p in PRECISIONS:
        pols[p].release()


@pytest.mark.parametrize("A", [1, 2, 3])
def test_fewer_actions(engines, A):
    """Policies with 1 to 3 actions (heads o < A, action twists of A entries) through forward_obs."""
    from twisterl_b200.nn import forward_obs
    rng = np.random.default_rng(A)
    tw = block_twists(rng, 16, 3, A=A)
    sd = _sd(512, 256, A=A, seed=A)
    w = te.Weights(sd)
    _, obs = _batch(engines, 0, 4, 4, 257, seed=A)
    perm = _perm(257, 3)
    for p in PRECISIONS:
        pol = _pol(sd, 256, tw)
        l, v = forward_obs(engines[p], pol, obs, perm)
        assert l.shape == (257, A)
        _measure(w, p, l, v, obs, perm, tw, obs_rows=True)
        pol.release()


@pytest.mark.parametrize("geom", ["pz4x4", "gw5x5"])
def test_collect_records(engines, geom):
    """The fused step path: a PPOCollector collect's recorded observations, twist indices, masked logits and values
    against the model on the unmasked entries."""
    import twisterl_b200 as tw_
    rng = np.random.default_rng(17)
    if geom == "pz4x4":
        N, tw, env = 16, block_twists(rng, 16, 2), tw_.env.Puzzle(4, 4, 12, 2, 256)
    else:
        N, tw, env = 25, block_twists(rng, 25, 2, values=4), tw_.env.GridWorld(5, 5, 64, 10)
    sd = _sd(512, 256 if N == 16 else 128, obs_size=N * N, seed=N)
    w = te.Weights(sd)
    for p in PRECISIONS:
        pol = _pol(sd, N * N, tw)
        d = tw_.collector.PPOCollector(600, 0.995, 0.995, 1, engine=engines[p]).collect(env, pol)
        obs, perm = d.obs_array.astype(np.int64), d.perms_array.astype(np.int64)
        assert set(np.unique(perm)) == {0, 1}
        l, v = d.logits_array, d.values_array
        ml, mv, _ = te.engine_forward(w, p, obs, perm, *tw)
        sl, sv = te.magnitude(w, obs, perm, *tw)
        live = l != np.float32(-1e10)
        m = max(float((np.abs(l - ml) / sl)[live].max()), te.rel_to_s(v, mv, sv))
        _record(p, m)
        assert live.any(axis=1).all() and m <= BAR[p], (p, m)
        pol.release()


@pytest.mark.parametrize("n", [1, 127, 128, 129, 255, 257, 40000])
def test_batch_sizes(engines, n):
    """Ragged tiles and, above 148 x 256 envs, more tiles than CTA pairs in a forward-only launch."""
    rng = np.random.default_rng(n)
    tw = block_twists(rng, 16, 2)
    sd = _sd(256, 128, seed=3)
    w = te.Weights(sd)
    pols = {p: _pol(sd, 256, tw) for p in PRECISIONS}
    b, obs = _batch(engines, 0, 4, 4, n, seed=n % 1000)
    perm = _perm(n, 2)
    out = _fwd_batch(engines, pols, b, perm)
    for p in PRECISIONS:
        _measure(w, p, *out[p], obs, perm, tw)
        pols[p].release()


def test_padding_is_exact(engines):
    """E = 384 runs zero-padded to a chunk pair: bit for bit the E = 512 policy whose fourth chunk has zero table columns,
    zero bias and zero W1 rows, at every precision."""
    sd = _sd(384, 256, seed=2)
    wide = {k: v.copy() for k, v in sd.items()}
    wide["embeddings.weight"] = np.concatenate([sd["embeddings.weight"], np.zeros((128, 256), np.float32)])
    wide["embeddings.bias"] = np.concatenate([sd["embeddings.bias"], np.zeros(128, np.float32)])
    wide["common.0.weight"] = np.concatenate([sd["common.0.weight"], np.zeros((256, 128), np.float32)], axis=1)
    tw = transpose_pair(4)
    b, _ = _batch(engines, 0, 4, 4, 300, seed=4)
    perm = _perm(300, 2)
    from twisterl_b200.nn import forward_batch
    for p in PRECISIONS:
        a, c = _pol(sd, 256, tw), _pol(wide, 256, tw)
        la, va = forward_batch(engines[p], a, b[p], perm_idx=perm)
        lc, vc = forward_batch(engines[p], c, b[p], perm_idx=perm)
        assert np.array_equal(la, lc) and np.array_equal(va, vc), p
        a.release(); c.release()


SCALE_CASES = [(e, s) for e in (0.01, 1.0, 8.0, 30.0, 200.0) for s in (0.01, 1.0, 8.0)]


@pytest.mark.parametrize("emb,w1", SCALE_CASES, ids=[f"emb{e}_w{s}" for e, s in SCALE_CASES])
def test_weight_scales(engines, emb, w1):
    """Embedding x {0.01 .. 200} and W1 x {0.01, 1, 8}: every precision against its model at the same bar; against the
    float64 forward the error is recorded (where each precision leaves its grade: the engine's printed table)."""
    sd = _sd(512, 256, seed=5, emb_scale=emb, w_scale=w1)
    w = te.Weights(sd)
    tw = transpose_pair(4)
    pols = {p: _pol(sd, 256, tw) for p in PRECISIONS}
    b, obs = _batch(engines, 0, 4, 4, 513, seed=6)
    perm = _perm(513, 2)
    out = _fwd_batch(engines, pols, b, perm)
    rl, rv = te.forward64(w, obs, perm, *tw)
    SCALES[(emb, w1)] = {}
    for p in PRECISIONS:
        _measure(w, p, *out[p], obs, perm, tw, graded=False)
        SCALES[(emb, w1)][p] = max(te.rel_err(out[p][0], rl), te.rel_err(out[p][1], rv))
        pols[p].release()


def test_f8c_h1_ceiling_on_device(engines):
    """f16f8c carries 16 h1 in fp16 (H1_SCALE8): beyond h1 = 4094 the fp16 hi saturates and a 2-bit residue carries the
    excess, beyond 7678 both saturate.  The kernel does exactly what the model says there, and leaves its grade."""
    from twisterl_b200.nn import forward_batch
    sd = _sd(512, 256, seed=8, emb_scale=1.0)
    # 64 features whose h1 (16 table entries of 200 .. 800) spans 3200 .. 12800; every operand stays inside fp16
    sd["embeddings.weight"][:64] = np.random.default_rng(8).uniform(200, 800, (64, 256)).astype(np.float32)
    sd["common.0.weight"][:, :64] *= np.float32(1e-3)
    w = te.Weights(sd)
    b, obs = _batch(engines, 0, 4, 4, 257, seed=8)
    pol = _pol(sd, 256)
    l, v = forward_batch(engines["f16f8c"], pol, b["f16f8c"])
    _measure(w, "f16f8c", l, v, obs, graded=False)
    rl, rv = te.forward64(w, obs)
    assert max(te.rel_err(l, rl), te.rel_err(v, rv)) > GRADE["f16f8c"]
    pol.release()
