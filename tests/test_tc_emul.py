"""CPU checks of tests/tc_emul.py, the operand model the tensor-core forward is held to in test_gpu_forward_emul.py: its
rounding helpers against exhaustive / known encodings, its f16x2 rung against the float64 forward within the analytic
bound of split operands, and its precision ladder against scripts/precision_ladder_emul.py and the reference's trained
puzzle15 outputs (tests/golden/policy15_trained.npz)."""
import importlib.util
from pathlib import Path

import numpy as np
import pytest

import tc_emul as te
from helpers import (gridworld_transpose_twists, obs_from_states, scramble_states, synth_state_dict, trained15,
                     transpose_twists)

ROOT = Path(__file__).resolve().parent.parent


def _finite_f16():
    v = np.arange(1 << 16, dtype=np.uint32).astype(np.uint16).view(np.float16)
    return np.unique(v[np.isfinite(v)].astype(np.float32))


def test_fp16_rz_on_every_fp16_value_and_midpoint():
    vals = _finite_f16()                                   # sorted, -65504 .. 65504, one zero
    assert np.array_equal(te.fp16_rz(vals), vals)
    pos = vals[vals >= 0]
    lo, hi = pos[:-1], pos[1:]
    mid = ((lo.astype(np.float64) + hi) / 2).astype(np.float32)    # exact in float32: fp16 has 13 fewer bits
    for x, want in ((mid, lo), (np.nextafter(hi, np.float32(0)), lo), (np.nextafter(lo, np.float32(np.inf)), lo)):
        assert np.array_equal(te.fp16_rz(x), want)
        assert np.array_equal(te.fp16_rz(-x), -want)
    # round to nearest, for contrast: the midpoints go to the even neighbour
    even = (lo.astype(np.float16).view(np.uint16) & 1) == 0
    assert np.array_equal(te.fp16_rn(mid), np.where(even, lo, hi))
    # beyond the largest finite value rz saturates, rn overflows
    big = np.array([65504, 65519, 65520, 1e6, 3e38], np.float32)
    assert np.array_equal(te.fp16_rz(big), np.full(5, 65504, np.float32))
    assert np.array_equal(te.fp16_rz(-big), np.full(5, -65504, np.float32))
    assert np.isinf(te.fp16_rn(np.float32(65520)))


def _decode(code, ebits, mbits, bias, fn):
    s, e, m = code >> (ebits + mbits), (code >> mbits) & ((1 << ebits) - 1), code & ((1 << mbits) - 1)
    if fn and e == (1 << ebits) - 1 and m == (1 << mbits) - 1:
        return None                                          # e4m3fn: S.1111.111 is NaN, no infinities
    if not fn and e == (1 << ebits) - 1:
        return None                                          # e5m2: IEEE-style inf / NaN
    v = (m / (1 << mbits)) * 2.0 ** (1 - bias) if e == 0 else (1 + m / (1 << mbits)) * 2.0 ** (e - bias)
    return -v if s else v


@pytest.mark.parametrize("fmt", ["e4m3", "e5m2"])
def test_fp8_roundings_against_their_encodings(fmt):
    ebits, mbits, bias, fn, top = (4, 3, 7, True, 448.0) if fmt == "e4m3" else (5, 2, 15, False, 57344.0)
    f = te.e4m3 if fmt == "e4m3" else te.e5m2
    codes = [(c, _decode(c, ebits, mbits, bias, fn)) for c in range(128)]
    codes = [(c, v) for c, v in codes if v is not None]
    vals = np.array([v for _, v in codes], np.float32)
    assert vals.max() == top and vals[1] == 2.0 ** (1 - bias - mbits)          # largest finite, smallest subnormal
    assert np.array_equal(f(vals), vals) and np.array_equal(f(-vals), -vals)
    # every midpoint ties to the neighbour with an even code (0 included: half the smallest subnormal rounds to zero)
    mid = ((vals[:-1].astype(np.float64) + vals[1:]) / 2).astype(np.float32)
    want = np.array([v if c % 2 == 0 else vn for (c, v), (_, vn) in zip(codes[:-1], codes[1:])], np.float32)
    assert np.array_equal(f(mid), want) and np.array_equal(f(-mid), -want)
    assert np.array_equal(f(np.nextafter(mid, np.float32(0))), vals[:-1])
    assert np.array_equal(f(np.nextafter(mid, np.float32(np.inf))), vals[1:])
    # satfinite: anything beyond the largest finite value (ties and infinities included) saturates, with its sign
    for x in (top * 1.03, top * 1.07, top * 2, 1e30, np.inf):
        assert f(np.float32(x)) == top and f(np.float32(-x)) == -top
    known = {"e4m3": [(2.0 ** -10, 0.0), (3 * 2.0 ** -11, 2.0 ** -9), (1.0625, 1.0), (1.1875, 1.25), (464.0, 448.0)],
             "e5m2": [(2.0 ** -17, 0.0), (3 * 2.0 ** -18, 2.0 ** -16), (1.125, 1.0), (1.375, 1.5), (61440.0, 57344.0)]}
    for x, y in known[fmt]:
        assert f(np.float32(x)) == np.float32(y), (x, y)


@pytest.mark.parametrize("fmt", ["e4m3", "e5m2"])
def test_fp8_roundings_match_torch_casts(fmt):
    torch = pytest.importorskip("torch")
    x = np.random.default_rng(4).standard_normal(200_000).astype(np.float32) * np.float32(2.0) ** \
        np.random.default_rng(5).integers(-22, 18, 200_000).astype(np.float32)
    top, dt, f = (448.0, torch.float8_e4m3fn, te.e4m3) if fmt == "e4m3" else (57344.0, torch.float8_e5m2, te.e5m2)
    ref = torch.from_numpy(np.clip(x, -top, top)).to(dt).to(torch.float32).numpy()
    assert np.array_equal(f(x), ref)


def test_fold_block_and_dispatch():
    assert te.fold_block(256) == 16 and te.fold_block(81, transpose_twists(3)[0]) == 9
    assert te.fold_block(625, gridworld_transpose_twists(5)[0]) == 25 and te.fold_block(144) == 12
    assert te.fold_block(200) == 0 and te.fold_block(81, [np.random.default_rng(0).permutation(81)]) == 0
    assert te.one_per_block([[0, 5, 10, 15]], 4) and not te.one_per_block([[0, 1, 10, 15]], 4)
    assert not te.one_per_block([[0, 5, 10]], 4)
    assert te.dispatch(0, 16, True) == (7, False, 0) and te.dispatch(8 | 3, 16, True) == (3, False, 0)
    assert te.dispatch(16 | 8 | 3, 16, True) == (3, True, 16) and te.dispatch(16 | 8 | 3, 16, False) == (3, False, 0)
    assert te.dispatch(16 | 8 | 3, 0, False) == (3, True, 0) and te.dispatch(8, 0, True) == (0, False, 0)


@pytest.mark.parametrize("E,H,scale", [(512, 256, 8.0), (384, 128, 8.0), (1024, 256, 30.0), (128, 128, 1.0)])
def test_f16x2_model_within_split_operand_bound(E, H, scale):
    """Terms 7 = every fp32 operand as fp16 hi + lo: each summand is exact to a few 2^-22 of its magnitude (hi + lo of
    the table, of W1, of h1 with its rz hi, and the dropped lo x lo product); with independent signs the sums stay far
    inside |model - float64| <= 2^-22 S (measured: ~1e-9 S), while a rung without the lo terms is >= 100x further out."""
    sd = synth_state_dict(E + H, 256, E, H, 4)
    sd["embeddings.weight"] = sd["embeddings.weight"] * np.float32(scale)
    w = te.Weights(sd)
    obs = obs_from_states(scramble_states(np.random.default_rng(E), 1024, 4, 4, 200))
    l64, v64 = te.forward64(w, obs)
    sl, sv = te.magnitude(w, obs)
    l7, v7 = te.tc_forward(w, obs, terms=7)
    m7 = max(te.rel_to_s(l7, l64, sl), te.rel_to_s(v7, v64, sv))
    assert m7 <= 2.0 ** -22
    for t in (3, 5, 6):
        lt, vt = te.tc_forward(w, obs, terms=t)
        assert max(te.rel_to_s(lt, l64, sl), te.rel_to_s(vt, v64, sv)) > 100 * m7, t


def test_model_ladder_reproduces_the_emulation_script_and_the_golden_outputs():
    """The rungs against the trained puzzle15 outputs of the reference: scripts/precision_ladder_emul.py's numbers
    (which round h1 to nearest and accumulate in float32) within a factor 2, f16x2 near the 1.1e-5 that
    test_gpu_precision.py records on the device, f16x2w16 / f16f8c inside 1e-3 and every cheaper rung outside it."""
    spec = importlib.util.spec_from_file_location("precision_ladder_emul", ROOT / "scripts" / "precision_ladder_emul.py")
    script = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(script)
    z, sd = trained15()
    w = te.Weights(sd)
    obs = obs_from_states(z["states"])
    err = lambda l, v: max(te.rel_err(l, z["logits"]), te.rel_err(v, z["values"]))
    model = {t: err(*te.tc_forward(w, obs, terms=t)) for t in range(8)}
    for (g1, g2), t in {(1, 1): 0, (2, 1): 1, (1, 2): 2, (2, 2): 3, (1, 3): 6, (2, 3): 7}.items():
        ref = err(*script.run("f16", g1, g2, sd, obs))
        assert ref / 2 - 2e-6 <= model[t] <= 2 * ref + 2e-6, (t, model[t], ref)
    assert 1e-6 < model[7] <= 1.1e-5
    assert model[3] <= 1e-3 and err(*te.engine_forward(w, "f16f8c", obs)[:2]) <= 1e-3
    for t in (0, 1, 2, 4, 5, 6):
        assert model[t] > 1e-3, (t, model[t])


def test_f8c_h1_ceiling():
    """f16f8c carries 16 h1 (H1_SCALE8) as an fp16 hi rounded toward zero plus an e5m2 residue.  Up to h1 = 4094 the hi
    holds it and the residue keeps the f16x2w16 grade (2^-13 of h1); above, the hi sits at 65504 and the 2-bit residue
    carries the excess (1/8 of it); from h1 = 7678 on both saturate."""
    h = np.array([1.0, 100.0, 4000.0, 4094.0, 4095.0, 5000.0, 7000.0, 7678.0, 8000.0, 1e5], np.float32)
    x = h * te.H1_SCALE8
    hi = te.fp16_rz(x)
    h1 = (hi.astype(np.float64) + te.e5m2(te.relu(x - hi))) / 16
    grade = h <= te.F8C_H1_GRADE
    assert np.all(np.abs(h1 - h)[grade] <= 2.0 ** -13 * h[grade])
    assert np.all(hi[~grade] == 65504)
    mid = ~grade & (h <= te.F8C_H1_MAX)
    assert np.all(np.abs(h1 - h)[mid] <= (h[mid] - te.F8C_H1_GRADE) / 8) and (np.abs(h1 - h)[mid] > 2.0 ** -13 * h[mid]).any()
    assert np.all(h1[h > te.F8C_H1_MAX] == te.F8C_H1_MAX)
