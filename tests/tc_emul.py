"""Exact CPU model of the operands of the tensor-core forward (k_forward_tc2, twisterl_b200/csrc/twr_forward_tc2.cu).

Every operand is rounded exactly as the kernel rounds it (k_tc2_pack / k_tc2_pack8 for the weights, split2 / split4 in
epilogue-1 for the hidden activations), and the products are then accumulated in float64.  What separates the kernel
from this model is only the order and precision of its fp32 tensor-core accumulation and of its fp32 heads -- orders of
magnitude below a dropped, misplaced or wrongly scaled term.  The launch-time choice of `launch_forward_tc2` (which
terms, fp8 or fp16 corrections, bias folded into the fp8 image or not) is modelled by `dispatch`.

Also here: the plain float64 forward of the policy (`forward64`) and the magnitude forward S (`magnitude`), the same
float64 chain over |weights|, |biases| and |activations|: the sum of |summand| each output is built from, which is the
normaliser of the kernel-vs-model measure.

Weights are a BasicPolicy state dict (tests/helpers.py: synth_state_dict); observations are rows of sparse one-hot
indices (what EnvBatch.observe() returns), twists the (obs_perms, act_perms) of nn.Policy."""
from __future__ import annotations

import math

import numpy as np

H1_SCALE8 = np.float32(16.0)            # twr_forward_tc2.cu: H1_SCALE8, TABLE8_SCALE, W8_SCALE, ONE8
TABLE8_SCALE = np.float32(1024.0)
W8_SCALE = np.float32(1.0 / 16.0)
ONE8 = 2.0 ** -10
E4M3_MAX, E5M2_MAX = 448.0, 57344.0
# f16f8c carries 16 h1 as fp16 hi + e5m2 residue: hi saturates at 65504 (cvt.rz.relu), so above h1 = 4094 the 2-bit
# residue carries the excess, and above (65504 + 57344) / 16 = 7678 the residue saturates too
F8C_H1_GRADE, F8C_H1_MAX = 65504.0 / 16.0, (65504.0 + E5M2_MAX) / 16.0


# ------------------------------------------------------------------------------------------------- roundings ---
def fp16_rn(x):
    """float32 -> fp16 (round to nearest even) -> float32: __float2half_rn, cvt.rn.f16x2.f32."""
    with np.errstate(over="ignore"):
        return np.asarray(x, np.float32).astype(np.float16).astype(np.float32)


def fp16_rz(x):
    """float32 -> fp16 rounded toward zero -> float32 (cvt.rz.f16x2.f32; saturates at +-65504 instead of overflowing):
    round to nearest, then one step toward zero wherever that grew the magnitude."""
    x = np.asarray(x, np.float32)
    with np.errstate(over="ignore"):
        h = x.astype(np.float16)
    grew = np.abs(h.astype(np.float32)) > np.abs(x)
    return np.where(grew, np.nextafter(h, np.float16(0)), h).astype(np.float32)


def _fp8(x, mbits, emin, maxv):
    # round to nearest even on a grid of `mbits` mantissa bits, subnormals below 2^emin; values beyond the largest
    # finite one saturate (the kernel converts with __NV_SATFINITE / .satfinite)
    x = np.asarray(x, np.float32).astype(np.float64)
    a = np.minimum(np.abs(x), maxv)
    _, ex = np.frexp(a)
    e = np.maximum(ex.astype(np.float64) - 1, emin)
    q = np.exp2(e - mbits)
    return (np.sign(x) * np.minimum(np.round(a / q) * q, maxv)).astype(np.float32)


def e4m3(x):
    """float32 -> e4m3 (fn: no infinities, max 448) round to nearest even, satfinite -> float32."""
    return _fp8(x, 3, -6, E4M3_MAX)


def e5m2(x):
    """float32 -> e5m2 (max finite 57344) round to nearest even, satfinite -> float32."""
    return _fp8(x, 2, -14, E5M2_MAX)


def relu(x):
    return np.maximum(x, 0).astype(np.asarray(x).dtype)


# ------------------------------------------------------------------------------------------------ the policy ---
class Weights:
    """A BasicPolicy state dict in the kernel's layouts, float32: table T [obs_size][E], bias b [E], W1 [E][H], b1 [H],
    action head Wa [H][A], ba [A], value head wv [H], bv."""

    def __init__(self, sd):
        f = lambda k: np.ascontiguousarray(sd[k], dtype=np.float32)
        self.T, self.b = f("embeddings.weight").T.copy(), f("embeddings.bias")
        self.W, self.b1 = f("common.0.weight").T.copy(), f("common.0.bias")
        self.Wa, self.ba = f("action.0.weight").T.copy(), f("action.0.bias")
        self.wv, self.bv = f("value.0.weight")[0].copy(), f("value.0.bias")
        self.obs_size, self.E = self.T.shape
        self.H, self.A = self.Wa.shape


def fold_block(obs_size, obs_perms=()):
    """PolicyDev::tc_fold (twr_engine.cu fold_block): N when obs_size = N * N and every twist maps each block of N rows
    onto another block, all blocks hit once; else 0.  Non-zero: the f16f8c image carries the embedding bias on block 0."""
    N = math.isqrt(obs_size)
    if N * N != obs_size or N > 32:
        return 0
    for pm in np.asarray(obs_perms, np.int64).reshape(-1, obs_size) if len(obs_perms) else ():
        tb = pm.reshape(N, N) // N
        if (tb != tb[:, :1]).any() or sorted(tb[:, 0].tolist()) != list(range(N)):
            return 0
    return N


def one_per_block(obs, fold):
    """twr_policy_forward_obs: does every row hold exactly one index of each block of `fold` rows?"""
    obs = np.asarray(obs, np.int64)
    if fold <= 0 or obs.shape[1] != fold:
        return False
    return all(sorted((r // fold).tolist()) == list(range(fold)) for r in obs)


def dispatch(tc_terms, tc_fold, blocks):
    """launch_forward_tc2's choice for ForwardArgs::tc_terms (0 = the f16x2 engine, 8|3 = f16x2w16, 16|8|3 = f16f8c,
    8|t after set_tc_terms(t)): (terms, f8, fold).  fp8 corrections exist for the terms of f16x2w16 only, and a policy
    whose fp8 image carries the folded bias uses it only for observations with one index per block."""
    terms = (tc_terms & 7) if tc_terms else 7
    f8 = bool(tc_terms & 16) and terms == 3 and (tc_fold == 0 or blocks)
    return terms, f8, (tc_fold if f8 and tc_fold > 0 else 0)


ENGINE_TERMS = {"f16x2": 0, "f16x2w16": 8 | 3, "f16f8c": 16 | 8 | 3}      # twr_engine.cu terms_of_precision


def twisted(obs, perm, obs_perms):
    """Twist-in (policy.rs:81-83): row r of an observation under twist p reads table row obs_perms[p][r]."""
    obs = np.asarray(obs, np.int64)
    if perm is None or len(obs_perms) == 0:
        return obs
    op = np.asarray(obs_perms, np.int64)
    perm = np.asarray(perm, np.int64)
    out = obs.copy()
    tw = perm >= 0
    out[tw] = op[perm[tw][:, None], obs[tw]]
    return out


def twist_out(logits, perm, act_perms):
    """Twist-out (policy.rs:95-97): output o of twist p is logit act_perms[p][o]."""
    if perm is None or len(act_perms) == 0:
        return logits
    ap = np.asarray(act_perms, np.int64)
    perm = np.asarray(perm, np.int64)
    out = logits.copy()
    tw = perm >= 0
    out[tw] = np.take_along_axis(logits[tw], ap[perm[tw]], axis=1)
    return out


def _heads(w, h2):
    return h2 @ w.Wa.astype(np.float64) + w.ba, h2 @ w.wv.astype(np.float64) + w.bv[0]


def _rows(n, chunk=4096):
    for s in range(0, n, chunk):
        yield slice(s, min(n, s + chunk))


def forward64(w, obs, perm=None, obs_perms=(), act_perms=()):
    """Policy::_raw_predict in float64 on the float32 weights: (logits [n][A], values [n])."""
    rows = twisted(obs, perm, obs_perms)
    T = w.T.astype(np.float64)
    L, V = np.zeros((len(rows), w.A)), np.zeros(len(rows))
    for s in _rows(len(rows)):
        h1 = np.maximum(T[rows[s]].sum(1) + w.b, 0)
        h2 = np.maximum(h1 @ w.W.astype(np.float64) + w.b1, 0)
        L[s], V[s] = _heads(w, h2)
    return twist_out(L, perm, act_perms), V


def magnitude(w, obs, perm=None, obs_perms=(), act_perms=()):
    """S: the float64 forward over |weights|, |biases| and |activations| -- per output, the sum of the magnitudes of
    everything it is built from.  (logits [n][A], values [n])"""
    rows = twisted(obs, perm, obs_perms)
    T = np.abs(w.T.astype(np.float64))
    L, V = np.zeros((len(rows), w.A)), np.zeros(len(rows))
    for s in _rows(len(rows)):
        h1 = T[rows[s]].sum(1) + np.abs(w.b)
        h2 = h1 @ np.abs(w.W.astype(np.float64)) + np.abs(w.b1)
        L[s] = h2 @ np.abs(w.Wa.astype(np.float64)) + np.abs(w.ba)
        V[s] = h2 @ np.abs(w.wv.astype(np.float64)) + abs(float(w.bv[0]))
    return twist_out(L, perm, act_perms), V


class Operands:
    """The weight operands of one (terms, f8, fold) launch, as k_tc2_pack / k_tc2_pack8 write them."""

    def __init__(self, w, terms, f8=False, fold=0):
        self.terms, self.f8, self.fold = terms, f8, fold
        if f8:
            # (table + bias on the rows of block 0) * 16 in fp32; fp16 hi, and the residue as e4m3(residue * 2^10)
            # times the one-hot value 2^-10
            k = np.arange(w.obs_size)[:, None]
            x = np.where(k < fold, w.T + w.b, w.T).astype(np.float32) * H1_SCALE8
            hi = fp16_rn(x)
            self.g1 = hi.astype(np.float64) + e4m3((x - hi) * TABLE8_SCALE).astype(np.float64) * ONE8
            ws = w.W * W8_SCALE
            self.w_hi, self.w_lo = fp16_rn(ws).astype(np.float64), e5m2(ws).astype(np.float64)
            self.bias = np.zeros(w.E, np.float32) if fold else w.b * H1_SCALE8
        else:
            hi = fp16_rn(w.T)
            self.g1 = hi.astype(np.float64) + (fp16_rn(w.T - hi).astype(np.float64) if terms & 1 else 0.0)
            whi = fp16_rn(w.W)
            self.w_hi = whi.astype(np.float64)
            self.w_lo = fp16_rn(w.W - whi).astype(np.float64) if terms & 4 else None
            self.bias = w.b

    def h1(self, d1):
        """epilogue-1: x = D1 + bias in fp32, split into the GEMM2 A operands (hi, correction or None)."""
        x = (d1 + self.bias).astype(np.float32)
        if self.f8:                                                 # split4
            hi = fp16_rz(relu(x))
            return hi.astype(np.float64), e5m2(relu(x - hi)).astype(np.float64)
        if self.terms & 2:                                          # split2 with the residue
            hi = fp16_rz(relu(x))
            return hi.astype(np.float64), fp16_rn(relu(x - hi)).astype(np.float64)
        return fp16_rn(relu(x)).astype(np.float64), None

    def d2(self, hi, lo):
        d = hi @ self.w_hi
        if lo is not None:
            d += lo @ (self.w_lo if self.f8 else self.w_hi)
        if not self.f8 and self.w_lo is not None:
            d += hi @ self.w_lo
        return d


def tc_forward(w, obs, perm=None, obs_perms=(), act_perms=(), terms=7, f8=False, fold=0, ops=None):
    """The model of one k_forward_tc2 launch: (logits [n][A], values [n]).  `ops` reuses the Operands of (terms, f8,
    fold) across calls."""
    ops = ops or Operands(w, terms, f8, fold)
    rows = twisted(obs, perm, obs_perms)
    L, V = np.zeros((len(rows), w.A)), np.zeros(len(rows))
    for s in _rows(len(rows)):
        d1 = ops.g1[rows[s]].sum(1)
        h2 = np.maximum(ops.d2(*ops.h1(d1)) + w.b1, 0)
        L[s], V[s] = _heads(w, h2)
    return twist_out(L, perm, act_perms), V


def engine_forward(w, precision, obs, perm=None, obs_perms=(), act_perms=(), tc_terms=None, obs_rows=False):
    """What an engine of `precision` computes for `obs` through the pair kernel (or, for "fp32", the SIMT kernel,
    modelled as the float64 forward).  tc_terms overrides the engine's ForwardArgs::tc_terms (set_tc_terms(t) = 8 | t).
    obs_rows: the rows come through twr_policy_forward_obs (host check of one index per block) instead of an env.
    Returns (logits, values, (terms, f8, fold))."""
    if precision == "fp32" and tc_terms is None:
        return (*forward64(w, obs, perm, obs_perms, act_perms), None)
    cfg = ENGINE_TERMS[precision] if tc_terms is None else tc_terms
    fold = fold_block(w.obs_size, obs_perms)
    blocks = one_per_block(obs, fold) if obs_rows else fold > 0 and np.asarray(obs).shape[1] == fold
    d = dispatch(cfg, fold, blocks)
    return (*tc_forward(w, obs, perm, obs_perms, act_perms, *d), d)


def rel_to_s(out, model, s):
    """max |out - model| / S over all outputs."""
    return float((np.abs(np.asarray(out, np.float64) - model) / s).max(initial=0.0))


def rel_err(out, ref):
    """The suite's usual measure: max |d| / max(1, |ref|)."""
    return float((np.abs(np.asarray(out, np.float64) - ref) / np.maximum(1.0, np.abs(ref))).max(initial=0.0))
