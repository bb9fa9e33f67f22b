"""Shared test helpers: seeded synthetic weights, twist sets, fixtures, and where to find a checkout of the reference."""
from __future__ import annotations

import json
import os
from pathlib import Path

import numpy as np

GOLDEN = Path(__file__).resolve().parent / "golden"
STAGED_REFERENCE = Path(__file__).resolve().parent.parent / "oracle" / "_ref" / "reference"


def reference_checkout() -> Path | None:
    """A checkout of the reference, AI4quantum/twisteRL: $TWISTERL_REFERENCE, else a copy staged under the git-ignored
    oracle/_ref/reference; None when neither holds one."""
    for cand in (os.environ.get("TWISTERL_REFERENCE"), STAGED_REFERENCE):
        if cand and (Path(cand) / "src" / "twisterl" / "rl" / "ppo.py").is_file():
            return Path(cand)
    return None


def synth_state_dict(seed, obs_size, emb, hidden, n_act):
    """Seeded N(0, 0.05^2) weights, small uniform biases (same generator as gen_golden.py)."""
    g = np.random.default_rng(seed)
    f = lambda *s: (g.standard_normal(s) * 0.05).astype(np.float32)
    b = lambda n: g.uniform(-0.05, 0.05, size=n).astype(np.float32)
    return {"embeddings.weight": f(emb, obs_size), "embeddings.bias": b(emb),
            "common.0.weight": f(hidden, emb), "common.0.bias": b(hidden),
            "action.0.weight": f(n_act, hidden), "action.0.bias": b(n_act),
            "value.0.weight": f(1, hidden), "value.0.bias": b(1)}


def synth_conv_state_dict(seed, n_in, v, emb, hidden, n_act):
    """Seeded weights of a Conv1dPolicy (src/twisterl/nn/policy.py:205-266): conv kernel [v, n_in, 1] without bias
    (larger scale than the Linear embedding: only N vectors are summed into each slice)."""
    g = np.random.default_rng(seed)
    f = lambda sc, *s: (g.standard_normal(s) * sc).astype(np.float32)
    b = lambda n: g.uniform(-0.05, 0.05, size=n).astype(np.float32)
    return {"conv_layer.weight": f(0.2, v, n_in, 1),
            "common.0.weight": f(0.05, hidden, emb), "common.0.bias": b(hidden),
            "action.0.weight": f(0.05, n_act, hidden), "action.0.bias": b(n_act),
            "value.0.weight": f(0.05, 1, hidden), "value.0.bias": b(1)}


def synth_deep_state_dict(seed, obs_size, emb, common, policy, value, n_act):
    """Seeded weights of a BasicPolicy with deeper stacks (common_layers=common, policy_layers=policy,
    value_layers=value): torch Sequential indices 0, 2, 4, .. (a ReLU sits between the Linears)."""
    g = np.random.default_rng(seed)
    f = lambda *s: (g.standard_normal(s) * 0.08).astype(np.float32)
    b = lambda n: g.uniform(-0.05, 0.05, size=n).astype(np.float32)
    sd = {"embeddings.weight": f(emb, obs_size), "embeddings.bias": b(emb)}
    width = emb
    for k, w in enumerate(common):
        sd[f"common.{2 * k}.weight"], sd[f"common.{2 * k}.bias"] = f(w, width), b(w)
        width = w
    for name, layers, last in (("action", policy, n_act), ("value", value, 1)):
        wd = width
        for k, w in enumerate(tuple(layers) + (last,)):
            sd[f"{name}.{2 * k}.weight"], sd[f"{name}.{2 * k}.bias"] = f(w, wd), b(w)
            wd = w
    return sd


def transpose_twists(w):
    """{identity, main-diagonal transpose} twist set for a square w x w puzzle (SURVEY.md 8a row T)."""
    N = w * w
    T = [(i % w) * w + (i // w) for i in range(N)]
    ident = list(range(N * N))
    tw = [0] * (N * N)
    for i in range(N):
        for v in range(N):
            tw[i * N + v] = T[i] * N + T[v]
    return [ident, tw], [[0, 1, 2, 3], [1, 0, 3, 2]]


def gridworld_transpose_twists(w):
    """{identity, main-diagonal transpose} twist set of a square w x w GridWorld (examples/grid_world/src/lib.rs): the cell
    values (empty / agent / goal / trap) keep their meaning, cells move to their transposed position and up<->left,
    down<->right trade places (actions 0 up, 1 down, 2 left, 3 right, lib.rs:127-136)."""
    N = w * w
    T = [(i % w) * w + (i // w) for i in range(N)]
    ident = list(range(N * N))
    tw = [0] * (N * N)
    for i in range(N):
        for v in range(N):
            tw[i * N + v] = T[i] * N + v
    return [ident, tw], [[0, 1, 2, 3], [2, 3, 0, 1]]


def trained15():
    z = np.load(GOLDEN / "policy15_trained.npz")
    sd = {k[2:]: z[k] for k in z.files if k.startswith("w.")}
    return z, sd


def replays():
    return json.loads((GOLDEN / "puzzle_replays.json").read_text())


def obs_from_states(states):
    """u8 board [n, N] -> sparse one-hot indices [n, N] (envs/puzzle.rs:183-185)."""
    s = np.asarray(states).astype(np.int32)
    N = s.shape[1]
    return np.arange(N, dtype=np.int32)[None, :] * N + s


def scramble_states(rng, n, w, h, max_moves):
    N = w * h
    states = np.zeros((n, N), dtype=np.uint8)
    for k in range(n):
        s = list(range(N)); z = 0
        for a in rng.integers(0, 4, size=int(rng.integers(0, max_moves + 1))):
            x, y = z % w, z // w
            if a == 0 and x > 0: t = z - 1
            elif a == 1 and y > 0: t = z - w
            elif a == 2 and x < w - 1: t = z + 1
            elif a == 3 and y < h - 1: t = z + w
            else: continue
            s[z] = s[t]; s[t] = 0; z = t
        states[k] = s
    return states
