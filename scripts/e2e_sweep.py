"""End-to-end (host-buffer) collect rate of twr_ppo_collect_host under different sub-batch splits, next to the plain
pinned D2H rate of the same bytes.  GPU box only:  python scripts/e2e_sweep.py [precision]"""
import ctypes as C
import os
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch  # noqa: E402

import bench  # noqa: E402
import twisterl_b200 as tw  # noqa: E402
from twisterl_b200 import _lib, collector as twc, nn as twn  # noqa: E402

precision = sys.argv[1] if len(sys.argv) > 1 else "f16x2w16"
E = 65536
sd = bench.synth_weights()
eng = tw.Engine(device=0, precision=precision, seed=0x5EED5EED)
pol = twn.Policy(twn.EmbeddingBag(sd["embeddings.weight"].T, sd["embeddings.bias"], True, [256], 0),
                 twn.Sequential([twn.Linear(sd["common.0.weight"].T.flatten(), sd["common.0.bias"], True)]),
                 twn.Sequential([twn.Linear(sd["action.0.weight"].T.flatten(), sd["action.0.bias"], False)]),
                 twn.Sequential([twn.Linear(sd["value.0.weight"].T.flatten(), sd["value.0.bias"], False)]), [], [])
env = tw.env.Puzzle(4, 4, 128, 2, 256)
L = _lib.load()
spec = tw.env.spec_from_env(env)
cap = int(L.twr_max_records(C.byref(spec), E))
hb, arrs, keep = twc._host_buffers(cap, 16, 4, E, pinned=True, obs_u8=True)
desc = pol.desc()
hpol = pol.device_handle(eng)
out = _lib.Collected()

# plain pinned D2H rate
src = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
dst = torch.empty(512 << 20, dtype=torch.uint8).pin_memory()
for _ in range(2):
    dst.copy_(src, non_blocking=True); torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(4):
    dst.copy_(src, non_blocking=True)
torch.cuda.synchronize()
print("pinned D2H: %.1f GB/s" % (4 * src.numel() / (time.perf_counter() - t0) / 1e9), flush=True)

R1 = 18944
cands = [None, "37888,27648", "18944,27648,18944", "18944,18944,27648", "27648,18944,18944", "18944,18944,18944,8704", "9472,28416,27648",
         "18944,37888,8704", "14208,23680,27648", "18944,23296,23296"]
for parts in cands:
    os.environ.pop("TWISTERL_B200_E2E_PARTS", None)
    if parts: os.environ["TWISTERL_B200_E2E_PARTS"] = parts
    for _ in range(2):
        _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), hpol, C.byref(desc), E, 0.995, 0.995, C.byref(hb), C.byref(out)))
    t0 = time.perf_counter(); n = 0
    for _ in range(6):
        _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), hpol, C.byref(desc), E, 0.995, 0.995, C.byref(hb), C.byref(out)))
        n += int(out.n_records)
    dt = time.perf_counter() - t0
    print(f"parts={parts or 'default':28s}  {n / dt:.4g} env-steps/s  {1e3 * dt / 6:.2f} ms/call", flush=True)
