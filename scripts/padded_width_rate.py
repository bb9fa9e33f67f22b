"""Tensor-core forward at embedding widths that are an odd number of 128-feature chunks (E = 128, 384; H = 256), which
the CTA-pair kernel runs zero-padded to the next chunk pair.

    python scripts/padded_width_rate.py [--envs 65536] [--precisions f16f8c,f16x2] [--repeats 10]

Per (precision, E): device time of one 65 536-env PPO collect on puzzle15 (difficulty 128, horizon 256; device events
around the whole collect, twr_engine_last_timing), and host time of one forward_batch over 65 536 scrambled envs
(twr_policy_forward: upload of the twist indices, one forward launch, copy-out of logits and values, synchronise).
Both are the median of --repeats calls after three warm-up calls.  With TWISTERL_B200_LIB two builds can be compared
on the same box.  GPU box only.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:                     # the number is then reported as unknown, not guessed
        out = f"unknown ({exc})"
    return name, out or "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--precisions", default="f16f8c,f16x2")
    ap.add_argument("--repeats", type=int, default=10)
    args = ap.parse_args()
    import bench
    import twisterl_b200 as tw
    from helpers import scramble_states
    from twisterl_b200 import collector as twc, nn as twn
    from twisterl_b200.env import EnvBatch

    name, power = gpu_info()
    print(f"# {name}, power limit {power}; library {os.environ.get('TWISTERL_B200_LIB') or 'in-tree build'}")
    st = scramble_states(np.random.default_rng(1), args.envs, 4, 4, 60)
    perm = np.full(args.envs, -1, dtype=np.int32)
    for precision in args.precisions.split(","):
        for E in (128, 384):
            eng = tw.Engine(device=0, precision=precision, seed=0x5EED5EED)
            pol = bench.synth_policy(twn, bench.synth_weights(0, 256, E, 256), 256)
            env = tw.env.Puzzle(4, 4, 128, 2, 256)
            col = twc.PPOCollector(args.envs, 0.995, 0.995, 32, engine=eng)
            eng.set_timing(True)
            coll = []
            for i in range(3 + args.repeats):
                c = col.collect_device(env, pol)
                if i >= 3:
                    coll.append(eng.last_timing()[1])
            eng.set_timing(False)
            b = EnvBatch(tw.env.spec_from_env(env), args.envs, eng)
            b.set_state(st)
            fwd = []
            for i in range(3 + args.repeats):
                t0 = time.perf_counter()
                twn.forward_batch(eng, pol, b, perm_idx=perm)
                if i >= 3:
                    fwd.append((time.perf_counter() - t0) * 1e3)
            print(f"{precision:7s} E={E:4d} H=256: collect {np.median(coll):8.2f} ms ({c.n_records} records), "
                  f"forward_batch {np.median(fwd):6.3f} ms", flush=True)
            b.close()
            pol.release()
            eng.close()


if __name__ == "__main__":
    main()
