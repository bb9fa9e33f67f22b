"""PPO collect rate of the wide Puzzle boards (5x5, the 24-puzzle, and 4x5) on one card: 65 536 episodes, difficulty 64
and 128 (depth_slope 2, max_depth 256), synthetic weights of bench.py's shape (E 512, H 256), on the fp32 and f16x2
engines.  These boards hold 5-bit cells in the 128-bit env state and their 625- / 400-row tables run the fp32 SIMT
forward on every engine.  Reported per case, medians over the timed iterations:
  env_steps_per_s      records of a device-resident collect (collect_device, which returns after its stream synchronise)
                       per second of wall clock
  launches_per_collect kernels launched by one collect (twr_engine_launch_count delta; the forward is one launch a step)
  records              records of one collect
and once: the oracle collector's rate on all host threads (orc.time_ppo_collect, a C restatement of the reference's
collector) on the same workload, the card name and its power limit, read in the same run.

    python scripts/wide_puzzle_rate.py [--iters 5] [--warmup 2] [--episodes 65536] [--out wide_puzzle_rate.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def _card():
    import torch
    try:
        power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as exc:                        # noqa: BLE001 -- reported, not fatal
        power = f"unavailable ({exc})"
    return torch.cuda.get_device_name(0), power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--episodes", type=int, default=65536)
    ap.add_argument("--oracle-episodes", type=int, default=2048)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import bench
    import twisterl_b200 as tw
    from oracle import orc
    from twisterl_b200 import nn as twn

    gpu, power = _card()
    rows = []
    for w, h in ((5, 5), (4, 5)):
        N = w * h
        sd = bench.synth_weights(obs_size=N * N)
        for precision in ("fp32", "f16x2"):
            eng = tw.Engine(device=0, precision=precision, seed=0x5EED5EED)
            pol = bench.synth_policy(twn, sd, N * N)
            for difficulty in (64, 128):
                env = tw.env.Puzzle(w, h, difficulty, 2, 256)
                col = tw.collector.PPOCollector(args.episodes, 0.995, 0.995, 32, engine=eng)
                rates, launches, records = [], [], 0
                for it in range(args.warmup + args.iters):
                    l0 = eng.launch_count()
                    t0 = time.perf_counter()
                    c = col.collect_device(env, pol)
                    dt = time.perf_counter() - t0
                    if it >= args.warmup:
                        records = int(c.n_records)
                        rates.append(records / dt)
                        launches.append(eng.launch_count() - l0)
                row = dict(board=f"{w}x{h}", precision=precision, difficulty=difficulty, episodes=args.episodes,
                           env_steps_per_s=statistics.median(rates), launches_per_collect=int(statistics.median(launches)),
                           records=records)
                print(json.dumps(row), flush=True)
                rows.append(row)
            pol.release()
            eng.close()
    threads = os.cpu_count() or 1
    oracle = []
    for w, h in ((5, 5), (4, 5)):
        N = w * h
        opol = orc.Policy.from_torch_state_dict(bench.synth_weights(obs_size=N * N))
        for difficulty in (64, 128):
            n, dt = orc.time_ppo_collect(orc.puzzle_spec(w, h, difficulty, 2, 256), opol, args.oracle_episodes, 0.995, 0.995,
                                         0x5EED5EED, 0, threads)
            row = dict(board=f"{w}x{h}", difficulty=difficulty, episodes=args.oracle_episodes, threads=threads,
                       env_steps_per_s=n / dt)
            print(json.dumps(dict(oracle=row)), flush=True)
            oracle.append(row)
    out = dict(gpu=gpu, power_limit_w=power, device=rows, oracle=oracle)
    print(json.dumps(dict(gpu=gpu, power_limit_w=power)))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
