"""Collect rates of GridWorld boards above 5x5 on one card.  PPO: 262 144 episodes (bench.py's gridworld_ppo size), max_steps
64, difficulty 10, synthetic weights of gridworld_ppo's shape (E 512, H 128), on the fp32 and f16f8c engines, for 5x5
(the anchor: the same workload as bench.py's gridworld_ppo extra), 6x6 and 8x8.  Boards above 32 cells run their
N*N-row table as the compact table of the 4N reachable rows: the pair kernel on f16f8c, the fp32 kernel's compact mode
on fp32.  AlphaZero: 512 episodes of 8x8 at 100 simulations per record (max_steps 32, difficulty 6).  Reported per case,
medians over the timed iterations:
  env_steps_per_s / records_per_s   records of a device-resident collect (collect_device, which returns after its
                                    stream synchronise) per second of wall clock
  launches_per_collect              kernels launched by one collect (twr_engine_launch_count delta)
  records                           records of one collect
and the card name and its power limit, read in the same run.

    python scripts/grid_world_rate.py [--iters 5] [--warmup 2] [--episodes 262144] [--out grid_world_rate.json]
"""
import argparse
import json
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


def _time(eng, collect, iters, warmup):
    rates, launches, records = [], [], 0
    for it in range(warmup + iters):
        l0 = eng.launch_count()
        t0 = time.perf_counter()
        c = collect()
        dt = time.perf_counter() - t0
        if it >= warmup:
            records = int(c.n_records)
            rates.append(records / dt)
            launches.append(eng.launch_count() - l0)
    return statistics.median(rates), int(statistics.median(launches)), records


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--episodes", type=int, default=262144)
    ap.add_argument("--az-episodes", type=int, default=512)
    ap.add_argument("--az-sims", type=int, default=100)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import bench
    import twisterl_b200 as tw
    from twisterl_b200 import nn as twn

    gpu, power = _card()
    rows = []
    for side in (5, 6, 8):
        N = side * side
        sd = bench.synth_weights(obs_size=N * N, hidden=128)
        for precision in ("fp32", "f16f8c"):
            eng = tw.Engine(device=0, precision=precision, seed=0x5EED5EED)
            pol = bench.synth_policy(twn, sd, N * N)
            env = tw.env.GridWorld(side, side, 64, 10)
            col = tw.collector.PPOCollector(args.episodes, 0.995, 0.995, 32, engine=eng)
            rate, launches, records = _time(eng, lambda: col.collect_device(env, pol), args.iters, args.warmup)
            row = dict(kind="ppo", board=f"{side}x{side}", precision=precision, episodes=args.episodes,
                       env_steps_per_s=rate, launches_per_collect=launches, records=records)
            print(json.dumps(row), flush=True)
            rows.append(row)
            if side == 8:
                az = tw.collector.AZCollector(args.az_episodes, args.az_sims, 1.41, 1, 32, engine=eng)
                az_env = tw.env.GridWorld(8, 8, 32, 6)
                rate, launches, records = _time(eng, lambda: az.collect_device(az_env, pol), max(1, args.iters // 2), 1)
                row = dict(kind="az", board="8x8", precision=precision, episodes=args.az_episodes, sims=args.az_sims,
                           records_per_s=rate, launches_per_collect=launches, records=records)
                print(json.dumps(row), flush=True)
                rows.append(row)
            pol.release()
            eng.close()
    out = dict(gpu=gpu, power_limit_w=power, rows=rows)
    print(json.dumps(dict(gpu=gpu, power_limit_w=power)))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
