"""Cost of gathering every rank's collect to the trainer rank (twr_gather_collected) at the headline shape: puzzle15,
65 536 episodes per rank, difficulty 128, f16f8c, synthetic weights (bench.py's).  One process per GPU, spawned here.

Per iteration every rank collects its shard (device-resident) and all ranks meet in an all-reduce; then rank 0's clock
times the gather alone.  Reported per W, medians over the timed iterations:
  collect_ms         collect time, max over ranks
  gather_ms          the gather on rank 0, from the all-reduce that follows the slowest collect to its merged result
  bytes_received     bytes that arrive over NCCL on rank 0 (every other rank's records and episode lengths)
  gbps               bytes_received / gather_ms
  records_per_s      records of the merged result / (collect_ms + gather_ms): what the trainer rank receives per second
  gpu, power_limit_w read on rank 0 in the same run

    python scripts/gather_rate.py [--worlds 2,4,8] [--iters 10] [--warmup 3] [--episodes 65536] [--difficulty 128]
"""
import argparse
import json
import os
import queue
import socket
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def _record_bytes(cells, actions):
    return 2 * cells + 4 * actions + 4 * 4 + 1 + 1      # obs u16, logits, values / rewards / advs / rets, action, perm


def _rank(rank, world, port, args, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import bench
    import twisterl_b200 as tw
    from twisterl_b200 import dist as twd, nn as twn
    eng = tw.Engine(device=rank, precision="f16f8c", seed=0x5EED5EED, rank=rank, world=world)
    comm = twd.Comm(eng)
    pol = bench.synth_policy(twn, bench.synth_weights(), 256)
    env = tw.env.Puzzle(4, 4, args.difficulty, 2, 256)
    col = tw.collector.PPOCollector(args.episodes, 0.995, 0.995, 32, engine=eng)
    rows = []
    for it in range(args.warmup + args.iters):
        t0 = time.perf_counter()
        own = col.collect_device(env, pol)               # returns after the collect's stream synchronise
        t1 = time.perf_counter()
        collect_ms = comm.max_over_ranks((t1 - t0) * 1e3)
        t2 = time.perf_counter()
        c = comm.gather_collected(0)
        t3 = time.perf_counter()
        if it >= args.warmup:
            rows.append(dict(collect_ms=collect_ms, gather_ms=(t3 - t2) * 1e3, records=int(c.n_records),
                             own_records=int(own.n_records)))
    if rank == 0:
        import torch
        try:
            power = subprocess.run(["nvidia-smi", "-i", str(rank), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=60).stdout.strip()
        except Exception as exc:                        # noqa: BLE001 -- reported, not fatal
            power = f"unavailable ({exc})"
        rb = _record_bytes(16, 4)
        med = lambda k: statistics.median(r[k] for r in rows)
        recv = statistics.median((r["records"] - r["own_records"]) * rb + (world - 1) * args.episodes * 4 for r in rows)
        out = dict(world=world, episodes_per_rank=args.episodes, difficulty=args.difficulty, precision="f16f8c",
                   iters=args.iters, collect_ms=med("collect_ms"), gather_ms=med("gather_ms"),
                   records=int(med("records")), bytes_received=int(recv), merged_bytes=int(med("records") * rb + world * args.episodes * 4),
                   gpu=torch.cuda.get_device_name(rank), power_limit_w=power)
        out["gbps"] = out["bytes_received"] / (out["gather_ms"] * 1e-3) / 1e9
        out["records_per_s"] = out["records"] / ((out["collect_ms"] + out["gather_ms"]) * 1e-3)
        q.put(out)
    pol.release()
    comm.close()
    eng.close()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", default="2,4,8")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--episodes", type=int, default=65536)
    ap.add_argument("--difficulty", type=int, default=128)
    args = ap.parse_args()
    import torch
    import torch.multiprocessing as mp
    n = torch.cuda.device_count()
    if n < 2:
        sys.exit(f"gather_rate.py needs at least 2 GPUs, found {n}")
    ctx = mp.get_context("spawn")
    for world in (int(w) for w in args.worlds.split(",")):
        if world > n:
            print(json.dumps(dict(world=world, skipped=f"{n} GPUs")), flush=True)
            continue
        q = ctx.Queue()
        port = _free_port()
        procs = [ctx.Process(target=_rank, args=(r, world, port, args, q)) for r in range(world)]
        for p in procs:
            p.start()
        res, deadline = None, time.time() + 900
        try:
            while res is None and time.time() < deadline and not any(p.exitcode not in (None, 0) for p in procs):
                try:
                    res = q.get(timeout=5)
                except queue.Empty:
                    pass
            if res is not None:
                print(json.dumps(res), flush=True)
        finally:
            for p in procs:
                p.join(timeout=120)
                if p.is_alive():
                    p.terminate()
                    p.join()
        if any(p.exitcode != 0 for p in procs):
            sys.exit(f"W={world}: a rank failed ({[p.exitcode for p in procs]})")


if __name__ == "__main__":
    main()
