#!/usr/bin/env python
"""bench.py -- rollout env-steps/s including the policy forward, puzzle15 PPO (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp32|f16x2|f16x2w16|f16f8c] [--no-extras]
                  [--dump-outputs DIR]

One "step" = one PPOCollector.collect of `--episodes` (default 65 536) puzzle15 episodes per GPU at
difficulty 128 (<= 257 records each): reset, per-step policy forward + Gumbel-max sampling + env step +
trajectory write, GAE, compaction into the reference's CollectedData layout.  Under torchrun every rank
runs its own env shard (weak scaling); NCCL carries only the per-step weight broadcast and the stats
all-reduce, both made by the library itself through its C ABI (twisterl_b200/dist.py).  `--impl reference` times the
CPU restatement of the reference collector (oracle/) on the host cores -- the Rust binary cannot be built in this
image (no cargo).

The JSON line carries the headline workload (BASELINE.json configs[1]) at top level and, under "extra", one entry per
other BASELINE config: puzzle8 PPO, grid_world 5x5 PPO, AlphaZero on puzzle8 (100 simulations at 65 536 episodes and the
reference's default 512 episodes x 1000 simulations), puzzle15 with twists at 1 M envs in total -- each with its own
roofline and (at N = 1) cpu_baseline.

`--dump-outputs DIR` writes what the last timed headline step returned -- the records and per-episode lengths of rank 0's
collect in float32, their row indices and the collect's stats in float64 -- as DIR/<name>.npy.  Inputs are seeded, so the
same arguments give the same inputs on every run; a collect of more than 2^18 records or episodes is stored as a fixed
seeded sample of them.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

FLOP_PER_STEP = {"puzzle15": 272_896, "puzzle8": 269_312, "gridworld": 145_152}   # SURVEY.md section 8d
# what the tensor pipe executes per env-step: the embedding as a dense one-hot GEMM over the hi and the lo table, and the
# hidden layer as 3 (f16x2) or 2 (f16x2w16) split products
EXECUTED_TENSOR_FLOP_PER_STEP = {"f16x2": 2 * (2 * 256 * 512) + 3 * (2 * 512 * 256), "f16x2w16": 2 * (2 * 256 * 512) + 2 * (2 * 512 * 256)}
DTYPE = {"fp32": "f32",
         "f16x2": "f16x2 (tcgen05; every operand split into fp16 hi+lo, f32 accumulate; 1e-5-grade)",
         "f16x2w16": "f16x2w16 (tcgen05; table and activations split into fp16 hi+lo, common-layer weight one fp16 term, f32 accumulate; "
                     "7e-4 worst case on the shipped trained weights, bar 1e-3)",
         "f16f8c": "f16f8c (tcgen05; main products one-hot x table and h1 x W in fp16, their two correction products "
                   "(table residue, activation residue) as fp8 MMAs, f32 accumulate; same 1e-3 bar as f16x2w16, "
                   "tests/test_gpu_precision.py)"}
METRIC = "rollout env-steps/sec incl. policy fwd (puzzle15 PPO)"
UNIT = "env-steps/s"


def synth_weights(seed=0, obs_size=256, emb=512, hidden=256, n_act=4):
    g = np.random.default_rng(seed)
    f = lambda *s: (g.standard_normal(s) * 0.05).astype(np.float32)
    return {"embeddings.weight": f(emb, obs_size), "embeddings.bias": np.zeros(emb, np.float32),
            "common.0.weight": f(hidden, emb), "common.0.bias": np.zeros(hidden, np.float32),
            "action.0.weight": f(n_act, hidden), "action.0.bias": np.zeros(n_act, np.float32),
            "value.0.weight": f(1, hidden), "value.0.bias": np.zeros(1, np.float32)}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(bf16=d.get("bf16_tflops_sustained", 1410.7), hbm=d.get("hbm_gbs", 6546.2), src="measured")
    return dict(bf16=1400.0, hbm=6650.0, src="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        self._nv = self._h = None
        try:                                   # NVML is initialised here, outside the timed region
            import pynvml as nv
            nv.nvmlInit()
            self._nv, self._h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
        except Exception as exc:               # NVML missing: report it rather than fail the bench
            self.reasons.add(f"nvml_unavailable:{type(exc).__name__}")

    def run(self):
        nv, h = self._nv, self._h
        if nv is None:
            return
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        try:
            while not self._halt.is_set():     # the timed region can be as short as ~80 ms: sample every 5 ms
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                self._halt.wait(0.005)
        except Exception as exc:
            self.reasons.add(f"nvml_error:{type(exc).__name__}")

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------ reference arm ---
def oracle_policy(sd):
    from oracle import orc
    return orc.Policy.from_torch_state_dict(sd)


def cpu_collect_rate(sd, episodes, difficulty, threads, repeats=1):
    """records/s of the CPU restatement of PPOCollector::collect (oracle/twr_oracle.c)."""
    from oracle import orc
    spec = orc.puzzle_spec(4, 4, difficulty, 2, 256)
    pol = oracle_policy(sd)
    best = 0.0
    recs = 0
    for i in range(repeats):
        n, dt = orc.time_ppo_collect(spec, pol, episodes, 0.995, 0.995, 0x5EED5EED, i, threads)
        best = max(best, n / dt)
        recs = n
    return best, recs


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sd = synth_weights()
    episodes = args.ref_episodes
    for _ in range(args.warmup):
        cpu_collect_rate(sd, max(64, episodes // 8), args.difficulty, cores)
    t0 = time.perf_counter()
    total = 0
    from oracle import orc
    spec = orc.puzzle_spec(4, 4, args.difficulty, 2, 256)
    pol = oracle_policy(sd)
    for i in range(args.steps):
        n, _ = orc.time_ppo_collect(spec, pol, episodes, 0.995, 0.995, 0x5EED5EED, 100 + i, cores)
        total += n
    dt = time.perf_counter() - t0
    v = total / dt
    sample = f"{episodes} episodes/step of puzzle15 difficulty {args.difficulty} ({total} records in {dt:.2f}s)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"puzzle15 PPO rollout, {episodes} episodes/step (bounded sample of the 65536-env "
                               "config), CPU restatement of the reference Rust collector"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


# ------------------------------------------------------------------------ our arm ---
def synth_policy(twn, sd, obs_size, obs_perms=(), act_perms=()):
    return twn.Policy(twn.EmbeddingBag(sd["embeddings.weight"].T, sd["embeddings.bias"], True, [obs_size], 0),
                      twn.Sequential([twn.Linear(sd["common.0.weight"].T.flatten(), sd["common.0.bias"], True)]),
                      twn.Sequential([twn.Linear(sd["action.0.weight"].T.flatten(), sd["action.0.bias"], False)]),
                      twn.Sequential([twn.Linear(sd["value.0.weight"].T.flatten(), sd["value.0.bias"], False)]),
                      [list(p) for p in obs_perms], [list(p) for p in act_perms])


def puzzle15_twists():
    """{identity, main-diagonal transpose} twist set of SURVEY.md section 8a row T (BASELINE config 5)."""
    T = [(i % 4) * 4 + (i // 4) for i in range(16)]
    return [list(range(256)), [T[i] * 16 + T[v] for i in range(16) for v in range(16)]], [[0, 1, 2, 3], [1, 0, 3, 2]]


def executed_flop(precision, obs_k, emb, hidden):
    """tensor-pipe flop per env-step of the pair kernel: dense one-hot GEMM1 over the hi and lo table (K padded to 64) and
    2 (f16x2w16) or 3 (f16x2) split products of the common layer"""
    k = ((obs_k + 63) // 64) * 64
    if precision == "f16f8c":       # the two fp8 correction products run at twice the fp16 rate: counted at half, i.e. in
        k8 = ((obs_k + 127) // 128) * 128      # fp16-equivalent pipe work (what the bf16 roof is comparable with)
        return 2 * k * emb + (2 * k8 * emb) // 2 + 2 * emb * hidden + (2 * emb * hidden) // 2
    return 2 * (2 * k * emb) + (3 if precision == "f16x2" else 2) * (2 * emb * hidden)


class Timer:
    """CUDA events on the stream every kernel of the engine is launched on (torch's current stream)."""

    def __init__(self, torch, stream):
        self.torch, self.stream = torch, stream

    def __enter__(self):
        self.e0, self.e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        self.e0.record(self.stream)
        return self

    def __exit__(self, *a):
        self.e1.record(self.stream)
        self.torch.cuda.synchronize()
        self.ms = self.e0.elapsed_time(self.e1)


DUMP_ROWS = 1 << 18       # records (and episodes) --dump-outputs keeps: 104 B a record in float32, about 33 MB in all


def dump_rows(n):
    """All n rows, or a fixed seeded sample of DUMP_ROWS of them: the same indices whenever n is the same."""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))


def dump_outputs(out_dir, eng, twc, c):
    """Write the arrays the last timed collect hands its caller (the CollectedData fields of PPOCollector.collect) to
    out_dir/<name>.npy, so that two builds run with the same arguments can be compared output for output."""
    import ctypes as C

    from twisterl_b200 import _lib
    R, E = int(c.n_records), int(c.num_episodes)
    # the whole collect comes to the host through the library's own copy-out, as PPOCollector.collect receives it, and
    # is sampled there: 66 B a puzzle15 record, about 1.1 GB of pageable host memory at 65 536 episodes of difficulty 128
    # (outside the timed region, and only with --dump-outputs)
    hb, arrs, _ = twc._host_buffers(R, c.n_cells, c.num_actions, E, pinned=False)
    _lib.check(_lib.load().twr_collected_to_host(eng._h, C.byref(hb)))
    rec, ep = dump_rows(R), dump_rows(E)
    out_dir.mkdir(parents=True, exist_ok=True)
    for k in ("obs", "logits", "values", "rewards", "advs", "rets", "actions", "perms"):
        np.save(out_dir / f"{k}.npy", arrs[k][rec].astype(np.float32))
    np.save(out_dir / "ep_len.npy", arrs["ep_len"][ep].astype(np.float32))
    np.save(out_dir / "record_index.npy", rec.astype(np.float64))
    np.save(out_dir / "episode_index.npy", ep.astype(np.float64))
    np.save(out_dir / "stats.npy", np.array([R, E, c.successes, c.reward_sum], dtype=np.float64))


def run_ours(args, rank, local_rank, world):
    import ctypes as C

    import torch

    import twisterl_b200 as tw
    from twisterl_b200 import _lib, collector as twc, dist as twd, nn as twn

    torch.cuda.set_device(local_rank)
    stream = torch.cuda.current_stream()
    eng = tw.Engine(device=local_rank, precision=args.precision, seed=0x5EED5EED, rank=rank, world=world,
                    stream=stream.cuda_stream)
    comm = twd.Comm(eng, rank=rank, world=world)          # NCCL communicator inside the engine (C ABI)
    L = _lib.load()

    sd = synth_weights()
    pol = synth_policy(twn, sd, 256, *(puzzle15_twists() if args.twists else ((), ())))
    env = tw.env.Puzzle(4, 4, args.difficulty, 2, 256)
    col = twc.PPOCollector(args.episodes, 0.995, 0.995, 32, engine=eng)
    hpol = pol.device_handle(eng)
    nblob = int(L.twr_policy_blob_floats(hpol))

    def one_step(collector=col, environment=env, policy=pol, handle=hpol):
        comm.broadcast_weights(handle, root=0)            # per-iteration weight broadcast (ncclBroadcast) + operand refresh
        c = collector.collect_device(environment, policy)
        # stats reduction (ncclAllReduce); the reduced numbers are read on the host every iteration, as a trainer logs them
        comm.allreduce([c.num_episodes, c.successes, c.reward_sum, c.n_records])
        return c

    def barrier():
        comm.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        one_step()
    # ---- timed region: device-resident inputs, CUDA events on the launching stream
    eng.set_timing(True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    l0 = eng.launch_count()
    records, fwd_ms, fwd_launches = 0, 0.0, 0
    with Timer(torch, stream) as tm:
        for _ in range(args.steps):
            last = one_step()
            records += int(last.n_records)
            f, _, n = eng.last_timing()
            fwd_ms += f; fwd_launches += n
    barrier()
    clocks = sampler.stop()
    ms = tm.ms
    launches = eng.launch_count() - l0
    eng.set_timing(False)
    ms = comm.max_over_ranks(ms)
    r0_records = records
    records, launches = comm.allreduce([records, launches])
    value = records / (ms * 1e-3)
    if args.dump_outputs and rank == 0:               # before the e2e collects below replace the engine's last result
        dump_outputs(Path(args.dump_outputs), eng, twc, last)

    # ---- e2e: the C-ABI call with HOST buffers (weights H2D, CollectedData D2H inside the timed region)
    cap = int(L.twr_max_records(C.byref(tw.env.spec_from_env(env)), args.episodes))
    hb, arrs, holders = twc._host_buffers(cap, 16, 4, args.episodes, pinned=True, obs_u8=True)   # obs as u8 indices (obs_size 256)
    desc = pol.desc()
    spec = tw.env.spec_from_env(env)
    out = _lib.Collected()
    e2e_steps = max(1, min(args.steps, 10))
    for _ in range(2 if args.warmup >= 2 else 1):
        _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), hpol, C.byref(desc), args.episodes, 0.995, 0.995,
                                          C.byref(hb), C.byref(out)))
    barrier()
    t0 = time.perf_counter()
    e2e_records = 0
    for _ in range(e2e_steps):
        _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), hpol, C.byref(desc), args.episodes, 0.995, 0.995,
                                          C.byref(hb), C.byref(out)))
        e2e_records += int(out.n_records)
    barrier()
    e2e_s = comm.max_over_ranks(time.perf_counter() - t0)
    e2e_records = comm.allreduce([e2e_records])[0]
    rec_per_step = e2e_records / e2e_steps / world
    d2h = int(rec_per_step * sum(a.dtype.itemsize * int(np.prod(a.shape[1:])) for k, a in arrs.items() if k != "ep_len")
              + arrs["ep_len"].nbytes)
    # bytes that actually cross PCIe: the observation indices (or, opt-in, the 16 tiles as nibbles: 8 B), action / twist /
    # reward as one byte, and the advantages not at all -- rebuilt on the host from rets - values (twr_ppo_collect_host); d2h_bytes_per_step counts what lands in
    # the caller's buffers
    nib = 8 if int(os.environ.get("TWISTERL_B200_E2E_NIB", "0") or 0) > 0 else 16      # opt-in wire format, see twr_ppo_collect_host
    pcie = int(rec_per_step * (nib + 16 + 4 + 4 + 1) + arrs["ep_len"].nbytes)
    h2d = nblob * 4
    # the host-memory ceiling of this box for the same bytes: one plain pinned cudaMemcpyAsync stream per rank, all ranks at once
    ceil_bytes = 256 << 20
    src = torch.empty(ceil_bytes, dtype=torch.uint8, device="cuda")
    dst = torch.empty(ceil_bytes, dtype=torch.uint8).pin_memory()
    dst.copy_(src, non_blocking=True); torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    d2h_gbs = world * 4 * ceil_bytes / comm.max_over_ranks(time.perf_counter() - t0) / 1e9
    del src, dst, hb, arrs, holders

    pk = peaks()
    line = None
    if rank == 0:
        achieved = r0_records * FLOP_PER_STEP["puzzle15"] / (fwd_ms * 1e-3) / 1e12 if fwd_ms > 0 else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE[args.precision],
            "data": "synthetic",
            "config": {"workload": f"examples/ppo_puzzle15_v1.json PPO rollout, {args.episodes} parallel envs per GPU, "
                                   f"difficulty {args.difficulty}, depth budget {2 * args.difficulty}, synthetic N(0,0.05^2) weights",
                       "episodes_per_gpu": args.episodes, "records_per_step": records / args.steps,
                       "l2": "working set per step (records + compacted output, > 1.5 GB at 65536 envs) exceeds the 126 MB L2; no flush needed",
                       "precision": args.precision, "twists": bool(args.twists), "collectives": comm.backend},
            "clocks": clocks,
            "e2e": {"value": e2e_records / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "pcie_d2h_bytes_per_step": pcie, "steps": e2e_steps, "api": "twr_ppo_collect_host (pinned host buffers)",
                    # all ranks copying at once: what the host memory system of this box sustains, and the env-steps/s a
                    # collect could reach if it were nothing but that copy
                    "pinned_d2h_ceiling_GBs": d2h_gbs, "d2h_bound_env_steps_per_s": d2h_gbs * 1e9 / (pcie / rec_per_step)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "k_forward_fp32" if args.precision == "fp32" else "k_forward_tc2",
                         "achieved": achieved, "peak": pk["bf16"], "unit": "TFLOP/s",
                         "frac": (achieved / pk["bf16"]) if achieved else None,
                         "traffic": TRAFFIC.get((args.precision, args.episodes)),
                         "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of the first (129-step) k_forward_tc2 launch of a collect "
                                         "(ncu --set full, profiles/r2p_tc2_summary.md); the launch writes its records "
                                         "(42 B x envs x steps), operands stay in L2",
                         "peak_source": pk["src"] + " bf16_tflops_sustained",
                         "forward_ms_per_launch": fwd_ms / max(fwd_launches, 1), "forward_share_of_step": fwd_ms / tm.ms,
                         "algorithmic_flop_per_env_step": FLOP_PER_STEP["puzzle15"]},
        }
        if args.precision != "fp32" and achieved:
            ex = executed_flop(args.precision, 256, 512, 256)
            line["roofline"]["executed_tensor_flop_per_env_step"] = ex
            line["roofline"]["executed"] = achieved * ex / FLOP_PER_STEP["puzzle15"]
            line["roofline"]["executed_frac"] = line["roofline"]["executed"] / pk["bf16"]
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            rate0, _ = cpu_collect_rate(sd, 256, args.difficulty, cores)
            episodes = int(min(65536, max(256, rate0 * 12 / (2 * args.difficulty + 1))))
            t0 = time.perf_counter()
            rate, recs = cpu_collect_rate(sd, episodes, args.difficulty, cores)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{episodes} episodes of the same workload ({recs} records, "
                                              f"{time.perf_counter() - t0:.1f}s), C restatement of the Rust collector"}
    pol.release()
    if not args.no_extras:
        try:
            extra = run_extras(args, torch, tw, twc, twn, eng, comm, stream, rank, world, pk)
        except Exception as exc:                                       # noqa: BLE001 -- the headline line is printed regardless
            extra = [{"error": f"{type(exc).__name__}: {exc}"[:300]}]
        if rank == 0:
            line["extra"] = extra
    if rank == 0:
        print(json.dumps(line), flush=True)
    comm.close()


# dram bytes (read + write) of one steady-state forward launch, from the committed ncu capture of the same command
# dram__bytes_read.sum + dram__bytes_write.sum of the first persistent launch of a 65 536-env collect (ncu --set full, launch 0
# of profiles/r2p_tc2_summary.md for f16f8c: 129 steps; of profiles/r2_tc2_summary.md for f16x2w16: 128 steps)
TRAFFIC = {("f16x2w16", 65536): 3_088_896 + 296_557_568, ("f16f8c", 65536): 3_399_680 + 297_932_032}


# ------------------------------------------------------------- the other BASELINE configs ---
def run_extras(args, torch, tw, twc, twn, eng, comm, stream, rank, world, pk):
    """One entry per BASELINE.json config besides the headline, measured like the headline (weights broadcast, collect,
    stats reduction per step; CUDA events; max over ranks)."""
    from oracle import orc                                # cpu_baseline legs only
    cores = os.cpu_count() or 1
    K, W = args.extra_steps, 2
    out = []

    def ppo(name, workload, env, ospec, obs_size, hidden, flop_key, obs_k, episodes, scaling, perms=((), ())):
        sd = synth_weights(obs_size=obs_size, hidden=hidden)
        pol = synth_policy(twn, sd, obs_size, *perms)
        col = twc.PPOCollector(episodes, 0.995, 0.995, 32, engine=eng)
        h = pol.device_handle(eng)

        def step():
            comm.broadcast_weights(h, root=0)
            c = col.collect_device(env, pol)
            comm.allreduce([c.num_episodes, c.successes, c.reward_sum, c.n_records])
            return int(c.n_records)
        for _ in range(W):
            step()
        eng.set_timing(True)
        comm.barrier(); torch.cuda.synchronize()
        recs, fwd = 0, 0.0
        with Timer(torch, stream) as tm:
            for _ in range(K):
                recs += step()
                fwd += eng.last_timing()[0]
        eng.set_timing(False)
        ms = comm.max_over_ranks(tm.ms)
        total = comm.allreduce([recs])[0]
        ach = recs * FLOP_PER_STEP[flop_key] / (fwd * 1e-3) / 1e12 if fwd > 0 else None
        e = {"workload": workload, "metric": "rollout env-steps/sec incl. policy fwd", "unit": UNIT, "value": total / (ms * 1e-3),
             "ms_per_step": ms / K, "steps": K, "warmup": W, "episodes_per_gpu": episodes, "scaling": scaling, "dtype": args.precision,
             "roofline": {"bound": "tensor", "kernel": "k_forward_tc2" if args.precision != "fp32" else "k_forward_fp32",
                          "achieved": ach, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": ach / pk["bf16"] if ach else None,
                          "traffic": None, "algorithmic_flop_per_env_step": FLOP_PER_STEP[flop_key],
                          "executed_tensor_flop_per_env_step": executed_flop(args.precision, obs_k, 512, hidden) if args.precision != "fp32" else None,
                          "forward_share_of_step": fwd / tm.ms}}
        if world == 1 and not args.no_cpu_baseline and rank == 0:
            opol = orc.Policy.from_torch_state_dict(sd, *perms)
            n0, dt0 = orc.time_ppo_collect(ospec, opol, 64 * cores, 0.995, 0.995, 0x5EED5EED, 0, cores)
            ep = int(max(64 * cores, min(episodes, 64 * cores * 2.5 / max(dt0, 1e-3))))
            n, dt = orc.time_ppo_collect(ospec, opol, ep, 0.995, 0.995, 0x5EED5EED, 1, cores)
            e["cpu_baseline"] = {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": f"{ep} episodes of the same workload ({n} records, {dt:.1f}s), C restatement of the Rust collector"}
        pol.release()
        out.append(e)

    def az(name, workload, episodes, sims, difficulty):
        sd = synth_weights(obs_size=81, hidden=256)
        pol = synth_policy(twn, sd, 81)
        env = tw.env.Puzzle(3, 3, difficulty, 2, 256)
        col = twc.AZCollector(episodes, sims, 1.41, 1, 32, engine=eng)
        h = pol.device_handle(eng)

        def step():
            comm.broadcast_weights(h, root=0)
            d = col.collect_device(env, pol)
            comm.allreduce([d.num_episodes, d.successes, d.reward_sum, d.n_records])
            return int(d.n_records)
        step()
        comm.barrier(); torch.cuda.synchronize()
        l0 = eng.launch_count()
        recs = 0
        with Timer(torch, stream) as tm:
            for _ in range(max(1, K // 2)):
                recs += step()
        launches = eng.launch_count() - l0
        ms = comm.max_over_ranks(tm.ms)
        total = comm.allreduce([recs])[0]
        # every record is one search of `sims` simulations, each with at most one leaf evaluation (+ the root's)
        ach = recs * (sims + 1) * FLOP_PER_STEP["puzzle8"] / (tm.ms * 1e-3) / 1e12
        e = {"workload": workload, "metric": "AlphaZero collection records/sec (one MCTS of num_mcts_searches simulations per record)",
             "unit": "records/s", "value": total / (ms * 1e-3), "ms_per_step": ms / max(1, K // 2), "steps": max(1, K // 2), "warmup": 1,
             "episodes_per_gpu": episodes, "num_mcts_searches": sims, "scaling": "weak", "dtype": args.precision,
             "leaf_evals_per_s_upper_bound": total * (sims + 1) / (ms * 1e-3), "gpu_launches": int(launches),
             "roofline": {"bound": "tensor", "kernel": "k_forward_tc2 (leaf batches) between k_mcts_* launches", "achieved": ach, "peak": pk["bf16"],
                          "unit": "TFLOP/s", "frac": ach / pk["bf16"], "traffic": None,
                          "note": "upper bound: terminal leaves skip the forward; small searches are launch-latency bound (two dependent "
                                  "launches per simulation), not pipe bound"}}
        if world == 1 and not args.no_cpu_baseline and rank == 0:
            opol = orc.Policy.from_torch_state_dict(sd)
            ospec = orc.puzzle_spec(3, 3, difficulty, 2, 256)
            t0 = time.perf_counter(); orc.az_collect(ospec, opol, 2, sims, 1.41, 1, seed=7); dt1 = (time.perf_counter() - t0) / 2
            per = int(max(1, min(64, 3.0 / max(dt1, 1e-4))))           # episodes per thread for ~3 s
            res = [0] * cores

            def work(i):
                res[i] = orc.az_collect(ospec, opol, per, sims, 1.41, 1, seed=7, collect_id=1, env_id_base=i * per)["n_records"]
            th = [threading.Thread(target=work, args=(i,)) for i in range(cores)]
            t0 = time.perf_counter()
            for t in th: t.start()
            for t in th: t.join()
            dt = time.perf_counter() - t0
            e["cpu_baseline"] = {"value": sum(res) / dt, "unit": "records/s", "cores": cores, "kind": "port",
                                 "sample": f"{per * cores} episodes ({sum(res)} records, {dt:.1f}s), C restatement of AZCollector + MCTS, one episode stream per thread"}
        pol.release()
        out.append(e)

    def guarded(fn, *fa):
        # an extra that fails (e.g. out of memory on a smaller device) must not take the headline line with it; the failure
        # is the same on every rank (same shapes), so the ranks stay in step
        try:
            fn(*fa)
        except Exception as exc:                                   # noqa: BLE001
            out.append({"workload": fa[1], "error": f"{type(exc).__name__}: {exc}"[:300]})

    guarded(ppo, "puzzle8_ppo", "examples/ppo_puzzle8_v1.json PPO rollout (3x3, difficulty 32 = diff_max, depth budget 64), 65536 envs per GPU",
            tw.env.Puzzle(3, 3, 32, 2, 256), orc.puzzle_spec(3, 3, 32, 2, 256), 81, 256, "puzzle8", 81, 65536, "weak")
    # GridWorld episodes are short (random walks end on the goal / trap after a handful of steps, 64 at most), so a collect
    # is bound by the latency of its <= 65 sequential steps unless the batch is large: 262144 envs per GPU
    guarded(ppo, "gridworld_ppo", "examples/grid_world/ppo_grid_world_5x5_v1.json PPO rollout (5x5, max_steps 64, difficulty 10 = diff_max), 262144 envs per GPU",
            tw.env.GridWorld(5, 5, 64, 10), orc.gridworld_spec(5, 5, 64, 10), 625, 128, "gridworld", 100, 262144, "weak")
    guarded(az, "puzzle8_az_100", "AlphaZero on puzzle8 (difficulty 8), 100 MCTS simulations per record, 65536 episodes per GPU", 65536, 100, 8)
    guarded(az, "puzzle8_az_1000", "AlphaZero on puzzle8 (difficulty 8), the reference's AZ defaults: 512 episodes x 1000 MCTS simulations (src/twisterl/defaults.py)",
            512, 1000, 8)
    per_gpu = (1 << 20) // world
    guarded(ppo, "puzzle15_twists_1M", f"puzzle15 PPO rollout with the {{identity, transpose}} twist set, 1048576 envs in total ({per_gpu} per GPU), difficulty 128",
            tw.env.Puzzle(4, 4, 128, 2, 256), orc.puzzle_spec(4, 4, 128, 2, 256), 256, 256, "puzzle15", 256, per_gpu, "strong", puzzle15_twists())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("TWISTERL_B200_PRECISION", "f16f8c"), choices=["fp32", "f16x2", "f16x2w16", "f16f8c"])
    ap.add_argument("--episodes", type=int, default=65536)
    ap.add_argument("--difficulty", type=int, default=128)
    ap.add_argument("--ref-episodes", type=int, default=2048)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline workload only")
    ap.add_argument("--extra-steps", type=int, default=3)
    ap.add_argument("--twists", action="store_true", help="enable the {identity, transpose} twist set on the headline workload")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline workload computed (rank 0's collect) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
