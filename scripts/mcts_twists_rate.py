"""MCTS-guided evaluation with and without twists (Policy::full_predict at every leaf) on puzzle15 with the shipped trained
weights, on both search paths: the persistent whole-search kernel and the lockstep kernels (TWISTERL_B200_MCTS_LOCKSTEP).

    python scripts/mcts_twists_rate.py [--sims 100] [--batches 128,4096] [--repeats 5]
    python scripts/mcts_twists_rate.py --dump DIR          # untwisted outputs of the searches, for a same-seed comparison
    python scripts/mcts_twists_rate.py --compare DIR_A DIR_B

Per (twists, batch, path): seconds per twr_evaluate_episodes call (best of --repeats after a warm-up, each call ends in a
device synchronise), and simulations per second of one twr_mcts_probs search over the same batch (batch x sims simulations
exactly; an evaluation runs a data-dependent number of searches).  The batch of 128 fits the persistent kernel, the batch
of 4096 does not: there the persistent row reports the lockstep path it falls back to.  --dump writes what the untwisted
searches return (visit counts on both paths, per-episode evaluate results, an AZ collect's arrays) as .npy files; two
builds run with the same arguments must give byte-identical files.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))

SEED = 0x5EED
SPEC = (4, 4, 6, 2, 64)                # puzzle15, difficulty 6, at most 64 steps


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:                     # the number is then reported as unknown, not guessed
        out = f"unknown ({exc})"
    return name, out or "unknown"


def set_path(lockstep: bool):
    if lockstep:
        os.environ["TWISTERL_B200_MCTS_LOCKSTEP"] = "1"
    else:
        os.environ.pop("TWISTERL_B200_MCTS_LOCKSTEP", None)


def evaluate(eng, pol, n, sims, cid):
    import twisterl_b200 as tw
    from twisterl_b200 import _lib
    spec = tw.env.spec_from_env(tw.env.Puzzle(*SPEC))
    s, r = C.c_float(), C.c_float()
    bs, bt = np.zeros(n, np.float32), np.zeros(n, np.float32)
    eng.set_collect_id(cid)
    _lib.check(_lib.load().twr_evaluate_episodes(eng._h, C.byref(spec), pol.device_handle(eng), n, 1, 1, sims, 1.41, 1,
                                                 C.byref(s), C.byref(r), _lib.ptr(bs), _lib.ptr(bt)))
    eng.synchronize()
    return bs, bt


def mcts_probs(eng, pol, batch, sims):
    from twisterl_b200 import _lib
    probs = np.zeros((batch.n, 4), np.float32); visits = np.zeros((batch.n, 4), np.int32)
    _lib.check(_lib.load().twr_mcts_probs(eng._h, pol.device_handle(eng), batch._h, sims, 1.41, 1, 0, 1, 0,
                                          _lib.ptr(probs), _lib.ptr(visits)))
    eng.synchronize()
    return probs, visits


def states_batch(eng, n):
    from helpers import scramble_states
    from twisterl_b200 import _lib
    from twisterl_b200.env import EnvBatch
    b = EnvBatch(_lib.EnvSpec(0, 4, 4, 6, 2, 64), n, eng)
    b.set_state(scramble_states(np.random.default_rng(n), n, 4, 4, 10))
    return b


def best_of(fn, repeats):
    fn()                                         # warm-up: module load, pool growth, kernel attributes
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter(); fn(); times.append(time.perf_counter() - t0)
    return min(times)


def path_taken(eng, pol, batch, sims):
    """'persistent' when the search took a few launches (up to four persistent ones and the root read-out), 'lockstep'
    when it took at least two per simulation."""
    n0 = eng.launch_count()
    mcts_probs(eng, pol, batch, sims)
    return "persistent" if eng.launch_count() - n0 <= 5 else "lockstep"


def rate(args):
    import twisterl_b200 as tw
    from helpers import trained15, transpose_twists
    from parity import make_policies
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}; engine precision {args.precision}; puzzle15 {SPEC}, trained15 weights, "
          f"{args.sims} simulations, deterministic, 1 search per episode, best of {args.repeats}")
    eng = tw.Engine(device=0, precision=args.precision, seed=SEED)
    _, sd = trained15()
    pols = {"none": make_policies(sd, 256)[0], "transpose": make_policies(sd, 256, *transpose_twists(4))[0]}
    rows = []
    for n in args.batches:
        batch = states_batch(eng, n)
        for lockstep in (False, True):
            set_path(lockstep)
            for twists, pol in pols.items():
                t_eval = best_of(lambda: evaluate(eng, pol, n, args.sims, 1), args.repeats)
                t_search = best_of(lambda: mcts_probs(eng, pol, batch, args.sims), args.repeats)
                row = dict(twists=twists, batch=n, requested="lockstep" if lockstep else "persistent",
                           path=path_taken(eng, pol, batch, args.sims), s_per_evaluate=round(t_eval, 5),
                           search_s=round(t_search, 6), sims_per_s=round(n * args.sims / t_search, 1))
                rows.append(row)
                print(f"  twists {twists:9s} batch {n:5d} requested {row['requested']:10s} ran {row['path']:10s} "
                      f"{t_eval:9.4f} s/evaluate   search {t_search * 1e3:8.2f} ms = {row['sims_per_s']:.3e} sims/s")
    set_path(False)
    print(json.dumps(dict(gpu=name, power_limit=power, precision=args.precision, sims=args.sims, spec=SPEC, rows=rows)))
    eng.close()


def dump(args):
    import twisterl_b200 as tw
    from helpers import trained15
    from parity import make_policies
    out = Path(args.dump)
    out.mkdir(parents=True, exist_ok=True)
    eng = tw.Engine(device=0, precision=args.precision, seed=SEED)
    pol, _ = make_policies(trained15()[1], 256)
    batch = states_batch(eng, 128)
    for lockstep in (False, True):
        set_path(lockstep)
        tag = "lockstep" if lockstep else "persistent"
        probs, visits = mcts_probs(eng, pol, batch, args.sims)
        np.save(out / f"mcts_visits_{tag}.npy", visits); np.save(out / f"mcts_probs_{tag}.npy", probs)
        bs, bt = evaluate(eng, pol, 128, args.sims, 3)
        np.save(out / f"evaluate128_{tag}.npy", np.stack([bs, bt]))
    set_path(False)
    bs, bt = evaluate(eng, pol, 4096, args.sims, 4)
    np.save(out / "evaluate4096.npy", np.stack([bs, bt]))
    eng.set_collect_id(5)
    d = tw.collector.AZCollector(256, 32, 1.41, 1, 1, engine=eng).collect(tw.env.Puzzle(4, 4, 6, 2, 64), pol)
    for key, arr in (("obs", d.obs_array), ("probs", d.logits_array), ("rewards", d.step_rewards), ("actions", d.step_actions),
                     ("remaining_values", d.additional_array("remaining_values")), ("ep_len", d.ep_len)):
        np.save(out / f"az_{key}.npy", np.asarray(arr))
    eng.close()
    print(f"dumped {len(list(out.glob('*.npy')))} arrays to {out}")


def compare(a, b):
    a, b = Path(a), Path(b)
    names = sorted(p.name for p in a.glob("*.npy"))
    assert names and names == sorted(p.name for p in b.glob("*.npy")), "the two dumps hold different arrays"
    bad = [n for n in names if (a / n).read_bytes() != (b / n).read_bytes()]
    for n in names:
        print(f"  {n:28s} {'identical' if n not in bad else 'DIFFERS'}")
    print(f"{len(names) - len(bad)}/{len(names)} arrays byte-identical")
    return 1 if bad else 0


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sims", type=int, default=100)
    ap.add_argument("--batches", type=lambda s: [int(x) for x in s.split(",")], default=[128, 4096])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--precision", default="f16x2")
    ap.add_argument("--dump", metavar="DIR")
    ap.add_argument("--compare", nargs=2, metavar=("DIR_A", "DIR_B"))
    args = ap.parse_args()
    if args.compare:
        sys.exit(compare(*args.compare))
    if args.dump:
        dump(args)
    else:
        rate(args)


if __name__ == "__main__":
    main()
