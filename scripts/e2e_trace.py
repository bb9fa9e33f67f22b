"""Host-collect timeline (TWISTERL_B200_E2E_TRACE) of the benchmark workload for the environment's current settings.
usage: e2e_trace.py [precision] ; knob: TWISTERL_B200_E2E_PARTS"""
import ctypes as C, os, sys, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import bench
import twisterl_b200 as tw
from twisterl_b200 import _lib, collector as twc, nn as twn
sd = bench.synth_weights()
eng = tw.Engine(device=0, precision=sys.argv[1] if len(sys.argv) > 1 else "f16x2w16", seed=0x5EED5EED)
pol = bench.synth_policy(twn, sd, 256)
env = tw.env.Puzzle(4, 4, 128, 2, 256)
L = _lib.load(); spec = tw.env.spec_from_env(env)
E = 65536
cap = int(L.twr_max_records(C.byref(spec), E))
hb, arrs, keep = twc._host_buffers(cap, 16, 4, E, pinned=True, obs_u8=True)
desc = pol.desc(); hpol = pol.device_handle(eng); out = _lib.Collected()
os.environ.pop("TWISTERL_B200_E2E_TRACE", None)
for _ in range(3):
    _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), hpol, C.byref(desc), E, 0.995, 0.995, C.byref(hb), C.byref(out)))
t0 = time.perf_counter()
for _ in range(5):
    _lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), hpol, C.byref(desc), E, 0.995, 0.995, C.byref(hb), C.byref(out)))
dt = (time.perf_counter() - t0) / 5
print(f"{dt * 1e3:.2f} ms per call, {out.n_records / dt:.4g} env-steps/s  (PARTS={os.environ.get('TWISTERL_B200_E2E_PARTS')}, cpus={os.cpu_count()})", flush=True)
os.environ["TWISTERL_B200_E2E_TRACE"] = "1"
_lib.check(L.twr_ppo_collect_host(eng._h, C.byref(spec), hpol, C.byref(desc), E, 0.995, 0.995, C.byref(hb), C.byref(out)))
keep = None
