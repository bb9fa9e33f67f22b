"""Per-CTA pipeline wait counters of k_forward_tc2 (twr_debug_forward_profile)."""
import sys
from pathlib import Path
import numpy as np
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import twisterl_b200 as tw
from helpers import synth_state_dict, scramble_states
from parity import make_policies
from twisterl_b200 import _lib
from twisterl_b200.env import EnvBatch

n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
sd = synth_state_dict(0, 256, 512, 256, 4)
pol, _ = make_policies(sd, 256)
eng = tw.Engine(device=0, precision=sys.argv[3] if len(sys.argv) > 3 else "f16x2", seed=1)
b = EnvBatch(_lib.EnvSpec(0, 4, 4, 64, 2, 256), n, eng)
b.reset()
flags = int(sys.argv[2]) if len(sys.argv) > 2 else 0
craw = np.zeros(148 * 16 + 256, dtype=np.int64)
c = craw[:148 * 16].reshape(148, 16)
for rep in range(3):
    _lib.check(_lib.load().twr_debug_forward_profile(eng._h, pol.device_handle(eng), b._h, _lib.ptr(craw), 164, flags))
print("flags", flags)
names = {0: "mma total", 1: "mma wait slot(TMA)", 2: "mma wait a1_full", 3: "mma wait a2_full", 4: "mma wait d2_empty",
         5: "tiles", 6: "mma slot wait in G1", 7: "mma slot wait G1 kb0", 8: "producer wait empty", 9: "epi total", 10: "epi wait d1_full", 11: "epi wait d2_full", 12: "epi wait a1_empty", 13: "epi1 busy", 14: "build_a1 (incl wait)", 15: "epi2+step busy"}
for k, v in names.items():
    col = c[:, k]
    print(f"{v:22s} cta0 {col[0]:9d}  mean {col.mean():11.1f}  min {col.min():9d}  max {col.max():9d}")

tr = craw[148 * 16:].reshape(8, 32)
t0 = tr[0][tr[0] > 0].min()
ev = {0: "mma:a1_full", 1: "mma:g1c0", 2: "mma:g1c1", 3: "mma:g1c2", 4: "mma:g1c3", 5: "mma:g2j0", 6: "mma:g2j1", 7: "mma:g2j2",
      8: "mma:g2j3", 9: "mma:end", 10: "epi:d1full0", 11: "epi:d1full1", 12: "epi:d1full2", 13: "epi:d1full3", 14: "epi:e1done0",
      15: "epi:e1done1", 16: "epi:e1done2", 17: "epi:e1done3", 18: "epi:d2full", 19: "epi:stepdone", 20: "bld:start",
      21: "bld:a1empty", 22: "bld:done"}
for item in range(4):
    row = sorted((int(tr[item][k] - t0), ev[k]) for k in ev if tr[item][k] > 0)
    print("item", item, " ".join(f"{n}@{t}" for t, n in row))
