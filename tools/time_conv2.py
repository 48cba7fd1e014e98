"""GPU timing of the conv2 fused block alone (W = 64).  python tools/time_conv2.py [B] [iters]
SNNQP_C2_SPLIT=<TT*10+ST> selects another TMEM-taps / input-stages split (developer experiment)."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic
B = int(sys.argv[1]) if len(sys.argv) > 1 else 296
n_it = int(sys.argv[2]) if len(sys.argv) > 2 else 10
T, H, C = 20, 128, 128
v = synthetic.make_variables(bits=8, prune_percentage=0.5, T=T, H=H, seed=1)
eng = CextNetEngine(pack_cextnet(v, 8, T, H), chunk=B)
fr = torch.as_tensor(synthetic.make_frames(B, T, H, H, seed=0), device="cuda")
ws = eng._workspace(B, B)
s1, s2 = ws["s1"][:B], ws["s2"][:B]
eng._conv(0, fr, s1, B, H, 2, 1)
fn = lambda: eng._conv(1, s1, s2, B, H // 2, C, 1)
for _ in range(2): fn()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
torch.cuda.synchronize(); e0.record()
for _ in range(n_it): fn()
e1.record(); torch.cuda.synchronize()
us = e0.elapsed_time(e1) / n_it * 1e3
print(f"conv2 B={B} packed={int(eng.packed_spikes)}: {us:9.1f} us = {us / B:6.3f} us/sample = "
      f"{24.16e9 * B / us / 1e6:7.1f} TOP/s, checksum {int(s2.sum().item())}")
