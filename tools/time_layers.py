"""GPU timing of each fused launch of the engine (CUDA events), per chunk.  python tools/time_layers.py [B] [chunk]"""
import os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic, _lib
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
chunk = int(sys.argv[2]) if len(sys.argv) > 2 else 16
T, H, C = 20, 128, 128
v = synthetic.make_variables(bits=8, prune_percentage=0.5, T=T, H=H, seed=1)
eng = CextNetEngine(pack_cextnet(v, 8, T, H), chunk=chunk)
fr = torch.as_tensor(synthetic.make_frames(B, T, H, H, seed=0), device="cuda")
eng.forward(fr); torch.cuda.synchronize()
ws = eng._workspace(B, min(chunk, B))
def timeit(name, fn, n=10):
  for _ in range(2): fn()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  torch.cuda.synchronize(); e0.record()
  for _ in range(n): fn()
  e1.record(); torch.cuda.synchronize()
  print(f"{name:28s} {e0.elapsed_time(e1) / n * 1e3:9.1f} us")
n = min(chunk, B)
s1, s2 = ws["s1"][:n], ws["s2"][:n]
timeit(f"conv1 ({n} samples)", lambda: eng._conv(0, fr[:n], s1, n, H, 2, 1))
timeit(f"conv2 ({n} samples)", lambda: eng._conv(1, s1, s2, n, H // 2, C, 1))
timeit(f"conv3 ({n} samples)", lambda: eng._conv(2, s2, ws["s3"][:n], n, H // 4, C, 1))
timeit(f"conv4+counts ({B})", lambda: eng._conv(3, ws["s3"], ws["p4"], B, H // 8, C, 1, counts=ws["cnt4"]))
timeit(f"tcja ({B})", lambda: eng._tcja(0, B, H // 8, None, ws["cnt4"], ws["att4"]))
timeit(f"conv5 att ({B})", lambda: eng._conv(4, ws["p4"], ws["p5"], B, H // 16, C, 1, att=ws["att4"], counts=ws["cnt5"]))
timeit(f"dense1 att ({B})", lambda: eng._dense(eng.pk.dense1, B, ws["p5"].view(B, T, -1), ws["att5"], ws["d1"]))
timeit(f"dense2 ({B})", lambda: eng._dense(eng.pk.dense2, B, ws["d1"], None, ws["d2"]))
timeit(f"forward ({B})", lambda: eng.forward(fr), 3)
timeit(f"forward_graph ({B})", lambda: eng.forward_graph(fr), 3)
