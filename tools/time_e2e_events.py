"""End-to-end throughput of the host input formats, and the event integration kernel, in one run:
python tools/time_e2e_events.py [B] [--out FILE]

At B = 4096, chunk 296, T = 20, H = 128, the engine's default LIF mode, it reports samples/s of
  forward              frames resident in HBM -> logits in HBM
  forward_host         dense uint8 frames in pinned host memory
  forward_host_zsf     zero-suppressed frames (input_pipeline.ZsfBatch)
  forward_host_events  packed events (input_pipeline.EventBatch): U16 on a 128 sensor, and U32 on a 256 sensor at
                       resolution_scale 2
all on the same inputs (the frames are the U16 batch integrated on the GPU, and every path must give the same logits),
plus the wire bytes per sample of each format, the integration kernel's events/s for int32 records, U16 and U32
words on the same events, and the host encoder's samples/s (host time).  The events are synthetic.make_events
(Poisson-like 0.15 events per frame cell); UNIQUE distinct samples are tiled to B.  One JSON object per line."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic, _lib  # noqa: E402
from snnquantprune_b200 import input_pipeline as ip  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 and not sys.argv[1].startswith("-") else 4096
OUT = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
T, H, CHUNK, UNIQUE = 20, 128, 296, 512
assert torch.cuda.is_available(), "needs a GPU"
lines = []


def emit(d):
  print(json.dumps(d), flush=True)
  lines.append(d)


def card():
  name = torch.cuda.get_device_name(0)
  try:
    pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                        capture_output=True, text=True, timeout=60).stdout.strip()
  except (OSError, subprocess.SubprocessError):
    pl = "unknown"
  return {"card": name, "power_limit": pl}


def tile(eb, reps):
  """An EventBatch of ``reps`` copies of ``eb`` back to back."""
  o = eb.offsets.numpy()
  n = int(o[-1])
  words = np.tile(eb.events.numpy(), reps)
  off = np.concatenate([[0]] + [o[1:] + k * n for k in range(reps)])
  return ip.EventBatch(torch.as_tensor(words).pin_memory(), torch.as_tensor(off).pin_memory(), eb.format,
                       eb.sensor_wh, eb.max_events_per_sample)


def timed(fn, n):
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  torch.cuda.synchronize()
  e0.record()
  for _ in range(n):
    fn()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / n


emit(dict(card(), B=B, T=T, H=H, chunk=CHUNK, unique_samples=UNIQUE))

# ---- inputs ----------------------------------------------------------------------------------------------------------
reps = B // UNIQUE
assert reps * UNIQUE == B
s16 = synthetic.make_events(UNIQUE, T, H, seed=0)
t0 = time.perf_counter()
eb16u = ip.encode_events(s16, H)
enc16 = time.perf_counter() - t0
s32 = synthetic.make_events(UNIQUE, T, 2 * H, seed=1, rate=0.15 / 4)      # 0.15 events per cell after rs = 2
t0 = time.perf_counter()
eb32u = ip.encode_events(s32, 2 * H)
enc32 = time.perf_counter() - t0
assert eb16u.format == _lib.EVENTS_U16 and eb32u.format == _lib.EVENTS_U32
n_ev = int(eb16u.offsets[-1])
emit({"host_encoder": "encode_events", "clock": "host (time.perf_counter)", "samples": UNIQUE,
      "u16_samples_per_s": UNIQUE / enc16, "u32_samples_per_s": UNIQUE / enc32,
      "events_per_sample_mean": n_ev / UNIQUE})
eb16, eb32 = tile(eb16u, reps), tile(eb32u, reps)
del s32

# ---- the integration kernel on the same events: int32 records vs U16 vs U32 words ------------------------------------
rec = np.concatenate(s16, 0)
addrs = torch.as_tensor(rec).cuda()
w16 = eb16u.events.cuda()
w32 = torch.as_tensor((rec[:, 0].astype(np.uint32) | (rec[:, 1].astype(np.uint32) << 15)
                       | ((rec[:, 2] != 0).astype(np.uint32) << 31)).view(np.int32)).cuda()
off = eb16u.offsets.cuda()
fr_k = torch.empty((UNIQUE, T, H, H, 2), device="cuda", dtype=torch.uint8)
mx = eb16u.max_events_per_sample
kern = {
    "i32x3": (lambda: ip.events_to_frames(addrs, off, T, H, out=fr_k, max_events_per_sample=mx), 12),
    "u16": (lambda: ip.events_to_frames_packed(w16, off, _lib.EVENTS_U16, T, H, out=fr_k, max_events_per_sample=mx), 2),
    "u32": (lambda: ip.events_to_frames_packed(w32, off, _lib.EVENTS_U32, T, H, out=fr_k, max_events_per_sample=mx), 4),
}
ref = None
for name, (fn, _) in kern.items():
  fn()
  got = fr_k.clone()
  ref = got if ref is None else ref
  assert torch.equal(got, ref), name
del ref, got
res = {k: [] for k in kern}
for _ in range(3):                                         # alternate the formats, keep the best of three
  for name, (fn, _) in kern.items():
    res[name].append(timed(fn, 10))
for name, (_, bpe) in kern.items():
  ms = min(res[name])
  byt = n_ev * bpe + fr_k.numel()
  emit({"kernel": "k_events_to_frames", "format": name, "samples": UNIQUE, "events": n_ev, "ms": ms,
        "ms_all": res[name], "events_per_s": n_ev / ms * 1e3, "algorithmic_bytes": byt, "GBps": byt / ms / 1e6})
del addrs, w16, w32, fr_k, rec, s16
torch.cuda.empty_cache()

# ---- end to end ------------------------------------------------------------------------------------------------------
v = synthetic.make_variables(bits=8, prune_percentage=0.5, T=T, H=H, seed=1)
eng = CextNetEngine(pack_cextnet(v, 8, T, H, device="cuda"), chunk=CHUNK)
frames = ip.events_to_frames_packed(eb16.events.cuda(), eb16.offsets.cuda(), eb16.format, T, H,
                                    max_events_per_sample=eb16.max_events_per_sample)[0]
host_frames = frames.cpu().pin_memory()
t0 = time.perf_counter()
zb = ip.zsf_encode(host_frames[:UNIQUE].numpy())
zenc = time.perf_counter() - t0
zb = ip.zsf_encode(host_frames.numpy())
frames32 = ip.events_to_frames_packed(eb32.events.cuda(), eb32.offsets.cuda(), eb32.format, T, 2 * H, 2,
                                      max_events_per_sample=eb32.max_events_per_sample)[0]
out = torch.empty((B, eng.pk.num_classes), dtype=torch.float32).pin_memory()
paths = {
    "forward": (lambda: eng.forward(frames), None),
    "forward_host": (lambda: eng.forward_host(host_frames, out), None),
    "forward_host_zsf": (lambda: eng.forward_host_zsf(zb, out), None),
    "forward_host_events_u16": (lambda: eng.forward_host_events(eb16, out_host=out), None),
    "forward_host_events_u32_rs2": (lambda: eng.forward_host_events(eb32, resolution_scale=2, out_host=out), "u32"),
}
want = eng.forward(frames).cpu()
want32 = eng.forward(frames32).cpu()
del frames32
for name, (fn, which) in paths.items():
  got = fn()
  torch.cuda.synchronize()
  assert torch.equal(got.cpu(), want32 if which else want), name
res = {k: [] for k in paths}
for _ in range(3):                                         # alternate the paths, keep the best of three
  for name, (fn, _) in paths.items():
    res[name].append(timed(fn, 4))
wire = {"forward": 0, "forward_host": host_frames[0].numel(), "forward_host_zsf": zb.nbytes / B,
        "forward_host_events_u16": eb16.nbytes / B, "forward_host_events_u32_rs2": eb32.nbytes / B}
base = B / min(res["forward"]) * 1e3
for name in paths:
  ms = min(res[name])
  emit({"path": name, "B": B, "ms": ms, "ms_all": res[name], "samples_per_s": B / ms * 1e3,
        "vs_forward": B / ms * 1e3 / base, "wire_bytes_per_sample": wire[name]})
i32 = (12 * int(eb16.offsets[-1]) + 8 * (B + 1)) / B
emit({"wire_bytes_per_sample": {"int32_records": i32, **{k: wire[k] for k in wire if k != "forward"}},
      "zsf_encoder_host_samples_per_s": UNIQUE / zenc})
if OUT:
  with open(OUT, "w") as f:
    f.write("\n".join(json.dumps(d) for d in lines) + "\n")
