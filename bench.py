#!/usr/bin/env python
"""Benchmark of the hot path: TCJA-SNN inference samples/s at T=20 on N B200s.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU reference arm
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR  # + the last timed step's logits in DIR

A "step" is one pass of the hot path (frames on device -> logits on device) over
one batch of synthetic event frames.  Workload at N GPUs = BASELINE.json
configs[4]: a batch of 4096 samples sharded over the N GPUs (4096 / N each:
strong scaling; --batch gives a fixed per-GPU batch instead), 8-bit weights, 50 %
global magnitude pruning, T=20, 128x128x2 frames, no collective on the hot path
(one NCCL all-reduce of the accuracy counters after the timed region).  Prints
ONE JSON line on rank 0.

The reference itself (JAX/Flax) cannot be installed or imported in this image
(no jax / flax / ml_collections wheels, no network; SURVEY.md F2), so
`--impl reference` and `cpu_baseline` time the oracle's fp32 restatement of the
same graph (oracle/ref_snn.py, torch-CPU contractions) on the host cores:
kind = "port".
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

GOP_PER_SAMPLE_T20 = 33.647      # dense-equivalent int8 GOP / sample (BASELINE.md section 4)
CONV2_GOP_PER_SAMPLE = 2 * 12.080
METRIC = "TCJA-SNN inference samples/sec (T=20)"
UNIT = "samples/s"
DUMP_MAX_BYTES = 48 << 20          # --dump-outputs: larger outputs are sampled (keeps a dump easy to store and compare)


def peaks():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    p = json.load(open(path))
    return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sus=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                src="measured")
  return dict(hbm=6650.0, bf16=1590.0, bf16_sus=1400.0, src="fallback")


class ClockSampler:
  """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line) through NVML
  (nvidia_ml_py) from a background thread every 10 ms -- nvidia-smi -lms block-buffers its output and loses the
  samples of a sub-second region when it is stopped."""

  def __init__(self, gpu_index: int):
    self.idx = gpu_index
    self.samples = []
    self.thread = None
    self.stop_flag = False

  def _run(self):
    try:
      import pynvml as N
      N.nvmlInit()
      h = N.nvmlDeviceGetHandleByIndex(self.idx)
      mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
      while not self.stop_flag:
        sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
        try:
          r = N.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
          r = N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        self.samples.append((sm, mx, int(r)))
        time.sleep(0.01)
    except Exception as e:          # no NVML: report no samples rather than fail the bench
      self.err = repr(e)

  def start(self):
    import threading
    self.stop_flag = False
    self.thread = threading.Thread(target=self._run, daemon=True)
    self.thread.start()

  def stop(self):
    out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    if self.thread is None:
      return out
    self.stop_flag = True
    self.thread.join(2)
    if not self.samples:
      return out
    bits = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4,
            "hw_power_brake_slowdown": 0x80}
    reasons = sorted({name for _, _, r in self.samples for name, b in bits.items() if r & b})
    return {"sm_mhz": statistics.median([x[0] for x in self.samples]), "sm_max_mhz": max(x[1] for x in self.samples),
            "reasons": reasons, "samples": len(self.samples)}


def cpu_reference_samples_per_s(bits, prune, T, H, sample_B, reps, threads):
  """The oracle's fp32 restatement of the reference graph on the host cores (BASELINE.md section 3: configs[0],
  batch 16, one warm-up pass on one sample, median of >= 5 passes)."""
  import torch
  from oracle import ref_snn
  from snnquantprune_b200 import synthetic
  torch.set_num_threads(threads)
  v = synthetic.make_variables(bits=bits, prune_percentage=prune, T=T, H=H, seed=1)
  fr = synthetic.make_frames(sample_B, T, H, H, seed=0)
  ref_snn.cextnet_forward(v, fr[:1], bits)
  times = []
  for _ in range(reps):
    t0 = time.perf_counter()
    ref_snn.cextnet_forward(v, fr, bits)
    times.append(time.perf_counter() - t0)
  return sample_B / statistics.median(times), times


def parity_of_timed_batch(v, bits, H, frames_np, gpu_logits_np, T, lif):
  """Checker (outside every timed region): the first samples of the batch that was just timed, through the
  integer-path oracle (oracle/ref_net.py, pinned to the executed reference by tests/test_from_reference_cpu.py),
  against the logits the timed engine produced for them."""
  import numpy as np
  from oracle import build as obuild, ref_net
  obuild.build()
  lo = ref_net.forward(ref_net.pack_network(v, bits, H), frames_np)
  d = np.abs(lo - gpu_logits_np)
  return {"samples": int(frames_np.shape[0]), "logits_max_abs_diff": float(d.max()),
          "logit_quantum": 1.0 / (T * 10), "argmax_agree": bool(np.array_equal(lo.argmax(-1), gpu_logits_np.argmax(-1))),
          "bit_identical_logits": bool(np.array_equal(lo, gpu_logits_np)),
          "oracle": f"oracle/ref_net.py integer path (reference-order LIF); engine ran conv1 with --lif {lif}"}


def lif_mode_parity(eng, packed, frames, logits, impl, args, dev):
  """Checker (outside every timed region): what the timed LIF mode changes against the reference op order, measured
  on the timed batch itself -- conv1's pooled spikes of the first chunk (flip rate; north-star bar 1e-4) and the logits
  of the first chunks -- plus the throughput of the other modes (5 steps each)."""
  import torch
  from snnquantprune_b200 import CextNetEngine, _lib
  n = min(frames.shape[0], args.chunk)
  H = packed.H
  out = {"timed_mode": args.lif, "flip_budget": 1e-4}
  exact = CextNetEngine(packed, impl=impl, chunk=args.chunk, device=dev, lif_mode=_lib.LIF_EXACT)
  if eng.packed_spikes and args.lif != "exact":
    a, b = eng._workspace(n, n)["s1"][:n], exact._workspace(n, n)["s1"][:n]
    eng._conv(0, frames[:n], a, n, H, 2, 1)
    exact._conv(0, frames[:n], b, n, H, 2, 1)
    x = torch.bitwise_xor(a, b)
    flips = int(sum(int(((x >> k) & 1).sum().item()) for k in range(8)))
    out["conv1_pooled_spikes"] = int(a.numel() * 8)
    out["conv1_flips_vs_reference_order"] = flips
    out["conv1_flip_rate"] = flips / (a.numel() * 8)
  m = min(frames.shape[0], 2 * args.chunk)
  le = exact.forward(frames[:m])
  out["reference_order_logits_first2"] = le[:2].cpu().numpy()          # checked against the oracle by the caller
  dl = (le - logits[:m]).abs()
  out["logits_vs_reference_order"] = {"samples": m, "max_abs_diff": float(dl.max().item()),
                                      "samples_changed": int((dl.max(dim=1).values > 1e-6).sum().item()),
                                      "argmax_agree_fraction": float((le.argmax(-1) == logits[:m].argmax(-1)).float().mean().item())}
  by_mode = {}
  for name, mode in (("tensor", _lib.LIF_TENSOR), ("fast", _lib.LIF_FAST), ("exact", _lib.LIF_EXACT)):
    e = CextNetEngine(packed, impl=impl, chunk=args.chunk, device=dev, lif_mode=mode)
    for _ in range(2):
      e.forward(frames)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(5):
      e.forward(frames)
    e1.record(); torch.cuda.synchronize()
    by_mode[name] = frames.shape[0] * 5 / (e0.elapsed_time(e1) / 1e3)
    del e
  out["samples_per_s_by_lif_mode_5_steps"] = by_mode
  return out


def run_reference(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return 0
  threads = os.cpu_count() or 1
  sample_B = args.ref_batch
  T, H = args.T, args.H
  import torch
  from oracle import ref_snn
  from snnquantprune_b200 import synthetic
  torch.set_num_threads(threads)
  v = synthetic.make_variables(bits=args.bits, prune_percentage=args.prune, T=T, H=H, seed=1)
  fr = synthetic.make_frames(sample_B, T, H, H, seed=0)
  t1 = None
  for _ in range(max(1, args.warmup)):
    t0 = time.perf_counter()
    ref_snn.cextnet_forward(v, fr[:1], args.bits)
    t1 = time.perf_counter() - t0                     # seconds per sample, last warm-up pass
  # bounded sample: the K timed steps together take about two and a half minutes at most, whatever K is
  sample_B = max(1, min(sample_B, int(270.0 / (max(1, args.steps) * max(t1, 1e-3)))))
  fr = fr[:sample_B]
  t0 = time.perf_counter()
  for _ in range(args.steps):
    ref_snn.cextnet_forward(v, fr, args.bits)
  dt = time.perf_counter() - t0
  val = sample_B * args.steps / dt
  sample = (f"{sample_B} samples/step of the same workload (bits={args.bits}, prune={args.prune}, T={T}, "
            f"{H}x{H}x2), oracle fp32 restatement (torch-CPU conv2d/matmul), {threads} threads")
  line = {
      "impl": "reference", "metric": METRIC.replace("T=20", f"T={args.T}"), "value": val, "unit": UNIT, "n_gpus": args.gpus,
      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
      "higher_is_better": True, "scaling": "strong" if args.batch is None else "weak", "vs_baseline": None,
      "dtype": "f32", "data": "synthetic",
      "config": dict(workload_config(args, args.batch if args.batch is not None else args.global_batch // max(1, args.gpus),
                                     max(1, args.gpus)), reference_samples_per_step=sample_B),
      "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
      "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "gpu_launches": 0,
      "note": "reference (JAX/Flax) cannot be installed in this image; this is the CPU port of the same graph",
  }
  print(json.dumps(line), flush=True)
  return 0


def workload_config(args, per_gpu_batch, n):
  return {"workload": f"TCJA-SNN CextNet eval forward, {args.bits}-bit DuQ weights, {int(args.prune * 100)}% global "
                      f"magnitude pruning, T={args.T}, {args.H}x{args.H}x2 synthetic DVS frames "
                      f"(BASELINE.json configs[4] batch-sharded)",
          "bits": args.bits, "prune_percentage": args.prune, "T": args.T, "frame": [args.H, args.H, 2],
          "per_gpu_batch": per_gpu_batch, "global_batch": per_gpu_batch * n, "parallelism": f"dp{n}",
          "l2_policy": f"inputs larger than L2 ({per_gpu_batch * args.T * args.H * args.H * 2 / 1e6:.0f} MB of frames per GPU per step)"}


def run_ours(args):
  import numpy as np
  import torch
  from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic, _lib
  from snnquantprune_b200 import dist as D

  # libraries (NCCL) may print to stdout: keep fd 1 clean for the single JSON line
  sys.stdout.flush()
  saved_stdout = os.dup(1)
  os.dup2(2, 1)
  rank, ws, local = D.init("nccl")
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  lib = _lib.lib()
  if lib.snnqp_device_ok() != 1:
    raise SystemExit("bench.py needs an sm_100 GPU: " + lib.snnqp_last_error().decode())
  impl = {"auto": _lib.IMPL_AUTO, "simt": _lib.IMPL_SIMT, "tcgen05": _lib.IMPL_TCGEN05}[args.kernels]

  if args.batch is None and args.global_batch % ws:
    raise SystemExit(f"--global-batch {args.global_batch} must be divisible by the number of GPUs ({ws})")
  B = args.batch if args.batch is not None else args.global_batch // ws
  T, H = args.T, args.H
  v = synthetic.make_variables(bits=args.bits, prune_percentage=args.prune, T=T, H=H, seed=1)
  packed = pack_cextnet(v, args.bits, T, H, device=dev)
  lif = {"tensor": _lib.LIF_TENSOR, "fast": _lib.LIF_FAST, "exact": _lib.LIF_EXACT}[args.lif]
  eng = CextNetEngine(packed, impl=impl, chunk=args.chunk, device=dev, lif_mode=lif)
  # distinct frames per rank (the shard this rank owns of the global batch)
  base = synthetic.make_frames(min(B, 64), T, H, H, seed=100 + rank)
  reps = (B + base.shape[0] - 1) // base.shape[0]
  host_frames = torch.from_numpy(np.concatenate([base] * reps, 0)[:B]).pin_memory()
  frames = host_frames.to(dev, non_blocking=True)
  labels = torch.from_numpy(synthetic.make_labels(B, seed=3 + rank)).to(dev)
  torch.cuda.synchronize()

  # ---- device-resident timing --------------------------------------------
  for _ in range(args.warmup):
    logits = eng.forward(frames)
  torch.cuda.synchronize()
  sampler = ClockSampler(local)
  D.barrier(); torch.cuda.synchronize()
  if rank == 0:
    sampler.start()
  lib.snnqp_launch_count(1)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(args.steps):
    logits = eng.forward(frames)
  e1.record()
  torch.cuda.synchronize(); D.barrier()
  launches = int(lib.snnqp_launch_count(0))
  clocks = sampler.stop() if rank == 0 else None
  ms = e0.elapsed_time(e1)
  t = torch.tensor([ms], device=dev, dtype=torch.float64)
  D.reduce_max(t)
  ms_max = float(t.item())
  value = B * ws * args.steps / (ms_max / 1e3)
  if args.dump_outputs:
    dump_logits(args.dump_outputs, D.gather_logits(logits, B * ws), rank)

  # ---- end to end: pinned host frames -> H2D -> forward -> logits D2H ------
  # the public host-memory call: chunked H2D on a copy stream overlapped with compute, logits copied back
  # Inputs travel in the zero-suppressed frame format (include/snnqp.h snnqp_expand_frames_zsf: cell bitmap + the
  # non-zero counts, encoded once by the data-loader side before the timed region, like the pinned dense frames
  # were); the dense-frame call is timed beside it.
  from snnquantprune_b200.input_pipeline import zsf_encode
  host_logits = torch.empty((B, packed.num_classes), dtype=torch.float32).pin_memory()
  eng_e2e = CextNetEngine(packed, impl=impl, chunk=args.e2e_chunk, device=dev, lif_mode=lif)
  e2e_steps = max(1, min(args.steps, args.e2e_steps))
  zb = zsf_encode(host_frames.numpy())

  def time_e2e(call):
    for _ in range(2):
      call()
    torch.cuda.synchronize(); D.barrier()
    e0.record()
    for _ in range(e2e_steps):
      call()
    e1.record()
    torch.cuda.synchronize(); D.barrier()
    tt = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    D.reduce_max(tt)
    return B * ws * e2e_steps / (float(tt.item()) / 1e3)

  e2e_value = time_e2e(lambda: eng_e2e.forward_host_zsf(zb, host_logits))
  torch.cuda.synchronize()
  e2e_logits_ok = bool(torch.equal(host_logits, logits.cpu()))       # same logits as the device-resident pass
  e2e_dense = time_e2e(lambda: eng_e2e.forward_host(host_frames, host_logits))

  # ---- dominant kernel (conv2 block), timed live with CUDA events ----------
  roof = dominant_kernel_roofline(eng, frames, args, dev)
  roof_kernels = per_kernel_rooflines(eng, frames, ms_max / args.steps, roof["peak"])
  # per-layer input densities of the synthetic run (a dead network would make the throughput meaningless)
  eng.forward(frames)
  rates = {k: round(v["mean"], 4) for k, v in eng.densities(frames).items()}
  lif_parity = lif_mode_parity(eng, packed, frames, logits, impl, args, dev) if (ws == 1 and not args.no_cpu_baseline) else None

  # ---- final accuracy reduction: the only collective, outside the timed region
  out = torch.zeros(2, device=dev, dtype=torch.float32)
  _lib.check(lib.snnqp_eval_metrics(_lib.ptr(logits), _lib.ptr(labels), B, packed.num_classes, _lib.ptr(out),
                                    _lib.stream()))
  cnt = torch.tensor([out[0].item(), out[1].item(), float(B)], device=dev, dtype=torch.float64)
  D.reduce_sums(cnt)

  if rank == 0:
    pk = peaks()
    cpu = parity = None
    if ws == 1 and not args.no_cpu_baseline:
      threads = os.cpu_count() or 1
      val, times = cpu_reference_samples_per_s(args.bits, args.prune, T, H, args.cpu_batch, args.cpu_passes, threads)
      cpu = {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
             "sample": f"BASELINE.json configs[0]: {args.cpu_batch} samples of the same workload, 1 warm-up, median of "
                       f"{args.cpu_passes} passes, oracle fp32 restatement of the reference graph (torch-CPU "
                       f"contractions); the JAX reference cannot run in this image"}
      parity = parity_of_timed_batch(v, args.bits, H, host_frames[:2].numpy(), logits[:2].cpu().numpy(), T, args.lif)
      le2 = lif_parity.pop("reference_order_logits_first2")
      if args.lif != "exact":          # the same two samples through this engine with --lif exact: bit parity with the oracle
        pe = parity_of_timed_batch(v, args.bits, H, host_frames[:2].numpy(), le2, T, "exact")
        parity["lif_exact_engine_bit_identical_logits"] = pe["bit_identical_logits"]
      parity["lif"] = lif_parity
    net_tops = value * GOP_PER_SAMPLE_T20 / 1e3 / ws          # dense-equivalent int8 TOP/s per GPU
    line = {
        "metric": METRIC.replace("T=20", f"T={args.T}"), "value": value, "unit": UNIT, "n_gpus": ws, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.batch is None else "weak", "vs_baseline": None,
        "dtype": "int8", "data": "synthetic",
        "config": dict(workload_config(args, B, ws),
                       arithmetic="int8 weights x u8 spikes/counts -> int32 accumulate (tcgen05 kind::i8), fp32 dequant + BatchNorm "
                                  "+ LIF epilogue; conv1 (--lif " + args.lif + "): " +
                                  ("kind::f16 with the BatchNorm scale folded into two fp16 weight pieces and the tau = 2 leak as "
                                   "tcgen05.mma scale-input-d (membranes in TMEM)" if args.lif == "tensor" else
                                   "exact kind::f16 accumulators, LIF on the CUDA cores")),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(zb.nbytes) * ws,
                "d2h_bytes_per_step": int(host_logits.numel() * 4) * ws, "steps": e2e_steps,
                "input_format": f"zero-suppressed frames (bitmap + {zb.value_bits}-bit non-zero counts), "
                                f"{zb.nbytes / B / 1e3:.0f} KB/sample instead of {host_frames.numel() / B / 1e3:.0f} KB dense uint8",
                "logits_equal_device_resident_pass": e2e_logits_ok,
                "dense_uint8_frames": {"value": e2e_dense, "unit": UNIT, "h2d_bytes_per_step": int(host_frames.numel()) * ws}},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roof,
        "roofline_kernels": roof_kernels,
        "cpu_baseline": cpu,
        "parity": parity,
        "network_roofline": {"bound": "tensor", "achieved": value * GOP_PER_SAMPLE_T20 / 1e3, "unit": "TOP/s",
                             "achieved_per_gpu": net_tops, "gop_per_sample": GOP_PER_SAMPLE_T20,
                             "peak_nominal_int8": 4500.0, "frac_nominal": net_tops / 4500.0,
                             "peak_2x_measured_bf16": 2 * pk["bf16_sus"],
                             "frac_2x_measured_bf16_sustained": net_tops / (2 * pk["bf16_sus"]),
                             "peak_measured_int8": roof["peak"], "frac_measured_int8": net_tops / roof["peak"],
                             "peaks": pk["src"]},
        "accuracy_vs_random_labels": cnt[0].item() / cnt[2].item(),
        "mean_nonzero_fraction_of_layer_inputs": rates,
        "kernels": args.kernels,
    }
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
  D.barrier()
  if torch.distributed.is_initialized():
    torch.distributed.destroy_process_group()
  return 0


def dump_logits(out_dir, logits, rank):
  """What the timed path hands its caller in the last timed step: the logits of the global batch in sample order, as
  DIR/logits.npy (float32).  The inputs are seeded, so two builds run with the same arguments can be compared output
  for output.  Beyond DUMP_MAX_BYTES a fixed, seeded sample of rows (in sample order) is written."""
  import numpy as np
  if rank != 0:
    return
  x = logits.cpu().numpy()
  if x.nbytes > DUMP_MAX_BYTES:
    rows = np.random.default_rng(0).choice(x.shape[0], DUMP_MAX_BYTES // x[0].nbytes, replace=False)
    x = x[np.sort(rows)]
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, "logits.npy"), x)


def dominant_kernel_roofline(eng, frames, args, dev):
  """conv2 block (72 % of the MACs): algorithmic int8 OPs per launch / measured
  launch duration.  Timed alone, back to back, on the launching stream."""
  import torch
  from snnquantprune_b200 import _lib
  L = _lib.lib()
  pk = eng.pk
  B = frames.shape[0]
  Bc = min(eng.chunk, B)
  eng.forward(frames)
  ws = eng._workspace(B, Bc)
  lay = pk.convs[1]
  C, Hh = pk.channels, pk.H // 2
  p = eng._bp(Bc, Hh, C, C, ws["s1"], ws["s2"], 1)
  call = lambda: _lib.check(L.snnqp_spiking_conv3x3_fwd(p, _lib.ptr(ws["s1"]), None, _lib.ptr(lay.wq),
                                                        _lib.ptr(lay.scale), _lib.ptr(lay.bias), _lib.ptr(ws["s2"]),
                                                        None, None, _lib.stream()))
  for _ in range(3):
    call()
  n = 10
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  torch.cuda.synchronize()
  e0.record()
  for _ in range(n):
    call()
  e1.record()
  torch.cuda.synchronize()
  ms = e0.elapsed_time(e1) / n
  ops = CONV2_GOP_PER_SAMPLE * 1e9 * Bc * (pk.T / 20.0) * (pk.H / 128.0) ** 2
  pkp = peaks()
  traffic = None
  tpath = os.path.join(ROOT, "profiles", "r2_conv2_traffic.json")
  if os.path.exists(tpath):
    tj = json.load(open(tpath))          # dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture
    if tj.get("T") == pk.T and eng.packed_spikes:
      traffic = tj["dram_bytes_per_sample"] * Bc          # per launch, like `achieved` (capture: 148 samples per launch)
  achieved = ops / (ms / 1e3) / 1e12
  # Denominator: MEASURED_PEAKS.json has no int8 figure (HBM GB/s and dense bf16 only), so the int8 tensor-pipe
  # ceiling is measured live on this GPU by the library's own probe (back-to-back tcgen05.mma.kind::i8
  # 128x256x32, no loads, no epilogue); 2 x the driver-measured bf16 burst and the nominal 4.5 POP/s sit beside it.
  import ctypes
  tops = ctypes.c_double(0.0)
  _lib.check(L.snnqp_diag_imma_peak(4000, 3, ctypes.byref(tops), _lib.stream()))
  peak = float(tops.value)
  return {"kernel": "conv2 fused block (snnqp_spiking_conv3x3_fwd, 64x64x128->128, T steps inside)",
          "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
          "traffic": traffic, "ms_per_launch": ms, "units_per_launch": f"{Bc} samples x T={pk.T}",
          "peak_source": "dense int8 tensor-pipe ceiling measured live by snnqp_diag_imma_peak (tcgen05.mma.kind::i8 "
                         "128x256x32 back to back on all SMs; TOP/s reported in the TFLOP/s unit slot); "
                         "MEASURED_PEAKS.json has no int8 figure",
          "peak_2x_measured_bf16_burst": 2 * pkp["bf16"], "frac_of_2x_measured_bf16_burst": achieved / (2 * pkp["bf16"]),
          "peak_nominal_int8": 4500.0, "frac_of_nominal_int8": achieved / 4500.0}


def per_kernel_rooflines(eng, frames, ms_step, int8_peak_tops):
  """One entry per fused launch with >= 10 % of the step: CUDA-event time of the launch on one head chunk, its share of
  the step, and BOTH rooflines -- dense-equivalent int8 OP/s against the measured tensor-pipe ceiling and algorithmic
  HBM bytes (SURVEY.md 8(d): u8 frames in, bit-packed pooled spikes out / in) against the measured copy bandwidth."""
  import torch
  pk = eng.pk
  B = frames.shape[0]
  n = min(eng.chunk, B)
  ws = eng._workspace(B, n)
  T, H, C = pk.T, pk.H, pk.channels
  hbm = peaks()["hbm"]
  scale = (T / 20.0) * (H / 128.0) ** 2
  px = lambda h: T * h * h * C / 8 / 1e6 if eng.packed_spikes else T * h * h * C / 1e6       # MB / sample
  specs = [
      ("conv1 fused block (k_conv1_tclif / k_conv1_umma: 128x128x2 -> 128, LIF, pool)", lambda: eng._conv(0, frames[:n], ws["s1"][:n], n, H, 2, 1),
       2 * 0.755 * scale, T * H * H * 2 / 1e6 + px(H // 2), n),
      ("conv2 fused block (k_conv3x3_tile, 64x64x128 -> 128)", lambda: eng._conv(1, ws["s1"][:n], ws["s2"][:n], n, H // 2, C, 1),
       2 * 12.080 * scale, px(H // 2) + px(H // 4), n),
      ("conv3 fused block (k_conv3x3_tile, 32x32x128 -> 128)", lambda: eng._conv(2, ws["s2"][:n], ws["s3"][:n], n, H // 4, C, 1),
       2 * 3.020 * scale, px(H // 4) + px(H // 8), n),
  ]
  out = []
  chunks_per_step = B / n
  for name, fn, gop, mb, units in specs:
    for _ in range(2):
      fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(5):
      fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    share = ms * chunks_per_step / ms_step
    if share < 0.10:
      continue
    tops = gop * units / ms                      # GOP / ms = TOP/s
    gbs = mb * units / ms
    out.append({"kernel": name, "ms_per_launch": ms, "samples_per_launch": units, "share_of_step": share,
                "tensor": {"achieved": tops, "peak": int8_peak_tops, "unit": "TOP/s", "frac": tops / int8_peak_tops},
                "hbm": {"achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                        "algorithmic_mb_per_sample": mb},
                "bound": "tensor" if tops / int8_peak_tops > gbs / hbm else "hbm",
                "limiter": (("LIF_TENSOR: the leak runs on the tensor core (membranes in TMEM), the CUDA cores keep compare / reset / "
                             "pool / pack: 3.17 issued instructions per neuron-step, issue active 70 %, tensor pipe 56 % "
                             "(profiles/r2_ncu_full_lif_tensor.json)" if eng.lif_mode == 2 else
                             "issue slots of the LIF epilogue: 5.75 issued instructions per neuron-step, issue active 74 %, "
                             "tensor pipe 13 % (profiles/r2_ncu_full_final.json)") + " -- far from both rooflines by construction")
                           if "conv1" in name else "tensor pipe (97 % active bit-packed, 99 % with u8 spikes; two MMA-issuing warps)"})
  return out


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--kernels", default="auto", choices=["auto", "simt", "tcgen05"])
  ap.add_argument("--lif", default="tensor", choices=["tensor", "fast", "exact"],
                  help="conv1's LIF arithmetic (include/snnqp.h SNNQP_LIF_*): tensor = leak on the tensor core (engine default, "
                       "tolerance parity), fast = single-rounding fma, exact = the reference's op order (bit parity)")
  ap.add_argument("--global-batch", type=int, default=4096,
                  help="samples per step over all GPUs (BASELINE.json configs[4]: batch 4096 sharded over 1/2/4/8 GPUs)")
  ap.add_argument("--batch", type=int, default=None, help="samples per GPU per step (overrides --global-batch: weak scaling)")
  ap.add_argument("--chunk", type=int, default=296, help="samples per head launch: a multiple of 37 makes the strip / item counts of conv1-3 exact multiples of the 148 persistent CTAs (296 -> 256 / 64 / 16 waves)")
  ap.add_argument("--bits", type=int, default=8)
  ap.add_argument("--prune", type=float, default=0.5)
  ap.add_argument("--T", type=int, default=20)
  ap.add_argument("--H", type=int, default=128)
  ap.add_argument("--e2e-steps", type=int, default=20)
  ap.add_argument("--cpu-passes", type=int, default=5)
  ap.add_argument("--e2e-chunk", type=int, default=296, help="largest H2D / head chunk of the end-to-end path (chunks grow from 16)")
  ap.add_argument("--cpu-batch", type=int, default=16)
  ap.add_argument("--ref-batch", type=int, default=16)
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="after the timed steps, write the logits of the last one to DIR/logits.npy (float32)")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl == "reference":
    ap.error("--dump-outputs applies to --impl ours (the reference arm's sample size follows its timing)")
  if args.warmup < 3 and args.impl == "ours":
    args.warmup = 3
  if args.impl == "reference":
    return run_reference(args)
  return run_ours(args)


if __name__ == "__main__":
  sys.exit(main())
