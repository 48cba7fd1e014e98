"""CPU tests of the host side: the C-ABI library loads and exports every symbol
include/snnqp.h declares (no compute without a GPU), errors are loud, the
façade mirrors the reference's argument checks, and the N>1 sharding logic
works under gloo with world_size 2."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build():
  import sys
  sys.path.insert(0, ROOT)
  from snnquantprune_b200.csrc import build as b
  return b.build()


def test_library_exports_every_declared_symbol():
  _build()
  from snnquantprune_b200 import _lib
  header = open(os.path.join(ROOT, "include", "snnqp.h")).read()
  header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
  declared = set(re.findall(r"\b(snnqp_[a-z0-9_]+)\s*\(", header))
  assert len(declared) >= 17
  lib = _lib.lib()
  for name in declared:
    assert hasattr(lib, name), f"libsnnqp.so does not export {name}"
  assert declared == set(_lib.SIGNATURES.keys())
  assert lib.snnqp_abi_version() == _lib.ABI_VERSION == int(re.search(r"#define SNNQP_ABI_VERSION (\d+)", header).group(1))


def test_binding_constants_match_the_header():
  """The enum-like #defines the Python binding mirrors (spike layouts, LIF modes, implementations)."""
  from snnquantprune_b200 import _lib
  header = open(os.path.join(ROOT, "include", "snnqp.h")).read()
  val = lambda name: int(re.search(rf"#define {name} (-?\d+)", header).group(1))
  assert (_lib.LIF_EXACT, _lib.LIF_FAST, _lib.LIF_TENSOR) == (val("SNNQP_LIF_EXACT"), val("SNNQP_LIF_FAST"), val("SNNQP_LIF_TENSOR"))
  assert (_lib.SPIKES_U8, _lib.SPIKES_BITS) == (val("SNNQP_SPIKES_U8"), val("SNNQP_SPIKES_BITS"))
  assert (_lib.IMPL_AUTO, _lib.IMPL_SIMT, _lib.IMPL_TCGEN05) == (val("SNNQP_IMPL_AUTO"), val("SNNQP_IMPL_SIMT"), val("SNNQP_IMPL_TCGEN05"))


def _no_gpu_worker():
  os.environ["CUDA_VISIBLE_DEVICES"] = ""        # before this process's first CUDA call: it sees no device at all
  from snnquantprune_b200 import _lib
  lib = _lib.lib()
  assert lib.snnqp_device_ok() == 0
  rc = lib.snnqp_pack_levels(None, None, None, 8, 4, None, None)
  assert rc == 2 and b"no CPU fallback" in lib.snnqp_last_error()
  with pytest.raises(ValueError):
    _lib.ptr(torch.zeros(4))          # CPU tensors are rejected by the binding
  from snnquantprune_b200 import CextNetEngine
  with pytest.raises(ValueError):
    CextNetEngine.forward(object.__new__(CextNetEngine), torch.zeros((1, 2, 32, 32, 2), dtype=torch.uint8))


def test_no_gpu_fails_loudly_not_silently():
  """Checked in a child process that sees no CUDA device, so it holds on machines with a GPU too."""
  import torch.multiprocessing as mp
  _build()
  p = mp.get_context("spawn").Process(target=_no_gpu_worker)
  p.start()
  p.join(120)
  assert p.exitcode == 0


def test_facade_argument_checks_mirror_reference():
  from snnquantprune_b200 import QuantConv, QuantDense, QuantConfig, DuQ
  cfg = QuantConfig(bits=8, prune_percentage=0.5)
  assert "weight" in cfg and "bias" not in cfg          # flax_qconv.py:147,177 probes
  assert isinstance(cfg.weight(bits=8, g_scale=0.0), DuQ)
  ok = QuantConv(features=128, kernel_size=(3, 3), padding=((1, 1), (1, 1)), use_bias=False, config=cfg)
  ok.check_supported(128)
  with pytest.raises(NotImplementedError):
    QuantConv(features=128, kernel_size=(3, 3), strides=(2, 2), use_bias=False, config=cfg).check_supported(128)
  with pytest.raises(NotImplementedError):
    QuantConv(features=128, kernel_size=(1, 1), use_bias=False, config=cfg).check_supported(128)
  with pytest.raises(NotImplementedError):
    QuantConv(features=128, kernel_size=(3, 3), use_bias=False, config=QuantConfig(weight=None)).check_supported(128)
  with pytest.raises(NotImplementedError):
    QuantConv(features=128, kernel_size=(3, 3), use_bias=False, feature_group_count=2, config=cfg).check_supported(128)
  with pytest.raises(NotImplementedError):
    QuantDense(features=10, use_bias=True)
  assert QuantDense(features=10, use_bias=False).output_shape((4, 7)) == (4, 10)


def test_flatten_perm_matches_reference_flatten():
  from snnquantprune_b200.pack import flatten_perm
  side, C = 2, 8
  x = np.arange(side * side * C).reshape(side, side, C)       # ours: [h][w][c]
  ref = np.transpose(x, (2, 0, 1)).reshape(-1)                 # models.py:189-190
  perm = flatten_perm(side, C)
  ours = x.reshape(-1)
  # packed column r multiplies ours[r] and must read the kernel row of the same neuron
  assert np.array_equal(ref[perm], ours)


def test_shard_bounds_cover_and_balance():
  from snnquantprune_b200.dist import shard_bounds
  for total in (0, 1, 7, 16, 4096, 4099):
    for ws in (1, 2, 4, 8):
      spans = [shard_bounds(total, r, ws) for r in range(ws)]
      assert spans[0][0] == 0 and spans[-1][1] == total
      assert all(spans[i][1] == spans[i + 1][0] for i in range(ws - 1))
      sizes = [hi - lo for lo, hi in spans]
      assert max(sizes) - min(sizes) <= 1


def _gloo_worker(rank, ws, port, out):
  os.environ.update(RANK=str(rank), WORLD_SIZE=str(ws), LOCAL_RANK=str(rank),
                    MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
  from snnquantprune_b200 import dist as D
  D.init(backend="gloo")
  total = 7
  lo, hi = D.shard_bounds(total, rank, ws)
  full = torch.arange(total * 11, dtype=torch.float32).reshape(total, 11)
  local = full[lo:hi].clone()                   # stands for this rank's logits
  labels = torch.arange(total) % 11
  hits = (local.argmax(-1) == labels[lo:hi]).float().sum()
  m = D.reduce_sums(torch.tensor([hits.item(), float(hi - lo)]))
  g = D.gather_logits(local, total)
  t = D.reduce_max(torch.tensor([float(rank + 1)]))
  D.barrier()
  ok = bool(torch.equal(g, full)) and m[1].item() == total and t.item() == ws
  out[rank] = ok
  torch.distributed.destroy_process_group()


def test_world_size_2_gloo_sharding_and_reduction():
  import torch.multiprocessing as mp
  ctx = mp.get_context("spawn")
  mgr = ctx.Manager()
  out = mgr.dict()
  port = 29600 + os.getpid() % 300
  procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, out)) for r in range(2)]
  [p.start() for p in procs]
  [p.join(120) for p in procs]
  assert all(p.exitcode == 0 for p in procs)
  assert out.get(0) is True and out.get(1) is True


# ---- evaluate(): the reference's eval loop (examples/eval.py:53-139) ----------------------------
def _toy_forward(frames):
  x = frames.float().mean(dim=(1, 2, 3))                        # (b, 2)
  w = torch.arange(22, dtype=torch.float32).reshape(2, 11) / 7.0
  return torch.sin(x @ w)


def _torch_metrics(logits, labels, acc):
  onehot = torch.nn.functional.one_hot(labels.long(), logits.shape[1]).float()
  acc[0] += (logits.argmax(-1) == labels).float().sum()
  acc[1] += ((logits - onehot) ** 2).sum()


def _toy_batches(n_batches=3, B=6):
  g = torch.Generator().manual_seed(5)
  return [{"dvs_matrix": torch.randint(0, 5, (B, 4, 8, 8, 2), generator=g, dtype=torch.uint8),
           "label": torch.randint(0, 11, (B,), generator=g)} for _ in range(n_batches)]


def _eval_worker(rank, ws, port, out):
  os.environ.update(RANK=str(rank), WORLD_SIZE=str(ws), LOCAL_RANK=str(rank),
                    MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
  from snnquantprune_b200 import dist as D
  from snnquantprune_b200.eval import evaluate
  D.init(backend="gloo")
  out[rank] = evaluate(_toy_forward, _toy_batches(), steps_per_eval=-1, metrics_fn=_torch_metrics)
  torch.distributed.destroy_process_group()


def test_evaluate_matches_reference_summary_single_and_sharded():
  from snnquantprune_b200.eval import evaluate
  batches = _toy_batches()
  # the reference: per-step compute_metrics (mse_loss mean, accuracy vector), then the mean over everything
  losses, accs = [], []
  for b in batches:
    lg = _toy_forward(b["dvs_matrix"])
    oh = torch.nn.functional.one_hot(b["label"], 11).float()
    losses.append(((lg - oh) ** 2).mean().item())
    accs.append((lg.argmax(-1) == b["label"]).float().mean().item())
  want = {"loss": float(np.mean(losses)), "accuracy": float(np.mean(accs))}
  got = evaluate(_toy_forward, batches, metrics_fn=_torch_metrics)
  assert got["samples"] == 18 and got["steps"] == 3
  assert abs(got["loss"] - want["loss"]) < 1e-6 and abs(got["accuracy"] - want["accuracy"]) < 1e-6
  assert evaluate(_toy_forward, batches, steps_per_eval=2, metrics_fn=_torch_metrics)["samples"] == 12
  # world_size 2 (gloo): same summary on both ranks, one all-reduce
  import torch.multiprocessing as mp
  ctx = mp.get_context("spawn")
  out = ctx.Manager().dict()
  port = 29950 + os.getpid() % 40
  procs = [ctx.Process(target=_eval_worker, args=(r, 2, port, out)) for r in range(2)]
  [p.start() for p in procs]
  [p.join(120) for p in procs]
  assert all(p.exitcode == 0 for p in procs)
  for r in range(2):
    assert out[r]["samples"] == 18
    assert abs(out[r]["loss"] - want["loss"]) < 1e-6 and abs(out[r]["accuracy"] - want["accuracy"]) < 1e-6


def test_evaluate_rejects_indivisible_batch_like_reference():
  from snnquantprune_b200.eval import evaluate
  os.environ["WORLD_SIZE"] = "4"
  try:
    with pytest.raises(ValueError, match="divisible by the number of devices"):
      evaluate(_toy_forward, _toy_batches(1, 6), metrics_fn=_torch_metrics)
  finally:
    del os.environ["WORLD_SIZE"]


def test_host_chunk_schedule_covers_batch_and_respects_cap():
  """forward_host's chunk schedule: contiguous cover of [0, B), every chunk <= engine.chunk, small first chunk,
  non-decreasing until the cap (the last chunk takes the remainder)."""
  from snnquantprune_b200.engine import CextNetEngine
  eng = object.__new__(CextNetEngine)
  for cap in (1, 2, 16, 128, 256):
    eng.chunk = cap
    for B in (1, 5, 16, 17, 512, 4096, 4099):
      sched = eng.host_chunks(B)
      assert sched[0][0] == 0 and sum(n for _, n in sched) == B
      assert all(b1 == b0 + n0 for (b0, n0), (b1, _) in zip(sched, sched[1:]))
      assert all(0 < n <= cap for _, n in sched)
      assert sched[0][1] == min(16, cap, B)
      body = [n for _, n in sched[:-1]]
      assert body == sorted(body)


LIF_CONSTANTS_OFF_DEFAULT = [(1.7, 0.8, 0.1), (3.0, 1.0, 0.0), (2.0, 0.75, 0.0), (2.0, 1.0, 0.125), (2.0, 0.5, -0.25),
                             (2.0, -0.5, 0.0), (4.0, 0.75, 0.25), (0.5, 1.0, 1.2)]


def test_engine_packed_spikes_needs_standard_lif_constants():
  """Bit-packed spikes come only from the production epilogues, which hard-code tau = 2, v_threshold = 1, v_reset = 0;
  the conv launchers refuse bit-packed output with any other constants.  So at the reference geometry the engine's
  default must turn packing off for such constants (else every production forward fails at conv1), and an explicit
  packed_spikes=True with them is refused in the constructor.  Only packed.H and packed.channels are read there."""
  from types import SimpleNamespace
  from snnquantprune_b200 import _lib
  from snnquantprune_b200.engine import CextNetEngine
  ref_geom = SimpleNamespace(H=128, channels=128)
  assert CextNetEngine(ref_geom, device="cpu").packed_spikes
  assert CextNetEngine(ref_geom, tau=2.0, v_threshold=1.0, v_reset=0.0, device="cpu").packed_spikes
  assert not CextNetEngine(ref_geom, impl=_lib.IMPL_SIMT, device="cpu").packed_spikes
  assert not CextNetEngine(SimpleNamespace(H=64, channels=128), device="cpu").packed_spikes
  for tau, vth, vr in LIF_CONSTANTS_OFF_DEFAULT:
    eng = CextNetEngine(ref_geom, tau=tau, v_threshold=vth, v_reset=vr, device="cpu")
    assert eng.packed_spikes is False, (tau, vth, vr)
    assert (eng.tau, eng.v_th, eng.v_reset) == (tau, vth, vr)
    assert CextNetEngine(ref_geom, tau=tau, v_threshold=vth, v_reset=vr, device="cpu",
                         packed_spikes=False).packed_spikes is False
    with pytest.raises(ValueError, match="standard LIF constants"):
      CextNetEngine(ref_geom, tau=tau, v_threshold=vth, v_reset=vr, device="cpu", packed_spikes=True)
  # the envelope check still comes first: outside it, packing is refused whatever the constants
  with pytest.raises(ValueError, match="tcgen05"):
    CextNetEngine(SimpleNamespace(H=64, channels=128), device="cpu", packed_spikes=True)


def test_cextnet_engine_cache_key_follows_content():
  """The facade caches its packed engine on a content digest: an in-place edit of the variable tree (what
  import_torch_tcja / re-calibration do) must change the key, an untouched tree must not."""
  from snnquantprune_b200 import synthetic
  from snnquantprune_b200.models import CextNet
  v = synthetic.make_variables(bits=8, prune_percentage=0.5, T=3, H=32, seed=2)
  d0 = CextNet.variables_digest(v)
  assert CextNet.variables_digest(v) == d0
  v["params"]["QuantConv_1"]["prune_0"]["mask"][0, 0, 0, 0] = 1 - v["params"]["QuantConv_1"]["prune_0"]["mask"][0, 0, 0, 0]
  d1 = CextNet.variables_digest(v)
  assert d1 != d0
  v["batch_stats"]["BatchNorm_2"]["var"][5] *= 1.5
  assert CextNet.variables_digest(v) != d1


def test_xla_ffi_shim_type_checks_against_mock_header(tmp_path):
  """csrc/xla_ffi_shim.cc (the XLA custom-call handlers a maintainer registers from JAX, INTEGRATION.md) is compiled
  against tests/mock_xla -- a stand-in for jaxlib's ffi.h whose Bind() DSL static_asserts that every handler is
  callable with exactly the bound context / argument / result / attribute types.  A deliberately wrong binding must
  fail, so the check is not vacuous.  (In the product build the TU is part of libsnnqp.so, empty without the header.)"""
  import shutil
  import subprocess
  gxx = shutil.which("g++")
  assert gxx
  inc = ["-I", os.path.join(ROOT, "tests", "mock_xla"), "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include"]
  src = os.path.join(ROOT, "snnquantprune_b200", "csrc", "xla_ffi_shim.cc")
  r = subprocess.run([gxx, "-std=c++17", "-fsyntax-only", *inc, src], capture_output=True, text=True)
  assert r.returncode == 0, r.stderr
  text = open(src).read()
  handlers = re.findall(r"XLA_FFI_DEFINE_HANDLER_SYMBOL\((\w+),", text)
  assert len(handlers) >= 13 and {"SnnqpSpikingConvCounts", "SnnqpSpikingConvAtt", "SnnqpSpikingDenseAtt",
                                  "SnnqpPackConv", "SnnqpPackMatrix", "SnnqpFoldAffine"} <= set(handlers)
  bad = tmp_path / "bad.cc"
  bad.write_text(text.replace('.Attr<int32_t>("group"));', '.Attr<float>("group").Attr<int32_t>("extra"));'))
  r = subprocess.run([gxx, "-std=c++17", "-fsyntax-only", *inc, str(bad)], capture_output=True, text=True)
  assert r.returncode != 0 and "not callable with the types bound" in r.stderr
