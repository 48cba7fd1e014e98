"""GPU parity tests (run with -m gpu on a B200): every entry point of the C-ABI
against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): int32 accumulators, spikes and membranes of
the integer-input layers bit-exact against the integer-path oracle; membrane
<= 1e-5 relative and spike flip rate <= 1e-4 where fp32 summation order or expf
differ (att-weighted layers, whole network vs the fp32 reference-order path)."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

import attref
from oracle import ref_int, ref_net, ref_quant, ref_snn
from snnquantprune_b200 import _lib, synthetic
from snnquantprune_b200._lib import BlockParams
from snnquantprune_b200 import pack as pk_mod

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
F32 = np.float32
DEV = "cuda"


def dev(a, dtype=None):
  t = torch.as_tensor(np.ascontiguousarray(a), device=DEV)
  return t if dtype is None else t.to(dtype)


def P(t):
  return _lib.ptr(t)


def preact_err(acc_gpu, acc_ref, scale, bias):
  """|v_gpu - v_ref| / max(|v_ref|, 1) with v = acc * scale + bias: the error of a
  real-input accumulator in membrane (threshold = 1) units."""
  vg = acc_gpu.astype(np.float64) * scale + bias
  vr = acc_ref.astype(np.float64) * scale + bias
  return np.max(np.abs(vg - vr) / np.maximum(np.abs(vr), 1.0))


def impls():
  return [_lib.IMPL_SIMT, _lib.IMPL_TCGEN05]


# ------------------------------------------------------------------ pack ----
@pytest.mark.parametrize("bits", [2, 4, 8])
def test_pack_kernels_bit_exact(cuda_lib, oracle_lib, bits):
  rng = np.random.default_rng(bits)
  k = (rng.standard_normal((3, 3, 128, 128)) * 0.2).astype(F32)
  mask = ref_quant.local_mask(k, 0.6)
  a = ref_quant.gaussian_init(k, bits); c = F32(a * 1.1)
  kd, md = dev(k), dev(mask)
  ad, cd = dev(np.array([a], F32)), dev(np.array([c], F32))
  st = _lib.stream()
  # levels, same layout
  q = torch.empty(k.shape, device=DEV, dtype=torch.int8)
  _lib.check(cuda_lib.snnqp_pack_levels(P(kd), P(md), P(ad), bits, k.size, P(q), st))
  q_ref = ref_int.duq_levels_c(k, mask, a, bits)
  assert np.array_equal(q.cpu().numpy(), q_ref)
  assert np.array_equal(q_ref, (ref_quant.duq_levels(k, a, bits) * (mask != 0)).astype(np.int8))
  # conv3x3 tile layout [9][cout][cin]
  nb = int(cuda_lib.snnqp_conv3x3_blob_bytes(128, 128))
  assert nb == 9 * 128 * 128 + 64
  blob = torch.zeros((nb,), device=DEV, dtype=torch.int8)
  _lib.check(cuda_lib.snnqp_pack_conv3x3(P(kd), P(md), P(ad), bits, 128, 128, P(blob), st))
  wq = blob[:9 * 128 * 128].view(9, 128, 128)
  assert np.array_equal(wq.cpu().numpy(), q_ref.reshape(9, 128, 128).transpose(0, 2, 1))
  # DuQ + prune forward (fp32)
  out = torch.empty_like(kd)
  _lib.check(cuda_lib.snnqp_duq_forward(P(kd), P(md), P(ad), P(cd), bits, k.size, P(out), st))
  assert np.array_equal(out.cpu().numpy(), ref_quant.effective_weight(k, a, c, mask, bits))
  # slab bitmap
  nz = torch.empty((36,), device=DEV, dtype=torch.uint8)
  _lib.check(cuda_lib.snnqp_conv3x3_slab_bitmap(P(wq), 128, 128, P(nz), st))
  ref_nz = (q_ref.reshape(9, 4, 32, 128) != 0).any(axis=(2, 3)).reshape(-1)
  assert np.array_equal(nz.cpu().numpy().astype(bool), ref_nz)
  assert np.array_equal(blob[9 * 128 * 128: 9 * 128 * 128 + 36].cpu().numpy().astype(bool), ref_nz)


def test_pack_matrix_perm_pad_and_golden_vectors(cuda_lib, oracle_lib):
  rng = np.random.default_rng(9)
  K, N = 37, 24
  k = (rng.standard_normal((K, N)) * 0.3).astype(F32)
  mask = (rng.uniform(size=k.shape) > 0.4).astype(F32)
  a = ref_quant.max_init(k, 4)
  perm = rng.permutation(K).astype(np.int32)
  wq = torch.empty((N, 48), device=DEV, dtype=torch.int8)
  kd, md, ad, pd = dev(k), dev(mask), dev(np.array([a], F32)), dev(perm)      # keep alive until the launch ran
  _lib.check(cuda_lib.snnqp_pack_matrix(P(kd), P(md), P(ad), 4, K, N, P(pd), 48, P(wq), _lib.stream()))
  q_ref = ref_int.duq_levels_c(k, mask, a, 4)
  exp = np.zeros((N, 48), np.int8)
  exp[:, :K] = q_ref[perm].T
  assert np.array_equal(wq.cpu().numpy(), exp)
  g = json.load(open(os.path.join(GOLD, "duq_vectors.json")))
  w = np.array(g["w"], F32); m = np.array(g["mask"], F32)
  for case in g["cases"]:
    q = torch.empty(w.shape, device=DEV, dtype=torch.int8)
    wd, mdd = dev(w), dev(m)
    ad, cd = dev(np.array([case["a"]], F32)), dev(np.array([case["c"]], F32))
    _lib.check(cuda_lib.snnqp_pack_levels(P(wd), None, P(ad), case["bits"], w.size, P(q), _lib.stream()))
    assert q.cpu().numpy().astype(np.int32).tolist() == case["levels"]
    out = torch.empty(w.shape, device=DEV, dtype=torch.float32)
    _lib.check(cuda_lib.snnqp_duq_forward(P(wd), P(mdd), P(ad), P(cd), case["bits"], w.size, P(out),
                                          _lib.stream()))
    assert np.array_equal(out.cpu().numpy(), np.array(case["forward"], F32))


def test_fold_affine_bit_exact(cuda_lib):
  rng = np.random.default_rng(10)
  n = 128
  bn = dict(scale=rng.uniform(0.5, 1.5, n).astype(F32), bias=rng.standard_normal(n).astype(F32))
  stt = dict(mean=rng.standard_normal(n).astype(F32), var=rng.uniform(0.01, 2, n).astype(F32))
  c = np.array([0.731], F32)
  for bits in (2, 4, 8):
    s_ref, b_ref = ref_int.fold_affine(c, bits, bn, stt, n)
    s, b = pk_mod.fold_affine(c, bits, n, DEV, bn, stt)
    assert np.array_equal(s.cpu().numpy(), s_ref) and np.array_equal(b.cpu().numpy(), b_ref)
    s_ref, b_ref = ref_int.fold_affine(c, bits, n=1, extra_div=256.0)
    s, b = pk_mod.fold_affine(c, bits, 1, DEV, extra_div=256.0)
    assert np.array_equal(s.cpu().numpy(), s_ref) and b.item() == 0.0


# ------------------------------------------------------- fused conv block ----
def run_conv(lib, x_tb, wq, scale, bias, Cout, pool, impl, att=None, tau=2.0, batch_major=False, counts=None,
             dumps=True, x_bits=False, y_bits=False, lif_mode=0, popcount=None):
  """x_tb: numpy (T,B,H,W,Cin) u8.  Calls snnqp_spiking_conv3x3_fwd through the
  C-ABI; returns numpy (spikes (T,B,Ho,Wo,C), u (B,H,W,C), acc (T,B,H,W,C)).
  ``popcount``: optional int32 CUDA tensor [B][T] passed as y_popcount."""
  T, B, H, W, Cin = x_tb.shape
  if x_bits:
    x_tb = np.packbits(x_tb, axis=-1, bitorder="little")          # SNNQP_SPIKES_BITS
  if batch_major:
    xs = dev(np.ascontiguousarray(np.swapaxes(x_tb, 0, 1)))
    xst, xsb = xs.stride(1), xs.stride(0)
  else:
    xs = dev(x_tb)
    xst, xsb = xs.stride(0), xs.stride(1)
  Ho, Wo = (H // 2, W // 2) if pool else (H, W)
  spikes = torch.full((T, B, Ho, Wo, Cout // 8 if y_bits else Cout), 7, device=DEV, dtype=torch.uint8)
  u = torch.empty((B, H, W, Cout), device=DEV, dtype=torch.float32)
  acc = torch.empty((T, B, H, W, Cout), device=DEV, dtype=torch.float32 if att is not None else torch.int32)
  p = BlockParams()
  p.T, p.B, p.H, p.W, p.Cin, p.Cout = T, B, H, W, Cin, Cout
  p.x_stride_t, p.x_stride_b = xst, xsb
  p.y_stride_t, p.y_stride_b = spikes.stride(0), spikes.stride(1)
  attd = None
  if att is not None:
    attd = dev(att)
    p.att_stride_t, p.att_stride_b = attd.stride(0), attd.stride(1)
  p.att_mod = Cin
  p.tau, p.v_threshold, p.v_reset = tau, 1.0, 0.0
  p.pool, p.impl = int(pool), impl
  p.x_format, p.y_format, p.lif_mode = int(x_bits), int(y_bits), lif_mode
  if popcount is not None:
    p.y_popcount = P(popcount)
  ud, accd = (u, acc) if dumps else (None, None)      # no instrumentation outputs -> the production (FAST) variant
  if dumps == "u":                                     # membranes only (conv1's LIF_TENSOR kernel has no accumulator dump)
    accd = None
  if counts is None:
    _lib.check(lib.snnqp_spiking_conv3x3_fwd(p, P(xs), P(attd), P(wq), P(scale), P(bias), P(spikes), P(ud),
                                             P(accd), _lib.stream()))
  else:
    _lib.check(lib.snnqp_spiking_conv3x3_counts_fwd(p, P(xs), P(attd), P(wq), P(scale), P(bias), P(spikes), P(ud),
                                                    P(accd), P(counts), _lib.stream()))
  torch.cuda.synchronize()
  sp = spikes.cpu().numpy()
  if y_bits:
    sp = np.unpackbits(sp, axis=-1, bitorder="little")
  return sp, u.cpu().numpy(), acc.cpu().numpy()


def make_layer(rng, cin, cout, bits, p_prune):
  k = (rng.standard_normal((3, 3, cin, cout)) * 0.2).astype(F32)
  mask = ref_quant.local_mask(k, p_prune)
  a = ref_quant.gaussian_init(k, bits)
  lay = {"kernel": k, "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)}, "prune_0": {"mask": mask}}
  q = ref_int.duq_levels_c(k, mask, a, bits)
  energy = (q.astype(np.float64).reshape(-1, cout) ** 2).sum(0) * (a / (2 ** (bits - 1) - 1)) ** 2
  bn = dict(scale=rng.uniform(0.8, 1.2, cout).astype(F32), bias=(0.5 + 0.1 * rng.standard_normal(cout)).astype(F32))
  stt = dict(mean=(0.02 * rng.standard_normal(cout)).astype(F32), var=np.maximum(0.25 * energy, 1e-6).astype(F32))
  return lay, q, bn, stt


@pytest.mark.parametrize("shape,bits,pool", [
    ((3, 2, 8, 64, 2), 8, True), ((2, 1, 6, 128, 2), 4, False), ((5, 3, 128, 128, 2), 8, True)])
def test_spiking_conv1_tcgen05_bit_exact(cuda_lib, oracle_lib, shape, bits, pool):
  T, B, H, W, Cin = shape
  rng = np.random.default_rng(H * 5 + bits)
  lay, q, bn, stt = make_layer(rng, 2, 128, bits, 0.3)
  x = np.minimum(rng.poisson(0.3, size=shape), 255).astype(np.uint8)
  x[0, 0, 0, 0, :] = 255; x[-1, -1, -1, -1, :] = 200         # extreme counts at the corners
  packed = pk_mod.pack_conv3x3(lay, bits, DEV, bn, stt)
  s_ref, info = ref_int.spiking_conv3x3(x, q, *ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128),
                                        pool=pool, want=True)
  if pool:
    from test_gpu_conv1_rounding_band import check_band, conv1_band
    band = conv1_band(x, q, *ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128), modes=("fast",))
  for bm in (True, False):
    s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, _lib.IMPL_TCGEN05, batch_major=bm)
    assert np.array_equal(acc, info["acc"]), "conv1 int32 accumulators differ"
    assert np.array_equal(s, s_ref)
    assert np.array_equal(u, info["u"])
    s_fast, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, _lib.IMPL_TCGEN05,
                            batch_major=bm, dumps=False)
    assert np.array_equal(s_fast, s_ref)
    if pool:
      s_bits, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, _lib.IMPL_TCGEN05,
                              batch_major=bm, dumps=False, y_bits=True)
      assert np.array_equal(s_bits, s_ref)                  # ballot-packed output, reference op-order LIF
      for lm in (_lib.LIF_FAST, 101, 102, 103):             # single-rounding LIF variants: the float64 band
        s_f, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, _lib.IMPL_TCGEN05,
                             batch_major=bm, dumps=False, y_bits=True, lif_mode=lm)
        check_band(band, "fast", s_f, None, (lm, bm))
        assert np.mean(s_f != s_ref) <= 1e-4, (lm, float(np.mean(s_f != s_ref)))


@pytest.mark.parametrize("shape,bits", [((5, 5, 128, 128, 2), 8), ((20, 2, 128, 128, 2), 4), ((3, 1, 12, 256, 2), 2),
                                        ((2, 37, 8, 128, 2), 8), ((1, 2, 4, 128, 2), 8)])
def test_spiking_conv1_lif_tensor_tolerance(cuda_lib, oracle_lib, shape, bits):
  """SNNQP_LIF_TENSOR: the tau = 2 leak of conv1 runs on the tensor core (tcgen05.mma scale-input-d, membranes in
  TMEM; the weights times the folded scale as two fp16 pieces, the bias as three, fp32 accumulation).  Held to the
  float64 rounding band (tests/test_gpu_conv1_rounding_band.py): every decided pooled output equals float64 and every
  synchronised final membrane is within its delta_T; the north-star flip bar (<= 1e-4 against the integer oracle) is
  asserted as well.  Shapes: 160 tiles (one full wave of the 148 persistent CTAs plus a ragged one), T = 20, two
  tiles per image row (W = 256), fewer tiles than CTAs (74), a single step of a single tile row (T = 1, H = 4); u8 and
  bit-packed output, both batch layouts, extreme counts."""
  from test_gpu_conv1_rounding_band import check_band, conv1_band
  T, B, H, W, Cin = shape
  rng = np.random.default_rng(H * 7 + bits)
  lay, q, bn, stt = make_layer(rng, 2, 128, bits, 0.3)
  x = np.minimum(rng.poisson(0.3, size=shape), 255).astype(np.uint8)
  x[0, 0, 0, 0, :] = 255; x[-1, -1, -1, -1, :] = 200
  packed = pk_mod.pack_conv3x3(lay, bits, DEV, bn, stt)
  s_ref, info = ref_int.spiking_conv3x3(x, q, *ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128),
                                        pool=True, want=True)
  band = conv1_band(x, q, *ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128), modes=("tensor",))
  assert T == 1 or 0.02 < s_ref.mean() < 0.9
  for lm in (_lib.LIF_TENSOR,):
    for bm in (True, False):
      for yb in (True, False):
        s, u, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05,
                           batch_major=bm, dumps="u", y_bits=yb, lif_mode=lm)
        check_band(band, "tensor", s, u, (shape, bm, yb))
        flips = int((s != s_ref).sum())
        assert flips <= 1e-4 * s_ref.size, (lm, bm, yb, flips)
        s2, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05,
                            batch_major=bm, dumps=False, y_bits=yb, lif_mode=lm)
        assert np.array_equal(s2, s), "production and membrane-dumping variants disagree"
  # outside the kernel's envelope (no pool) the mode means the reference op order: bit-exact
  s_np, info_np = ref_int.spiking_conv3x3(x[:, :1], q, *ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128),
                                          pool=False, want=True)
  s, u, acc = run_conv(cuda_lib, x[:, :1], packed.wq, packed.scale, packed.bias, 128, False, _lib.IMPL_TCGEN05,
                       lif_mode=_lib.LIF_TENSOR)
  assert np.array_equal(s, s_np) and np.array_equal(u, info_np["u"]) and np.array_equal(acc, info_np["acc"])


@pytest.mark.parametrize("shape,bits,pool", [
    ((3, 2, 8, 8, 2), 8, True), ((2, 1, 16, 12, 2), 4, False), ((4, 2, 32, 32, 2), 2, True)])
def test_spiking_conv1_counts_bit_exact(cuda_lib, oracle_lib, shape, bits, pool):
  T, B, H, W, Cin = shape
  rng = np.random.default_rng(H * 3 + bits)
  lay, q, bn, stt = make_layer(rng, 2, 128, bits, 0.3)
  x = np.minimum(rng.poisson(0.4, size=shape), 255).astype(np.uint8)
  x[0, 0, 0, 0, :] = 255                                    # maximum count
  packed = pk_mod.pack_conv3x3(lay, bits, DEV, bn, stt)
  s_ref, info = ref_int.spiking_conv3x3(x, q, *ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128),
                                        pool=pool, want=True)
  for bm in (False, True):
    s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, _lib.IMPL_SIMT, batch_major=bm)
    assert np.array_equal(acc, info["acc"])
    assert np.array_equal(s, s_ref)
    assert np.array_equal(u, info["u"])
  assert 0.02 < s_ref.mean() < 0.9


@pytest.mark.parametrize("impl", impls())
@pytest.mark.parametrize("shape,bits,pool,prune", [
    ((3, 2, 16, 16, 128), 8, True, 0.5), ((2, 1, 32, 32, 128), 4, True, 0.8),
    ((2, 2, 64, 64, 128), 8, True, 0.5), ((3, 1, 16, 16, 128), 2, False, 0.9),
    ((1, 1, 8, 8, 128), 8, False, 0.0)])
def test_spiking_conv_binary_bit_exact(cuda_lib, oracle_lib, impl, shape, bits, pool, prune):
  T, B, H, W, Cin = shape
  p0 = BlockParams(); p0.T, p0.B, p0.H, p0.W, p0.Cin, p0.Cout, p0.pool, p0.impl = T, B, H, W, Cin, 128, int(pool), impl
  rng = np.random.default_rng(H + bits + T)
  lay, q, bn, stt = make_layer(rng, 128, 128, bits, prune)
  x = (rng.uniform(size=shape) < 0.25).astype(np.uint8)
  packed = pk_mod.pack_conv3x3(lay, bits, DEV, bn, stt)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=pool, want=True)
  cnt = torch.zeros((B, T, 128), device=DEV, dtype=torch.int32)
  try:
    s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl, batch_major=True,
                         counts=cnt)
  except _lib.SnnqpError as e:
    if impl == _lib.IMPL_TCGEN05 and e.code == 3:
      pytest.skip("shape outside the tcgen05 kernel's envelope: " + str(e))
    raise
  assert np.array_equal(acc, info["acc"]), "int32 accumulators differ"
  assert np.array_equal(s, s_ref), f"spike flips: {np.mean(s != s_ref)}"
  assert np.array_equal(u, info["u"]), "membrane differs"
  assert np.array_equal(cnt.cpu().numpy(), info["spikes"].sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2))
  assert 0.02 < s_ref.mean() < 0.9
  # production variant (no instrumentation outputs): same spikes, same counts
  cnt.zero_()
  s_fast, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl, batch_major=True,
                          counts=cnt, dumps=False)
  assert np.array_equal(s_fast, s_ref)
  assert np.array_equal(cnt.cpu().numpy(), info["spikes"].sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2))
  s_fast, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl, batch_major=False,
                          dumps=False)
  assert np.array_equal(s_fast, s_ref)
  if impl == _lib.IMPL_TCGEN05:
    # bit-packed spikes (SNNQP_SPIKES_BITS): packed input through the expander warps with the instrumented epilogue,
    # packed input and packed output with the production epilogue (pool only), both time/batch orders
    s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl, batch_major=True, x_bits=True)
    assert np.array_equal(acc, info["acc"]) and np.array_equal(s, s_ref) and np.array_equal(u, info["u"])
    if pool:
      for bm in (True, False):
        cnt.zero_()
        s_fast, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl, batch_major=bm,
                                counts=cnt if bm else None, dumps=False, x_bits=True, y_bits=True)
        assert np.array_equal(s_fast, s_ref)
        if bm:
          assert np.array_equal(cnt.cpu().numpy(), info["spikes"].sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2))
  else:
    with pytest.raises(_lib.SnnqpError):          # no silent fallback: the SIMT kernels speak SNNQP_SPIKES_U8 only
      run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl, dumps=False, x_bits=True)


@pytest.mark.parametrize("cin,cout", [(128, 96), (2, 96), (64, 64)])
def test_spiking_conv_simt_cout_not_dividing_block(cuda_lib, oracle_lib, cin, cout):
  """Cout = 96 does not divide the SIMT block (512 / 256 threads): the spare threads must not redo a neighbour
  block's quad -- spike counts (TCJA input) would be double-counted."""
  T, B, H, W, bits = 3, 2, 16, 16, 8
  rng = np.random.default_rng(cin + cout)
  lay, q, bn, stt = make_layer(rng, cin, cout, bits, 0.4)
  x = (rng.uniform(size=(T, B, H, W, cin)) < 0.3).astype(np.uint8)
  packed = pk_mod.pack_conv3x3(lay, bits, DEV, bn, stt)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, cout)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  cnt = torch.zeros((B, T, cout), device=DEV, dtype=torch.int32) if cin != 2 else None
  s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, cout, True, _lib.IMPL_SIMT, batch_major=True,
                       counts=cnt)
  assert np.array_equal(acc, info["acc"]) and np.array_equal(s, s_ref) and np.array_equal(u, info["u"])
  if cnt is not None:
    assert np.array_equal(cnt.cpu().numpy(), info["spikes"].sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2))


@pytest.mark.parametrize("impl", impls())
@pytest.mark.parametrize("keep", [0.5, 0.1, 0.0])
def test_block_sparse_slab_skip(cuda_lib, oracle_lib, impl, keep):
  """north_star item 4: weight K-slabs (tap x 32 input channels x all outputs) zeroed by a
  block-structured mask are skipped by the MMA issuer.  Unstructured magnitude masks never
  produce such slabs (SURVEY.md F10), so the path is exercised with structured masks:
  50 % / 90 % / 100 % of the 36 slabs removed (the last one = a fully pruned layer)."""
  rng = np.random.default_rng(int(keep * 100) + 3)
  T, B, H = 3, 2, 16
  lay, _, bn, stt = make_layer(rng, 128, 128, 8, 0.3)
  slab_keep = rng.uniform(size=36) < keep
  mask = lay["prune_0"]["mask"].reshape(9, 4, 32, 128).copy()
  mask[~slab_keep.reshape(9, 4)] = 0
  lay["prune_0"]["mask"] = mask.reshape(3, 3, 128, 128)
  a = lay["DuQ_0"]["a"][0]
  q = ref_int.duq_levels_c(lay["kernel"], lay["prune_0"]["mask"], a, 8)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  nz = packed.slab_nz.cpu().numpy().astype(bool)
  assert np.array_equal(nz, (q.reshape(9, 4, 32, 128) != 0).any(axis=(2, 3)).reshape(-1))
  assert nz.sum() <= slab_keep.sum() and (keep > 0 or nz.sum() == 0)
  x = (rng.uniform(size=(T, B, H, H, 128)) < 0.3).astype(np.uint8)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, impl, batch_major=True)
  assert np.array_equal(acc, info["acc"]) and np.array_equal(s, s_ref) and np.array_equal(u, info["u"])
  s_fast, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, impl, batch_major=True,
                          dumps=False)
  assert np.array_equal(s_fast, s_ref)


def test_spiking_conv_tau_not_power_of_two_and_extremes(cuda_lib, oracle_lib):
  rng = np.random.default_rng(77)
  lay, q, bn, stt = make_layer(rng, 128, 128, 8, 0.5)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  for x in (np.zeros((2, 1, 8, 8, 128), np.uint8), np.ones((2, 1, 8, 8, 128), np.uint8)):
    s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, tau=3.0, want=True)
    s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_SIMT, tau=3.0)
    assert np.array_equal(acc, info["acc"]) and np.array_equal(s, s_ref) and np.array_equal(u, info["u"])


@pytest.mark.parametrize("impl", impls())
@pytest.mark.parametrize("pool", [False, True])
def test_spiking_conv_att_within_tolerance(cuda_lib, oracle_lib, impl, pool):
  """conv5: real-valued input att * spikes.  SIMT: fp32 FMAs (summation order differs
  from the float64 oracle); tcgen05: 24-bit fixed-point attention as three exact
  int8 contractions.  Bar: membrane <= 1e-5 relative, flips <= 1e-4."""
  rng = np.random.default_rng(31)
  T, B, H = 4, 3, 8
  lay, q, bn, stt = make_layer(rng, 128, 128, 8, 0.5)
  x = (rng.uniform(size=(T, B, H, H, 128)) < 0.3).astype(np.uint8)
  att = rng.uniform(0.0, 1.0, size=(T, B, 128)).astype(F32)
  att[0, 0, :4] = [1.0, 0.0, 1e-8, 0.99999994]                 # saturated / vanishing attention
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  accf = ref_int.conv3x3_att_accf(x, att, q)
  s_ref, u_ref = ref_int.lif_from_acc(accf, scale, bias)
  cnt = torch.zeros((B, T, 128), device=DEV, dtype=torch.int32)
  s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl, att=att,
                       batch_major=True, counts=cnt)
  assert preact_err(acc, accf, scale, bias) <= 1e-5
  # given the kernel's own accumulators the epilogue (LIF, pool, counts) is bit-exact
  s2, u2 = ref_int.lif_from_acc(acc, scale, bias)
  assert np.array_equal(u, u2)
  assert np.array_equal(s, ref_int.maxpool2_u8(s2) if pool else s2)
  assert np.array_equal(cnt.cpu().numpy(), s2.sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2))
  assert np.mean(s2 != s_ref) <= 1e-4
  same = (s2 == s_ref).all(axis=0)
  assert np.max((np.abs(u - u_ref) / np.maximum(np.abs(u_ref), 1.0))[same]) <= 1e-5


def test_qconv_plain_forward(cuda_lib, oracle_lib):
  from snnquantprune_b200 import QuantConv, QuantConfig
  rng = np.random.default_rng(41)
  lay, q, _, _ = make_layer(rng, 128, 128, 8, 0.5)
  x = (rng.uniform(size=(2, 8, 8, 128)) < 0.3).astype(np.uint8)
  conv = QuantConv(features=128, kernel_size=(3, 3), padding=((1, 1), (1, 1)), use_bias=False,
                   config=QuantConfig(bits=8, prune_percentage=0.5), bits=8)
  y = conv.apply({"params": lay}, dev(x)).cpu().numpy()
  acc = ref_int.conv3x3_acc(x, q)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, n=128)
  assert np.array_equal(y, ref_int.fmaf(acc.astype(F32), scale, bias))
  ref_f = ref_snn.quant_conv(lay, x.astype(F32), 8, ((1, 1), (1, 1)))     # reference op order
  assert np.max(np.abs(y - ref_f)) <= 1e-5 * max(1.0, np.abs(ref_f).max())


# ------------------------------------------------------------ dense / tcja ----
def run_dense(lib, x, wq, scale, bias, N, att=None, att_mod=0, impl=_lib.IMPL_SIMT):
  """x: numpy (T,B,K); the device copy is batch-major [B][T][K] (rows (b,t) contiguous)."""
  T, B, K = x.shape
  xs = dev(np.ascontiguousarray(np.swapaxes(x, 0, 1)))
  spikes = torch.empty((T, B, N), device=DEV, dtype=torch.uint8)
  u = torch.empty((B, N), device=DEV, dtype=torch.float32)
  acc = torch.empty((T, B, N), device=DEV, dtype=torch.float32 if att is not None else torch.int32)
  p = BlockParams()
  p.T, p.B, p.H, p.W, p.Cin, p.Cout = T, B, 1, 1, K, N
  p.x_stride_t, p.x_stride_b = xs.stride(1), xs.stride(0)
  p.y_stride_t, p.y_stride_b = spikes.stride(0), spikes.stride(1)
  attd = None
  if att is not None:
    attd = dev(att); p.att_stride_t, p.att_stride_b = attd.stride(0), attd.stride(1)
  p.att_mod = att_mod
  p.tau, p.v_threshold, p.v_reset = 2.0, 1.0, 0.0
  p.impl = impl
  _lib.check(lib.snnqp_spiking_dense_fwd(p, P(xs), P(attd), P(wq), P(scale), P(bias), P(spikes), P(u), P(acc),
                                         _lib.stream()))
  torch.cuda.synchronize()
  return spikes.cpu().numpy(), u.cpu().numpy(), acc.cpu().numpy()


@pytest.mark.parametrize("impl", impls())
@pytest.mark.parametrize("T,B,K,N,bits", [(5, 3, 512, 110, 8), (3, 9, 100, 40, 4), (2, 1, 2048, 512, 2),
                                          (20, 19, 512, 110, 8), (4, 45, 256, 300, 8)])
def test_spiking_dense_binary_bit_exact(cuda_lib, oracle_lib, impl, T, B, K, N, bits):
  rng = np.random.default_rng(K + N)
  k = (rng.standard_normal((K, N)) * (5.0 / np.sqrt(K))).astype(F32)
  mask = ref_quant.local_mask(k, 0.5)
  a = ref_quant.gaussian_init(k, bits)
  lay = {"kernel": k, "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)}, "prune_0": {"mask": mask}}
  packed = pk_mod.pack_dense(lay, bits, DEV)
  q = ref_int.duq_levels_c(k, mask, a, bits)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], bits, n=N)
  x = (rng.uniform(size=(T, B, K)) < 0.2).astype(np.uint8)
  acc_ref = ref_int.dense_acc(x, q)
  s_ref, u_ref = ref_int.lif_from_acc(acc_ref, scale, bias)
  try:
    s, u, acc = run_dense(cuda_lib, x, packed.wq, packed.scale, packed.bias, N, impl=impl)
  except _lib.SnnqpError as e:
    if impl == _lib.IMPL_TCGEN05 and e.code == 3:
      pytest.skip("shape outside the tcgen05 dense kernel's envelope: " + str(e))
    raise
  assert np.array_equal(acc, acc_ref) and np.array_equal(s, s_ref) and np.array_equal(u, u_ref)
  assert s_ref.mean() > 0.01


@pytest.mark.parametrize("impl", impls())
@pytest.mark.parametrize("T,B", [(4, 5), (20, 11)])
def test_spiking_dense_att_within_tolerance(cuda_lib, oracle_lib, impl, T, B):
  rng = np.random.default_rng(55)
  K, N, Cc = 2048, 512, 128
  k = (rng.standard_normal((K, N)) * (7.0 / np.sqrt(K))).astype(F32)
  a = ref_quant.gaussian_init(k, 8)
  lay = {"kernel": k, "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)},
         "prune_0": {"mask": ref_quant.local_mask(k, 0.5)}}
  packed = pk_mod.pack_dense(lay, 8, DEV)
  q = ref_int.duq_levels_c(k, lay["prune_0"]["mask"], a, 8)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, n=N)
  x = (rng.uniform(size=(T, B, K)) < 0.15).astype(np.uint8)
  att = rng.uniform(0.05, 1, size=(T, B, Cc)).astype(F32)
  att_k = np.tile(att, (1, 1, K // Cc))                       # k % 128 -> channel
  accf = ref_int.dense_att_accf(x, att_k, q)
  s_ref, u_ref = ref_int.lif_from_acc(accf, scale, bias)
  s, u, acc = run_dense(cuda_lib, x, packed.wq, packed.scale, packed.bias, N, att=att, att_mod=Cc, impl=impl)
  assert preact_err(acc, accf, scale, bias) <= 1e-5
  assert np.mean(s != s_ref) <= 1e-4
  s2, u2 = ref_int.lif_from_acc(acc, scale, bias)
  assert np.array_equal(s, s2) and np.array_equal(u, u2)


def test_tcja_maxpool_vote_metrics(cuda_lib, oracle_lib):
  rng = np.random.default_rng(61)
  T, B, H, Cc = 6, 3, 8, 128
  s = (rng.uniform(size=(T, B, H, H, Cc)) < 0.2).astype(np.uint8)
  kt = (rng.standard_normal((4, T, T)) * 0.6).astype(F32); kc = (rng.standard_normal((4, Cc, Cc)) * 0.25).astype(F32)
  lays = []
  for k in (kt, kc):
    a = ref_quant.gaussian_init(k, 8)
    lays.append({"kernel": k, "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)},
                 "prune_0": {"mask": ref_quant.local_mask(k, 0.3)}})
  qt = pk_mod.pack_levels(lays[0], 8, DEV); qc = pk_mod.pack_levels(lays[1], 8, DEV)
  st, _ = pk_mod.fold_affine(lays[0]["DuQ_0"]["c"], 8, 1, DEV, extra_div=float(H * H))
  sc, _ = pk_mod.fold_affine(lays[1]["DuQ_0"]["c"], 8, 1, DEV, extra_div=float(H * H))
  sd = dev(s)
  att = torch.empty((T, B, Cc), device=DEV, dtype=torch.float32)
  cnt = torch.empty((B, T, Cc), device=DEV, dtype=torch.int32)
  p = BlockParams(); p.T, p.B, p.H, p.W, p.Cin, p.Cout = T, B, H, H, Cc, Cc
  p.x_stride_t, p.x_stride_b = sd.stride(0), sd.stride(1)
  p.att_stride_t, p.att_stride_b = att.stride(0), att.stride(1)
  _lib.check(cuda_lib.snnqp_tcja_fwd(p, P(sd), P(qt), P(qc), P(st), P(sc), P(cnt), P(att), _lib.stream()))
  att_ref, info = ref_int.tcja_att(s, qt.cpu().numpy(), st.item(), qc.cpu().numpy(), sc.item(), want=True)
  assert np.array_equal(cnt.cpu().numpy(), np.transpose(info["cnt"], (1, 0, 2)))
  got = att.cpu().numpy()
  # exact up to the device expf (<= 2 ulp): att must be one of the values that error allows
  cands, _ = attref.tcja_candidates(np.transpose(info["acc_t"], (2, 0, 1)), np.transpose(info["acc_c"], (1, 0, 2)),
                                    st.item(), sc.item())
  attref.tcja_check(got, cands, "k_tcja_att_mma")
  # against the reference-order float path (means, fp32 convs, sigmoid)
  y_ref, att_f = ref_snn.tcja({"t": lays[0], "c": lays[1]}, ("t", "c"), s.astype(F32), 8, return_att=True)
  assert np.max(np.abs(got - att_f)) <= 1e-5
  # maxpool
  y = torch.empty((T, B, H // 2, H // 2, Cc), device=DEV, dtype=torch.uint8)
  p.y_stride_t, p.y_stride_b = y.stride(0), y.stride(1)
  _lib.check(cuda_lib.snnqp_maxpool2_fwd(p, P(sd), P(y), _lib.stream()))
  assert np.array_equal(y.cpu().numpy(), ref_int.maxpool2_u8(s))
  # vote + metrics
  sp = (rng.uniform(size=(T, B, 110)) < 0.25).astype(np.uint8)
  spd = dev(sp)
  logits = torch.empty((B, 11), device=DEV, dtype=torch.float32)
  _lib.check(cuda_lib.snnqp_vote_fwd(P(spd), T, B, 110, 10, spd.stride(0), spd.stride(1), P(logits), _lib.stream()))
  assert np.array_equal(logits.cpu().numpy(), ref_int.vote(sp))
  labels = np.array([int(np.argmax(ref_int.vote(sp)[0])), 3, 5], np.int32)
  out = torch.zeros(2, device=DEV)
  labd = dev(labels)
  _lib.check(cuda_lib.snnqp_eval_metrics(P(logits), P(labd), B, 11, P(out), _lib.stream()))
  m = ref_snn.eval_metrics(ref_int.vote(sp), labels)
  assert out[0].item() == float(m["accuracy"].sum())
  assert np.isclose(out[1].item() / (B * 11), float(m["loss"]), rtol=1e-5)


# ------------------------------------------------------------ whole network ----
def engine_for(v, bits, T, H, impl=_lib.IMPL_AUTO, chunk=16, lif_mode=_lib.LIF_EXACT):
  """Bit-exact comparisons run the reference-op-order LIF (the engine's default is LIF_FAST for conv1)."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet
  return CextNetEngine(pack_cextnet(v, bits, T, H, device=DEV), impl=impl, chunk=chunk, lif_mode=lif_mode)


@pytest.mark.parametrize("name", ["cextnet_T4_H32_b8_p50", "cextnet_T3_H32_b4_p80", "cextnet_T3_H32_b2_p90"])
def test_network_against_golden_fixture(cuda_lib, name):
  z = np.load(os.path.join(GOLD, name + ".npz"))
  m = json.loads(str(z["meta"]))
  v = synthetic.make_variables(bits=m["bits"], prune_percentage=m["prune"], T=m["T"], H=m["H"], seed=m["seed_w"])
  fr = synthetic.make_frames(m["B"], m["T"], m["H"], m["H"], seed=m["seed_x"])
  import sys
  sys.path.insert(0, GOLD)
  import make_golden
  # same image on the GPU box: a different stream is a broken environment, not a reason to skip
  assert make_golden.variables_digest(v) == m["variables_sha"] and make_golden.sha(fr) == m["frames_sha"], \
      "numpy RNG stream differs from the one the fixture was made with"
  c = {}
  logits = engine_for(v, m["bits"], m["T"], m["H"]).forward(dev(fr), collect=c).cpu().numpy()
  for k in ("s1", "s2", "s3", "s4"):          # integer-input layers: bit-exact
    got = np.swapaxes(c[k].cpu().numpy(), 0, 1)
    assert np.array_equal(np.packbits(got.reshape(-1)), z[k + "_bits"]), k
  assert np.max(np.abs(np.swapaxes(c["att4"].cpu().numpy(), 0, 1) - z["att4"]) / z["att4"]) <= 2e-6
  nflip = 0
  for k in ("s5", "d1", "d2"):                # downstream of expf / fp32 sums: flip budget
    got = np.swapaxes(c[k].cpu().numpy(), 0, 1).reshape(-1)
    ref = np.unpackbits(z[k + "_bits"])[:got.size]
    assert np.mean(got != ref) <= 1e-4, k
    nflip += int((got != ref).sum())
  tol = 1e-6 + min(nflip, 16) / (m["T"] * 10)   # one flipped output spike = 1 / (T * 10) of a logit
  assert np.max(np.abs(logits - z["logits_int"])) <= tol
  assert np.max(np.abs(logits - z["logits_float"])) <= tol


def test_network_layerwise_teacher_forced_and_float_path(cuda_lib, oracle_lib):
  """Free-running GPU forward; the oracle is fed the GPU's own attention so that
  every integer-input layer can be compared bit for bit, then the whole thing is
  compared with the reference-order float path under the north-star tolerances."""
  bits, p, T, H, B = 8, 0.5, 6, 64, 3
  v = synthetic.make_variables(bits=bits, prune_percentage=p, T=T, H=H, seed=33)
  fr = synthetic.make_frames(B, T, H, H, seed=34)
  c = {}
  logits = engine_for(v, bits, T, H).forward(dev(fr), collect=c).cpu().numpy()
  tb = lambda k: np.ascontiguousarray(np.swapaxes(c[k].cpu().numpy(), 0, 1))
  forced = {"att4": tb("att4"), "s5": tb("s5"), "att5": tb("att5"), "d1": tb("d1")}
  co = {}
  lo = ref_net.forward(ref_net.pack_network(v, bits, H), fr, collect=co, forced=forced)
  for i, k in enumerate(("s1", "s2", "s3", "s4"), 1):
    assert np.array_equal(tb(k), co[k]), k
    assert np.array_equal(c[f"conv{i}_acc"].cpu().numpy(), co[f"conv{i}_acc"]), f"conv{i} accumulators"
    assert np.array_equal(c[f"conv{i}_u"].cpu().numpy(), co[f"conv{i}_u"]), f"conv{i} membrane"
  assert np.array_equal(tb("p4"), co["p4"])
  assert np.max(np.abs(tb("att4") - co["att4"]) / co["att4"]) <= 2e-6
  acc5 = c["conv5_acc"].cpu().numpy()
  pk5 = ref_net.pack_network(v, bits, H)["conv"][4]
  assert preact_err(acc5, co["conv5_acc"], pk5["scale"], pk5["bias"]) <= 1e-5
  assert np.mean(tb("s5") != co["s5"]) <= 1e-4
  assert np.array_equal(c["dense2_acc"].cpu().numpy(), co["dense2_acc"])
  assert np.array_equal(tb("d2"), co["d2"])
  assert np.array_equal(logits, lo)
  # reference-order float path, free running
  cf = {}
  lf = ref_snn.cextnet_forward(v, fr, bits, collect=cf)
  nflip = 0
  for k, kf in (("s1", "pool1"), ("s2", "pool2"), ("s3", "pool3"), ("s4", "conv4_spikes"),
                ("s5", "conv5_spikes"), ("d1", "dense1_spikes"), ("d2", "dense2_spikes")):
    d = tb(k) != (cf[kf] != 0)
    assert np.mean(d) <= 1e-4, k
    nflip += int(d.sum())
  for i in range(1, 6):
    ug, uf = c[f"conv{i}_u"].cpu().numpy(), cf[f"conv{i}_u"]
    bad = np.abs(ug - uf) > 1e-5 * np.maximum(np.abs(uf), 1.0)
    # every neuron within 1e-5 unless a counted flip sits upstream of it (3x3xC fan-out per layer and step)
    assert bad.sum() <= 2048 * nflip, (i, int(bad.sum()), nflip)
  assert np.max(np.abs(logits - lf)) <= 1e-6 + min(nflip, 16) / (T * 10)


def test_config3_T10_ten_classes(cuda_lib, oracle_lib):
  """BASELINE.json configs[3]: the spikingjelly-input variant -- same graph with T=10 and 10
  classes (dense2 -> 100 outputs, TCJA conv_t features = 10), 8-bit weights."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet
  bits, T, H, B, ncls = 8, 10, 64, 2, 10
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, num_classes=ncls, seed=41)
  fr = synthetic.make_frames(B, T, H, H, seed=42)
  eng = CextNetEngine(pack_cextnet(v, bits, T, H, num_classes=ncls, device=DEV), lif_mode=_lib.LIF_EXACT)
  c = {}
  logits = eng.forward(dev(fr), collect=c).cpu().numpy()
  assert logits.shape == (B, ncls)
  tb = lambda k: np.ascontiguousarray(np.swapaxes(c[k].cpu().numpy(), 0, 1))
  forced = {"att4": tb("att4"), "s5": tb("s5"), "att5": tb("att5"), "d1": tb("d1")}
  co = {}
  lo = ref_net.forward(ref_net.pack_network(v, bits, H), fr, collect=co, forced=forced)
  for k in ("s1", "s2", "s3", "s4"):
    assert np.array_equal(tb(k), co[k]), k
  assert np.array_equal(tb("d2"), co["d2"]) and np.array_equal(logits, lo)
  lf = ref_snn.cextnet_forward(v, fr, bits)
  assert np.max(np.abs(logits - lf)) <= 2.0 / (T * 10)
  assert np.array_equal(eng.forward(dev(fr)).cpu().numpy(), logits)      # production path, same logits


def test_fused_tail_equals_instrumented_tail(cuda_lib):
  """The production forward (pooled spikes + spike counts fused into the conv
  epilogues, no un-pooled tensors) must give exactly the logits of the
  instrumented forward that materialises every intermediate; so must a CUDA-graph replay."""
  bits, T, H, B = 8, 20, 128, 3
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  frd = dev(synthetic.make_frames(B, T, H, H, seed=4))
  eng = engine_for(v, bits, T, H)
  l_fused = eng.forward(frd).cpu().numpy()
  l_inst = eng.forward(frd, collect={}).cpu().numpy()
  assert np.array_equal(l_fused, l_inst)
  host = torch.from_numpy(synthetic.make_frames(B, T, H, H, seed=4)).pin_memory()
  out_host = torch.empty((B, 11), dtype=torch.float32).pin_memory()
  eng2 = engine_for(v, bits, T, H, chunk=2)                   # 2 chunks: exercises the double-buffered H2D path
  eng2.forward_host(host, out_host); eng2.forward_host(host, out_host)
  torch.cuda.synchronize()
  assert np.array_equal(out_host.numpy(), l_fused)
  l_graph = eng.forward_graph(frd).cpu().numpy()
  l_graph2 = eng.forward_graph(frd).cpu().numpy()
  assert np.array_equal(l_graph, l_fused) and np.array_equal(l_graph2, l_fused)


def test_full_size_properties(cuda_lib):
  """BASELINE sizes (H=128, T=20): size-independent properties -- samples are
  independent (batch permutation equivariance, chunking invariance) and a
  replayed forward is bit-identical."""
  bits, T, H, B = 8, 20, 128, 6
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  fr = synthetic.make_frames(B, T, H, H, seed=0)
  frd = dev(fr)
  eng = engine_for(v, bits, T, H, chunk=4)
  l1 = eng.forward(frd).cpu().numpy()
  l2 = eng.forward(frd).cpu().numpy()
  assert np.array_equal(l1, l2)
  perm = np.array([3, 0, 5, 1, 4, 2])
  lp = eng.forward(dev(fr[perm])).cpu().numpy()
  assert np.array_equal(lp, l1[perm])
  l3 = engine_for(v, bits, T, H, chunk=1).forward(frd).cpu().numpy()
  assert np.array_equal(l3, l1)
  assert l1.std() > 0 and 0.0 < l1.mean() < 1.0


def test_full_size_one_sample_against_oracle(cuda_lib, oracle_lib):
  """configs[0] geometry (T=20, 128x128), one sample, integer-path oracle."""
  bits, T, H, B = 8, 20, 128, 1
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  fr = synthetic.make_frames(B, T, H, H, seed=0)
  c = {}
  logits = engine_for(v, bits, T, H).forward(dev(fr), collect=c).cpu().numpy()
  tb = lambda k: np.ascontiguousarray(np.swapaxes(c[k].cpu().numpy(), 0, 1))
  forced = {"att4": tb("att4"), "s5": tb("s5"), "att5": tb("att5"), "d1": tb("d1")}
  co = {}
  lo = ref_net.forward(ref_net.pack_network(v, bits, H), fr, collect=co, forced=forced)
  for k in ("s1", "s2", "s3", "s4"):
    assert np.array_equal(tb(k), co[k]), k
  assert np.array_equal(c["conv2_acc"].cpu().numpy(), co["conv2_acc"])
  assert np.mean(tb("s5") != co["s5"]) <= 1e-4
  assert np.array_equal(logits, lo)
  rates = {k: float(tb(k).mean()) for k in ("s1", "s2", "s3", "s4", "s5", "d1", "d2")}
  assert min(rates.values()) > 0.01, rates


def test_error_behaviour(cuda_lib):
  p = BlockParams(); p.T, p.B, p.H, p.W, p.Cin, p.Cout = 1, 1, 7, 8, 128, 128
  p.tau = 2.0
  d = torch.zeros(16, device=DEV, dtype=torch.uint8)
  rc = cuda_lib.snnqp_spiking_conv3x3_fwd(p, P(d), None, P(d), P(d), P(d), P(d), None, None, _lib.stream())
  assert rc == 3 and b"even" in cuda_lib.snnqp_last_error()
  p.H = 8; p.tau = 0.0
  rc = cuda_lib.snnqp_spiking_conv3x3_fwd(p, P(d), None, P(d), P(d), P(d), P(d), None, None, _lib.stream())
  assert rc == 1
  rc = cuda_lib.snnqp_pack_levels(P(d), None, P(d), 9, 4, P(d), _lib.stream())
  assert rc == 3
  rc = cuda_lib.snnqp_vote_fwd(P(d), 2, 1, 11, 10, 11, 22, P(d), _lib.stream())
  assert rc == 1
  lay = {"kernel": np.zeros((3, 3, 128, 128), F32), "DuQ_0": {"a": np.array([-1.0], F32), "c": np.array([-1.0], F32)},
         "prune_0": {"mask": np.ones((3, 3, 128, 128), F32)}}
  with pytest.raises(NotImplementedError):
    pk_mod.pack_conv3x3(lay, 8, DEV)


def test_auto_impl_notes_simt_fallback_once(cuda_lib, oracle_lib):
  """SNNQP_IMPL_AUTO outside the tcgen05 envelopes still runs (dp4a kernels) but says so once through
  snnqp_last_error(): a 10x performance cliff must not be silent."""
  rng = np.random.default_rng(5)
  lay, q, bn, stt = make_layer(rng, 128, 128, 8, 0.5)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  x = (rng.uniform(size=(2, 1, 6, 6, 128)) < 0.3).astype(np.uint8)          # H = W = 6: no tcgen05 kernel takes it
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_AUTO)
  assert np.array_equal(s, s_ref) and np.array_equal(acc, info["acc"])
  msg = cuda_lib.snnqp_last_error().decode()
  assert ("SIMT" in msg and "reported once" in msg) or msg == "" or "note" not in msg      # first fallback of the process says so


def test_spiking_block_facade(cuda_lib, oracle_lib):
  from snnquantprune_b200 import SpikingBlock, QuantConv, QuantDense, QuantConfig, multi_step_LIF, BatchNorm, atan
  rng = np.random.default_rng(71)
  lay, q, bn, stt = make_layer(rng, 128, 128, 8, 0.5)
  cfg = QuantConfig(bits=8, prune_percentage=0.5)
  blk = SpikingBlock(connection_fn=QuantConv(features=128, kernel_size=(3, 3), padding=((1, 1), (1, 1)),
                                             use_bias=False, config=cfg, bits=8),
                     neural_dynamics=multi_step_LIF(tau=2.0, spike_fn=atan), norm_fn=BatchNorm())
  x = (rng.uniform(size=(3, 2, 8, 8, 128)) < 0.3).astype(np.uint8)
  xd = dev(x)
  carry = SpikingBlock.initialize_carry(xd, blk.connection_fn, blk.norm_fn)
  assert tuple(carry.shape) == (2, 8, 8, 128) and float(carry.abs().sum()) == 0.0
  variables = {"params": {"connection_fn": lay, "norm_fn": bn}, "batch_stats": {"norm_fn": stt}}
  u, s = blk.apply(variables, carry, xd)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=False, want=True)
  assert np.array_equal(s.cpu().numpy(), s_ref) and np.array_equal(u.cpu().numpy(), info["u"])
  # un-fused LIF step mirrors the reference op order
  lif = multi_step_LIF(tau=2.0, spike_fn=atan)
  u0 = torch.zeros(5, device=DEV); xin = torch.tensor([2.0, 1.9999, 0.5, -1.0, 4.0], device=DEV)
  u1, s1 = lif(u0, xin)
  ur, sr = ref_snn.lif_step(np.zeros(5, F32), xin.cpu().numpy())
  assert np.array_equal(u1.cpu().numpy(), ur) and np.array_equal(s1.cpu().numpy(), sr)


def test_evaluate_driver_matches_oracle_metrics(cuda_lib):
  """evaluate() (the reference's eval loop, examples/eval.py:53-139) over pinned host batches through
  forward_host + snnqp_eval_metrics == compute_metrics of the oracle on the same logits."""
  from snnquantprune_b200.eval import evaluate
  bits, T, H, B = 8, 4, 32, 5
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=51)
  eng = engine_for(v, bits, T, H, chunk=2)
  rng = np.random.default_rng(52)
  batches, losses, accs = [], [], []
  for i in range(3):
    fr = synthetic.make_frames(B, T, H, H, seed=60 + i)
    lab = rng.integers(0, 11, size=B)
    batches.append({"dvs_matrix": torch.as_tensor(fr).pin_memory(), "label": torch.as_tensor(lab)})
    lg = eng.forward(dev(fr)).cpu().numpy()
    m = ref_snn.eval_metrics(lg, lab)
    losses.append(float(m["loss"])); accs.append(float(np.mean(m["accuracy"])))
  got = evaluate(lambda f: eng.forward_host(f), batches, num_classes=11)
  assert got["samples"] == 3 * B and got["steps"] == 3
  assert np.isclose(got["loss"], np.mean(losses), rtol=1e-5)
  assert np.isclose(got["accuracy"], np.mean(accs), atol=1e-7)


def test_packed_file_round_trip_gives_identical_logits(cuda_lib, tmp_path):
  """pack -> save_packed -> load_packed -> forward: the on-disk format is device-layout-exact."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet
  from snnquantprune_b200 import checkpoint_io as cio
  bits, T, H, B = 4, 5, 64, 3
  v = synthetic.make_variables(bits=bits, prune_percentage=0.8, T=T, H=H, seed=71)
  fr = dev(synthetic.make_frames(B, T, H, H, seed=72))
  pk = pack_cextnet(v, bits, T, H, device=DEV)
  want = CextNetEngine(pk).forward(fr).cpu().numpy()
  path = str(tmp_path / "net.snnqp")
  cio.save_packed(pk, path)
  back = cio.load_packed(path, device=DEV)
  for k, t in cio._tensors_of(pk).items():
    assert torch.equal(t, cio._tensors_of(back)[k]), k
  assert np.array_equal(CextNetEngine(back).forward(fr).cpu().numpy(), want)


def test_spike_tile_skip_on_structured_frames(cuda_lib):
  """Spike-side tile skip (SURVEY.md 8f N3): with bit-packed spikes an all-zero input box issues no MMAs.  On
  spatially structured DVS-like frames (a moving blob on a silent sensor) most boxes are empty; the logits must be
  exactly those of the u8 path (which never skips), and on i.i.d. frames nothing is skipped."""
  import ctypes
  from snnquantprune_b200 import CextNetEngine, pack_cextnet
  bits, T, H, B = 8, 20, 128, 4
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  pk = pack_cextnet(v, bits, T, H, device=DEV)
  sk, tot = ctypes.c_int64(0), ctypes.c_int64(0)
  rates = {}
  for name, fr in (("blob", synthetic.make_frames_blob(B, T, H, H, seed=3)), ("iid", synthetic.make_frames(B, T, H, H, seed=3))):
    frd = dev(fr)
    want = CextNetEngine(pk, lif_mode=_lib.LIF_EXACT, packed_spikes=False).forward(frd).cpu().numpy()
    _lib.check(cuda_lib.snnqp_tile_skip_stats(None, None, 1))
    got = CextNetEngine(pk, lif_mode=_lib.LIF_EXACT, packed_spikes=True).forward(frd).cpu().numpy()
    _lib.check(cuda_lib.snnqp_tile_skip_stats(ctypes.byref(sk), ctypes.byref(tot), 1))
    assert np.array_equal(got, want), name
    assert tot.value == B * T * (32 + 8 + 2)               # strips of conv2 / conv3 / conv4 per sample-step
    rates[name] = sk.value / tot.value
  assert rates["blob"] >= 0.5 and rates["iid"] == 0.0, rates


@pytest.mark.parametrize("lif_mode", [_lib.LIF_EXACT, _lib.LIF_FAST])
def test_fused_head_equals_separate_launches(cuda_lib, lif_mode):
  """snnqp_spiking_head_fwd (conv1 of chunk k+1 and conv2 of chunk k in one persistent kernel, TMEM / shared memory /
  registers carved between the two roles) gives exactly the spikes of the two separate launches: per-launch check
  of both halves, conv1-only and conv2-only launches, then whole forwards over several (ragged) chunk schedules."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet
  bits, T, H, B = 8, 20, 128, 40
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  pk = pack_cextnet(v, bits, T, H, device=DEV)
  fr = dev(synthetic.make_frames(B, T, H, H, seed=8))
  sep = CextNetEngine(pk, chunk=B, lif_mode=lif_mode, fused_head=False)
  fus = CextNetEngine(pk, chunk=B, lif_mode=lif_mode, fused_head=True)
  C = pk.channels
  # separate launches
  s1 = torch.empty((B, T, H // 2, H // 2, C // 8), device=DEV, dtype=torch.uint8)
  s2 = torch.empty((B, T, H // 4, H // 4, C // 8), device=DEV, dtype=torch.uint8)
  sep._conv(0, fr, s1, B, H, 2, 1)
  sep._conv(1, s1, s2, B, H // 2, C, 1)
  # fused: both halves at once on different sample ranges (conv1 on all B, conv2 on the first 17 samples of s1)
  f1 = torch.zeros_like(s1); f2 = torch.zeros_like(s2)
  fus._head_fused(fr, B, f1, s1, 17, f2)
  assert torch.equal(f1, s1), "conv1 half"
  assert torch.equal(f2[:17], s2[:17]), "conv2 half"
  # each half alone
  f1.zero_(); f2.zero_()
  fus._head_fused(fr[:5], 5, f1, None, 0, None)
  assert torch.equal(f1[:5], s1[:5])
  fus._head_fused(None, 0, None, s1, B, f2)
  assert torch.equal(f2, s2)
  # whole forward, several chunk schedules (single chunk, equal chunks, ragged tail)
  want = sep.forward(fr)
  for chunk in (B, 20, 37, 16):
    got = CextNetEngine(pk, chunk=chunk, lif_mode=lif_mode, fused_head=True).forward(fr)
    assert torch.equal(got, want), chunk
