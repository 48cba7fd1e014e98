"""The attention path (TCJA -> conv5 on att4 * pool(s4) -> TCJA -> dense1 on att5 * pool(s5)) bit for bit against an
emulation of its arithmetic (tests/attref.py).

- conv5 / dense1 on tcgen05 (k_conv_att_umma, k_dense_umma<3>): 24-bit fixed-point att (round to nearest even, 1.0
  clamped to 1 - 2^-24), three exact byte-plane contractions, the fp32 recombination in its fixed order.  Accumulators,
  spikes (pooled and un-pooled), final membranes and spike counts must equal the emulation exactly.
- conv5 / dense1 on SIMT (k_conv3x3_simt<true>, k_dense_simt<true>): one sequential fp32 fma chain per output.
- TCJA (k_tcja_att_mma, k_tcja_att, k_tcja_att_dp4a): integer counts exact; att one of the values the documented expf
  error (<= 2 ulp) allows.

CPU tests check the emulation itself: the fixed-point edges, the recombination against a direct fp32 evaluation, the
emulated accumulators against float64 within their derived bounds, and a float64 rounding band on the emulated LIF
(every decided spike equals float64).  Since the gpu tests show that each kernel IS its emulation, the band holds for
the kernels too."""
import multiprocessing
import os

import numpy as np
import pytest
import torch

import attref as ar
from oracle import ref_int, ref_quant
from snnquantprune_b200 import _lib
from snnquantprune_b200 import pack as pk_mod
from snnquantprune_b200._lib import BlockParams

F32 = np.float32
DEV = "cuda"
gpu = pytest.mark.gpu
P = _lib.ptr

# att values at the edges of the fixed-point conversion, with their 24-bit words (round half to even, clamp)
EDGES = [
    (0.0, 0),
    (2.0 ** -25, 0),                       # 0.5 -> tie to even 0
    (3 * 2.0 ** -25, 2),                   # 1.5 -> 2
    (5 * 2.0 ** -25, 2),                   # 2.5 -> 2
    (255 * 2.0 ** -24, 0x0000FF),
    (2.0 ** -16, 0x000100),                # carry into b1
    (2.0 ** -8 - 2.0 ** -24, 0x00FFFF),
    (2.0 ** -8, 0x010000),                 # carry into b2
    (0.5 - 2.0 ** -26, 0x800000),          # not an fp32: the fp32 value is 0.5
    (0.5 - 2.0 ** -25, 0x800000),          # 2^23 - 0.5 -> tie to even 2^23
    (0.5 - 3 * 2.0 ** -26, 0x7FFFFF),      # 2^23 - 0.75
    (1.0 - 2.0 ** -24, 0xFFFFFF),
    (1.0, 0xFFFFFF),                       # 2^24 clamped
]
EDGE_ATT = np.array([a for a, _ in EDGES], F32)


def dev(a):
  return torch.as_tensor(np.ascontiguousarray(a), device=DEV)


def conv_layer(seed, mask_keep=None, const_q=None):
  """A 128 -> 128 conv5 layer with BatchNorm; mask_keep: number of the 36 K-slabs kept (block-sparse); const_q: every
  level +127 or -127 (all weights at the clip)."""
  rng = np.random.default_rng(seed)
  k = (rng.standard_normal((3, 3, 128, 128)) * 0.2).astype(F32)
  mask = ref_quant.local_mask(k, 0.5)
  a = ref_quant.gaussian_init(k, 8)
  if const_q is not None:
    k = np.full(k.shape, const_q * 2 * a, F32)
    mask = np.ones_like(k)
  if mask_keep is not None:
    keep = np.zeros(36, bool)
    keep[rng.permutation(36)[:mask_keep]] = True
    mask = mask.reshape(9, 4, 32, 128).copy()
    mask[~keep.reshape(9, 4)] = 0
    mask = mask.reshape(3, 3, 128, 128)
  lay = {"kernel": k, "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)}, "prune_0": {"mask": mask}}
  q = ref_int.duq_levels_c(k, mask, a, 8)
  energy = np.maximum((q.astype(np.float64).reshape(-1, 128) ** 2).sum(0), 1.0) * (a / 127) ** 2
  bn = dict(scale=rng.uniform(0.8, 1.2, 128).astype(F32), bias=(0.5 + 0.1 * rng.standard_normal(128)).astype(F32))
  stt = dict(mean=(0.02 * rng.standard_normal(128)).astype(F32), var=(0.25 * energy).astype(F32))
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  return lay, q, bn, stt, scale, bias


def dense_layer(seed, K=2048, N=512, const_q=None):
  rng = np.random.default_rng(seed)
  k = (rng.standard_normal((K, N)) * (7.0 / np.sqrt(K))).astype(F32)
  a = ref_quant.gaussian_init(k, 8)
  mask = ref_quant.local_mask(k, 0.5)
  if const_q is not None:
    k = np.full(k.shape, const_q * 2 * a, F32)
    mask = np.ones_like(k)
  lay = {"kernel": k, "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)}, "prune_0": {"mask": mask}}
  q = ref_int.duq_levels_c(k, mask, a, 8)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, n=N)
  return lay, q, scale, bias


def edge_att(rng, T, B, C=128):
  """att with every edge value at every channel position (rotated over (t, b)), the rest uniform in [0, 1]."""
  att = rng.uniform(0.0, 1.0, size=(T, B, C)).astype(F32)
  n = len(EDGE_ATT)
  for i in range(T * B):
    t, b = divmod(i, B)
    sel = (np.arange(C) + i) % (2 * n)
    att[t, b, sel < n] = EDGE_ATT[sel[sel < n]]
  return att


# =============================================================================================== CPU: the oracle ====
def test_att_fix24_edge_table():
  got = ar.att_fix24(EDGE_ATT)
  assert got.tolist() == [w for _, w in EDGES]
  b2, b1, b0 = ar.att_bytes(EDGE_ATT)
  assert ((b2 << 16) | (b1 << 8) | b0).tolist() == [w for _, w in EDGES]
  assert ar.att_bytes(np.array([2.0 ** -16], F32)) == (0, 1, 0)
  # the fixed point misses att by <= 2^-25, or 2^-24 at the clamp
  a = np.concatenate([EDGE_ATT, np.random.default_rng(0).uniform(0, 1, 10000).astype(F32)])
  err = np.abs(a.astype(np.float64) - ar.att_fix24(a) * 2.0 ** -24)
  assert np.all(err <= ar.fix_bound(a)) and err.max() == 2.0 ** -24


def test_combine_matches_direct_fp32(oracle_lib):
  """att_combine's emulation against C fmaf on the converted planes, with |S_i| below and above 2^24 (where the
  int -> float conversions and the fmas round)."""
  rng = np.random.default_rng(1)
  for lim in (2 ** 20, 2 ** 24, 2 ** 27, 2 ** 31 - 1):
    S = rng.integers(-lim, lim, size=(3, 50000), dtype=np.int64)
    S[:, :8] = np.array([lim - 1, -lim, 2 ** 24 + 1, 2 ** 24 + 3, -(2 ** 24) - 1, 0, 1, lim // 3])[None, :]
    a = S.astype(np.int32).astype(F32)                  # (a2, a1, a0), each conversion rounded to nearest
    f1 = ref_int.fmaf(a[1], F32(256), a[2])
    f = ref_int.fmaf(a[0], F32(65536), f1)
    want = (f * F32(2.0 ** -24)).astype(F32)
    got = ar.combine(S[0], S[1], S[2])
    assert np.array_equal(got, want), lim
  # below 2^24 every plane value is exact: the combine is exact while f stays below 2^24 too
  S = rng.integers(0, 2 ** 8, size=(3, 1000))
  assert np.array_equal(ar.combine(S[0] * 0, S[1], S[2]).astype(np.float64), (S[1] * 256.0 + S[2]) * 2.0 ** -24)


def _f64_truth(x, att, q, dense=False):
  """Exact sum att x q (att taken as a real, x != 0 a spike) in float64, and A = sum |att x q|, and the fixed-point
  term sum |q| fix_bound(att) over the spiking inputs."""
  m = (np.asarray(x) != 0).astype(np.float64)
  qa = np.abs(np.asarray(q).astype(np.int64))
  if dense:
    a64, fb = att.astype(np.float64), ar.fix_bound(att)
    f = lambda v, w: ar.dense_f64(v, w)
    ex, A, fix = f(m * a64, q), f(m * a64, qa), f(m * fb, qa)
  else:
    a64, fb = att.astype(np.float64)[:, :, None, None, :], ar.fix_bound(att)[:, :, None, None, :]
    ex, A, fix = ar.conv_f64(m * a64, q), ar.conv_f64(m * a64, qa), ar.conv_f64(m * fb, qa)
  return ex, A, fix


@pytest.mark.parametrize("kind", ["conv", "dense"])
def test_emulated_accumulators_within_derived_bound(oracle_lib, kind):
  """The emulated tcgen05 accumulator differs from the exact float64 sum by at most the fixed-point term plus the
  combine's five roundings (attref.tc_acc_bound); the emulated SIMT fma chain by at most gamma_n sum |att x q|.  Both
  at random att, at the edge table and at the all-on / att ~ 1 / |q| = 127 extreme where |S_i| > 2^24."""
  rng = np.random.default_rng(3)
  cases = []
  if kind == "conv":
    _, q, *_ = conv_layer(5)
    x = (rng.uniform(size=(2, 2, 8, 8, 128)) < 0.3).astype(np.uint8)
    cases.append((x, edge_att(rng, 2, 2), q))
    _, qx, *_ = conv_layer(6, const_q=-1)
    cases.append((np.ones((1, 2, 8, 8, 128), np.uint8), np.full((1, 2, 128), 1.0 - 2.0 ** -24, F32), qx))
  else:
    _, q, _, _ = dense_layer(7, K=2048, N=64)
    x = (rng.uniform(size=(2, 3, 2048)) < 0.2).astype(np.uint8)
    cases.append((x, np.tile(edge_att(rng, 2, 3), (1, 1, 16)), q))
    _, qx, _, _ = dense_layer(8, K=2048, N=64, const_q=1)
    cases.append((np.ones((1, 2, 2048), np.uint8), np.full((1, 2, 2048), 1.0, F32), qx))
  n = 1152 if kind == "conv" else 2048
  big = 0
  for x, att, q in cases:
    ex, A, fix = _f64_truth(x, att, q, dense=(kind == "dense"))
    tc, S = (ar.conv_att_tc_acc if kind == "conv" else ar.dense_att_tc_acc)(x, att, q, want=True)
    big += int((np.abs(S) > 2 ** 24).sum())
    err = np.abs(tc.astype(np.float64) - ex)
    bound = ar.tc_acc_bound(fix, S) + n * 2.0 ** -53 * A
    assert np.all(err <= bound), (kind, float((err / bound).max()))
    simt = (ar.conv_att_simt_acc if kind == "conv" else ar.dense_att_simt_acc)(x, att, q)
    err = np.abs(simt.astype(np.float64) - ex)
    assert np.all(err <= ar.gamma(n) * A * (1 + 2.0 ** -10) + n * 2.0 ** -53 * A), kind
  assert big > 0                       # the extreme case reached the rounding conversions


# ========================================================================== CPU: float64 band on the emulation ====
def att_band(ex, bnd, scale, bias, acc, label=""):
  """Float64 band of the reference-order LIF (tau 2, threshold 1, reset 0) fed by an accumulator within bnd of the
  exact sum ex.  Per step, h = (ex s + b) / 2, U = h + u / 2, and the kernel's U misses it by at most
      e_t = EPS (|h| + |h - u/2| + |U|) + |s| bnd / 2
  (v = fma(acc, s, b), v - u and u + d/2 round once each; the accumulator error enters v times |s|), times 1 + 2^-10
  plus 2^-50 (|U| + 1).  delta_t = e_t + delta_{t-1} / 2 while synchronised (as conv1_band in
  test_gpu_conv1_rounding_band.py).  The emulated accumulators acc then go through ref_int.lif_from_acc: every decided
  spike must equal float64 and every synchronised u_T lie within delta_T.  Returns the undecided fraction of the
  neuron-steps."""
  s, b = np.asarray(scale, F32).astype(np.float64), np.asarray(bias, F32).astype(np.float64)
  spk, u32 = ref_int.lif_from_acc(acc, scale, bias)
  T = ex.shape[0]
  u = np.zeros(ex.shape[1:])
  d = np.zeros(ex.shape[1:])
  sync = np.ones(ex.shape[1:], bool)
  undecided = 0
  for t in range(T):
    h = (ex[t] * s + b) * 0.5
    U = h + u * 0.5
    e = ar.EPS * (np.abs(h) + np.abs(h - u * 0.5) + np.abs(U)) + np.abs(s) * bnd[t] * 0.5
    e = e * (1.0 + 2.0 ** -10) + 2.0 ** -50 * (np.abs(U) + 1.0)
    d = e + d * 0.5
    fire = U >= 1.0
    dfire, dsil = sync & (U - d >= 1.0), sync & (U + d < 1.0)
    dec = dfire | dsil
    bad = dec & (spk[t].astype(bool) != fire)
    assert not bad.any(), (label, t, "decided spikes differ from float64", int(bad.sum()))
    undecided += int((~dec).sum())
    sync &= dec
    d = np.where(dfire, 0.0, d)
    u = np.where(fire, 0.0, U)
  err = np.abs(u32.astype(np.float64) - u)
  assert not (sync & (err > d)).any(), (label, "synchronised membranes outside delta_T")
  return undecided / ex.size


def sigmoid_att(rng, shape):
  """TCJA-like attention: a sigmoid of a wide logit, most values near 1, some exactly 1.0 in fp32."""
  z = rng.normal(3.0, 3.0, size=shape)
  z[..., :4] = 20.0
  return (1.0 / (1.0 + np.exp(-z))).astype(F32)


def test_band_on_emulated_attention_path(oracle_lib):
  """T = 20 at production-like data: conv5 (8 x 8, 128 channels) and dense1 (K = 2048, N = 512) fed by spikes at 30 /
  15 % density and sigmoid-shaped att.  Reports the undecided fraction of each path."""
  rng = np.random.default_rng(11)
  T = 20
  _, q, _, _, scale, bias = conv_layer(12)
  x = (rng.uniform(size=(T, 4, 8, 8, 128)) < 0.3).astype(np.uint8)
  att = sigmoid_att(rng, (T, 4, 128))
  assert (att == 1.0).any()
  ex, A, fix = _f64_truth(x, att, q)
  tc, S = ar.conv_att_tc_acc(x, att, q, want=True)
  f64err = 1152 * 2.0 ** -53 * A
  res = {"conv5 tcgen05": att_band(ex, ar.tc_acc_bound(fix, S) + f64err, scale, bias, tc, "conv5 tcgen05"),
         "conv5 simt": att_band(ex, ar.gamma(1152) * A + f64err, scale, bias, ar.conv_att_simt_acc(x, att, q),
                                "conv5 simt")}
  _, qd, sd, bd = dense_layer(13)
  xd = (rng.uniform(size=(T, 16, 2048)) < 0.15).astype(np.uint8)
  attd = np.tile(sigmoid_att(rng, (T, 16, 128)), (1, 1, 16))
  ex, A, fix = _f64_truth(xd, attd, qd, dense=True)
  tc, S = ar.dense_att_tc_acc(xd, attd, qd, want=True)
  f64err = 2048 * 2.0 ** -53 * A
  res["dense1 tcgen05"] = att_band(ex, ar.tc_acc_bound(fix, S) + f64err, sd, bd, tc, "dense1 tcgen05")
  res["dense1 simt"] = att_band(ex, ar.gamma(2048) * A + f64err, sd, bd, ar.dense_att_simt_acc(xd, attd, qd),
                                "dense1 simt")
  print("undecided fraction of the neuron-steps: " + ", ".join(f"{k} {v:.2e}" for k, v in res.items()))
  # the SIMT bound is the a-priori gamma_n sum |att x q|, far above the chain's typical error: a wider band
  assert res["conv5 tcgen05"] < 1e-3 and res["dense1 tcgen05"] < 1e-3
  assert res["conv5 simt"] < 0.05 and res["dense1 simt"] < 0.05


# ================================================================================= GPU: conv5 and dense1 ====
def launch_conv(lib, x, att_d, packed, impl, *, pool, tau=2.0, batch_major=True, dumps=True, v_th=1.0, v_reset=0.0):
  """snnqp_spiking_conv3x3_counts_fwd on x (T, B, H, 8, 128) u8 (device copy batch-major or time-major) with att_d a
  device view (T, B, 128) of any strides.  Returns spikes (T, B, Ho, Wo, C), and with dumps u_T, acc, counts."""
  T, B, H, W, C = x.shape
  if batch_major:
    xs = dev(np.swapaxes(x, 0, 1))
    xst, xsb = xs.stride(1), xs.stride(0)
  else:
    xs = dev(x)
    xst, xsb = xs.stride(0), xs.stride(1)
  Ho, Wo = (H // 2, W // 2) if pool else (H, W)
  spikes = torch.full((T, B, Ho, Wo, C), 7, device=DEV, dtype=torch.uint8)
  u = torch.full((B, H, W, C), np.nan, device=DEV) if dumps else None
  acc = torch.full((T, B, H, W, C), np.nan, device=DEV) if dumps else None
  cnt = torch.zeros((B, T, C), device=DEV, dtype=torch.int32) if dumps else None
  p = BlockParams()
  p.T, p.B, p.H, p.W, p.Cin, p.Cout = T, B, H, W, C, C
  p.x_stride_t, p.x_stride_b = xst, xsb
  p.y_stride_t, p.y_stride_b = spikes.stride(0), spikes.stride(1)
  p.att_stride_t, p.att_stride_b = att_d.stride(0), att_d.stride(1)
  p.att_mod = C
  p.tau, p.v_threshold, p.v_reset = tau, v_th, v_reset
  p.pool, p.impl = int(pool), impl
  _lib.check(lib.snnqp_spiking_conv3x3_counts_fwd(p, P(xs), P(att_d), P(packed.wq), P(packed.scale), P(packed.bias),
                                                  P(spikes), P(u), P(acc), P(cnt), _lib.stream()))
  torch.cuda.synchronize()
  out = [spikes.cpu().numpy()]
  if dumps:
    out += [u.cpu().numpy(), acc.cpu().numpy(), cnt.cpu().numpy()]
  return out


def att_device(att, layout, pad):
  """att (T, B, C) fp32 -> a device view (T, B, C) stored batch-major [B][T][C + pad] or time-major [T][B][C + pad]."""
  T, B, C = att.shape
  if layout == "bt":
    buf = torch.zeros((B, T, C + pad), device=DEV)
    buf[:, :, :C] = dev(np.swapaxes(att, 0, 1))
    return buf[:, :, :C].transpose(0, 1)
  buf = torch.zeros((T, B, C + pad), device=DEV)
  buf[:, :, :C] = dev(att)
  return buf[:, :, :C]


def first_diff(name, got, want):
  if np.array_equal(got, want):
    return ""
  d = np.argwhere(got != want)
  return f"{name}: {len(d)} elements differ, first {d[:4].tolist()}"


def check_conv(lib, x, att, q, packed, scale, bias, impl, *, tau=2.0, layout="bt", pad=0, batch_major=True, v_th=1.0,
               v_reset=0.0):
  """Un-pooled launch with every dump against the emulation, then the pooled production variant (no dumps)."""
  emu = ar.conv_att_tc_acc(x, att, q) if impl == _lib.IMPL_TCGEN05 else ar.conv_att_simt_acc(x, att, q)
  s_e, u_e = ref_int.lif_from_acc(emu, scale, bias, tau, v_th, v_reset)
  att_d = att_device(att, layout, pad)
  lif = dict(tau=tau, v_th=v_th, v_reset=v_reset)
  s, u, acc, cnt = launch_conv(lib, x, att_d, packed, impl, pool=False, batch_major=batch_major, **lif)
  msgs = [first_diff("acc", acc, emu), first_diff("spikes", s, s_e), first_diff("u_final", u, u_e),
          first_diff("spike_counts", cnt, s_e.sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2))]
  (sp,) = launch_conv(lib, x, att_d, packed, impl, pool=True, batch_major=batch_major, dumps=False, **lif)
  msgs.append(first_diff("pooled production spikes", sp, ref_int.maxpool2_u8(s_e)))
  msgs = [m for m in msgs if m]
  assert not msgs, msgs
  assert s_e.any() and not s_e.all()
  return s_e


CONV_TC_CASES = {
    # name: (T, B, H, layout, att pad, tau, slabs kept, edge att)
    "T1_B300_H16": (1, 300, 16, "bt", 0, 2.0, None, False),
    "T5_B300_H8_edges": (5, 300, 8, "bt", 0, 2.0, None, True),
    "T5_B301_H8_tb_pad": (5, 301, 8, "tb", 4, 2.0, None, False),
    "T5_B150_H16_sparse": (5, 150, 16, "bt", 3, 2.0, 20, True),
    "T20_B24_H8_tau3": (20, 24, 8, "tb", 0, 3.0, None, True),
    "T20_B12_H16_sparse": (20, 12, 16, "bt", 1, 2.0, 9, False),
}


@gpu
@pytest.mark.parametrize("case", list(CONV_TC_CASES))
def test_conv_att_tcgen05_bit_exact(cuda_lib, oracle_lib, case):
  """k_conv_att_umma equals the byte-plane emulation exactly: fp32 accumulators, un-pooled spikes, u_T, spike_counts,
  and the pooled spikes of the production variant.  B = 300 gives two or three items per CTA at T <= 5; H = 16 two
  strips per image; att batch-major or time-major, padded rows; tau = 3 takes lif_step; block-sparse slab masks."""
  T, B, H, layout, pad, tau, keep, edges = CONV_TC_CASES[case]
  rng = np.random.default_rng(40 + list(CONV_TC_CASES).index(case))
  lay, q, bn, stt, scale, bias = conv_layer(T * 1000 + B, mask_keep=keep)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  x = (rng.uniform(size=(T, B, H, 8, 128)) < 0.3).astype(np.uint8)
  att = edge_att(rng, T, B) if edges else rng.uniform(0.0, 1.0, size=(T, B, 128)).astype(F32)
  check_conv(cuda_lib, x, att, q, packed, scale, bias, _lib.IMPL_TCGEN05, tau=tau, layout=layout, pad=pad,
             batch_major=(layout == "bt"))


@gpu
@pytest.mark.parametrize("T,B,H,layout,pad,tau", [(3, 2, 8, "bt", 0, 2.0), (2, 3, 16, "tb", 4, 3.0), (1, 1, 8, "bt", 1, 2.0)])
def test_conv_att_simt_bit_exact(cuda_lib, oracle_lib, T, B, H, layout, pad, tau):
  """k_conv3x3_simt<true> equals the sequential fma chain (kh, kw, channel ascending) exactly."""
  rng = np.random.default_rng(T * 100 + B)
  lay, q, bn, stt, scale, bias = conv_layer(T + 50)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  x = (rng.uniform(size=(T, B, H, 8, 128)) < 0.3).astype(np.uint8)
  check_conv(cuda_lib, x, edge_att(rng, T, B), q, packed, scale, bias, _lib.IMPL_SIMT, tau=tau, layout=layout, pad=pad)


def launch_dense(lib, x, att_d, packed, N, impl, dumps=True, tau=2.0, v_th=1.0, v_reset=0.0):
  """snnqp_spiking_dense_fwd, x (T, B, K) u8 batch-major on the device, att_d a (T, B, 128) device view."""
  T, B, K = x.shape
  xs = dev(np.swapaxes(x, 0, 1))
  spikes = torch.full((T, B, N), 7, device=DEV, dtype=torch.uint8)
  u = torch.full((B, N), np.nan, device=DEV) if dumps else None
  acc = torch.full((T, B, N), np.nan, device=DEV) if dumps else None
  p = BlockParams()
  p.T, p.B, p.H, p.W, p.Cin, p.Cout = T, B, 1, 1, K, N
  p.x_stride_t, p.x_stride_b = K, T * K                 # rows (b, t) contiguous (torch keeps any stride of a size-1 T)
  p.y_stride_t, p.y_stride_b = spikes.stride(0), spikes.stride(1)
  p.att_stride_t, p.att_stride_b = att_d.stride(0), att_d.stride(1)
  p.att_mod = 128
  p.tau, p.v_threshold, p.v_reset = tau, v_th, v_reset
  p.impl = impl
  _lib.check(lib.snnqp_spiking_dense_fwd(p, P(xs), P(att_d), P(packed.wq), P(packed.scale), P(packed.bias), P(spikes),
                                         P(u), P(acc), _lib.stream()))
  torch.cuda.synchronize()
  return [spikes.cpu().numpy()] + ([u.cpu().numpy(), acc.cpu().numpy()] if dumps else [])


def check_dense(lib, x, att, q, packed, scale, bias, impl, emu_impl=None, pad=0, layout="bt", tau=2.0, v_th=1.0,
                v_reset=0.0):
  emu_impl = impl if emu_impl is None else emu_impl
  K, N = q.shape
  att_k = np.tile(att, (1, 1, K // 128))
  emu = ar.dense_att_tc_acc(x, att_k, q) if emu_impl == _lib.IMPL_TCGEN05 else ar.dense_att_simt_acc(x, att_k, q)
  s_e, u_e = ref_int.lif_from_acc(emu, scale, bias, tau, v_th, v_reset)
  att_d = att_device(att, layout, pad)
  lif = dict(tau=tau, v_th=v_th, v_reset=v_reset)
  s, u, acc = launch_dense(lib, x, att_d, packed, N, impl, **lif)
  (sp,) = launch_dense(lib, x, att_d, packed, N, impl, dumps=False, **lif)
  msgs = [first_diff("acc", acc, emu), first_diff("spikes", s, s_e), first_diff("u_final", u, u_e),
          first_diff("production spikes", sp, s_e)]
  msgs = [m for m in msgs if m]
  assert not msgs, msgs
  assert s_e.any() and not s_e.all()


@gpu
@pytest.mark.parametrize("T,B", [(1, 323), (3, 101), (5, 4800), (16, 23), (20, 17), (32, 9)])
def test_dense_att_tcgen05_bit_exact(cuda_lib, oracle_lib, T, B):
  """k_dense_umma<3> (K = 2048, N = 512, att_mod = 128) equals the emulation exactly at every dense_tile split: NB
  samples of T steps per column tile (T = 1: 160 x 1, 3: 48 x 3, 5: 32 x 5, 16: 10 x 16, 20: 8 x 20, 32: 4 x 32),
  ragged last tiles; T = 5, B = 4800 gives 150 column tiles (600 items) -- more than the SMs."""
  rng = np.random.default_rng(T)
  lay, q, scale, bias = dense_layer(200 + T)
  packed = pk_mod.pack_dense(lay, 8, DEV)
  x = (rng.uniform(size=(T, B, 2048)) < 0.15).astype(np.uint8)
  att = edge_att(rng, T, B) if B < 1000 else rng.uniform(0.0, 1.0, size=(T, B, 128)).astype(F32)
  check_dense(cuda_lib, x, att, q, packed, scale, bias, _lib.IMPL_TCGEN05, layout="bt" if T % 2 else "tb")


@gpu
def test_dense_att_simt_and_unaligned_att_fallback(cuda_lib, oracle_lib):
  """k_dense_simt<true> equals the sequential fma chain (k ascending).  An att row stride that is not a multiple of 4
  cannot be read as float4: IMPL_AUTO must run SIMT, and the result is the SIMT emulation's."""
  rng = np.random.default_rng(17)
  lay, q, scale, bias = dense_layer(18)
  packed = pk_mod.pack_dense(lay, 8, DEV)
  x = (rng.uniform(size=(3, 6, 2048)) < 0.15).astype(np.uint8)
  att = edge_att(rng, 3, 6)
  check_dense(cuda_lib, x, att, q, packed, scale, bias, _lib.IMPL_SIMT)
  check_dense(cuda_lib, x, att, q, packed, scale, bias, _lib.IMPL_AUTO, emu_impl=_lib.IMPL_SIMT, pad=2)
  check_dense(cuda_lib, x, att, q, packed, scale, bias, _lib.IMPL_AUTO, emu_impl=_lib.IMPL_TCGEN05, pad=4)


@gpu
@pytest.mark.parametrize("sign", [1, -1])
def test_att_extreme_sums(cuda_lib, oracle_lib, sign):
  """All spikes on, att ~ 1, every level +127 or -127: |S_2| > 2^24 (conv ~3.7e7, dense ~6.6e7), so the int -> float
  conversions and the combine's fmas round.  Both implementations of conv5 and dense1 equal their emulations."""
  rng = np.random.default_rng(5 + sign)
  att = (1.0 - rng.integers(0, 4, size=(2, 3, 128)) * 2.0 ** -24).astype(F32)
  att[0, 0, :8] = 1.0
  lay, q, bn, stt, scale, bias = conv_layer(90 + sign, const_q=sign)
  assert (np.abs(q) == 127).all()
  # bias chosen so that the threshold falls between the image's interior (9 taps) and its border (4 or 6 taps)
  full = ar.conv_att_tc_acc(np.ones((1, 1, 8, 8, 128), np.uint8), att[:1, :1], q)
  bias = (1.5 - scale.astype(np.float64) * full.mean(axis=(0, 1, 2, 3))).astype(F32)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  packed.bias.copy_(dev(bias))
  x = np.ones((2, 3, 8, 8, 128), np.uint8)
  x[1, 1, 3] = 0
  _, S = ar.conv_att_tc_acc(x, att, q, want=True)
  assert (np.abs(S[0]) > 2 ** 24).any()
  for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
    check_conv(cuda_lib, x, att, q, packed, scale, bias, impl)
  lay, q, scale, bias = dense_layer(95 + sign, const_q=sign)
  xd = np.ones((2, 3, 2048), np.uint8)
  xd[1, 2, ::3] = 0
  # a full row gives v = 2.5 (fires) for +127 and v = 0.5 (silent) for -127; the row missing a third of its inputs
  # the other way round
  full = ar.dense_att_tc_acc(np.ones((1, 1, 2048), np.uint8), np.tile(att[:1, :1], (1, 1, 16)), q)[0, 0]
  bias = ((2.5 if sign > 0 else 0.5) - scale.astype(np.float64) * full).astype(F32)
  packed = pk_mod.pack_dense(lay, 8, DEV)
  packed.bias.copy_(dev(bias))
  for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
    check_dense(cuda_lib, xd, att, q, packed, scale, bias, impl)


@gpu
def test_nonbinary_x_is_a_spike(cuda_lib, oracle_lib):
  """With att, an x byte of 2 or 255 counts as a spike, exactly like 1, on both implementations (the tcgen05 byte
  planes cannot carry a count): outputs for x in {0, 1, 2, 255} equal those for x != 0."""
  rng = np.random.default_rng(23)
  lay, q, bn, stt, scale, bias = conv_layer(24)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  x = rng.choice(np.array([0, 0, 0, 0, 1, 2, 255], np.uint8), size=(3, 4, 8, 8, 128))
  att = rng.uniform(0, 1, size=(3, 4, 128)).astype(F32)
  att_d = att_device(att, "bt", 0)
  xb = (x != 0).astype(np.uint8)
  for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
    for pool in (False, True):
      got = launch_conv(cuda_lib, x, att_d, packed, impl, pool=pool)
      want = launch_conv(cuda_lib, xb, att_d, packed, impl, pool=pool)
      for g, w in zip(got, want):
        assert np.array_equal(g, w, equal_nan=True), (impl, pool)
  lay, q, scale, bias = dense_layer(25)
  packed = pk_mod.pack_dense(lay, 8, DEV)
  x = rng.choice(np.array([0, 0, 0, 0, 0, 1, 2, 255], np.uint8), size=(3, 5, 2048))
  att_d = att_device(rng.uniform(0, 1, size=(3, 5, 128)).astype(F32), "bt", 0)
  for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
    got = launch_dense(cuda_lib, x, att_d, packed, 512, impl)
    want = launch_dense(cuda_lib, (x != 0).astype(np.uint8), att_d, packed, 512, impl)
    for g, w in zip(got, want):
      assert np.array_equal(g, w, equal_nan=True), impl


# ======================================================================================== GPU: the TCJA kernels ====
TCJA_T = (1, 2, 16, 17, 20, 32)
TCJA_HW = {64: (8, 8), 255: (15, 17), 256: (16, 16), 1024: (32, 32)}


def tcja_case(T, HW, big=False, seed=0):
  """Counts (B = 3, C = 128) with some channels fully active (count = HW, so the high byte plane is used at HW >= 256),
  weights clustered at +-127, and scales that put pr = co * to around +-10 (big: around +-1e4, so att is exactly 0
  and exactly 1).  Returns cnt (B, T, C) int32, q_t (4, T, T), q_c (4, C, C) int8, st, sc."""
  rng = np.random.default_rng(seed + 7 * T + HW)
  B, C = 3, 128
  cnt = rng.integers(0, HW + 1, size=(B, T, C)).astype(np.int32)
  cnt[:, :, rng.permutation(C)[:24]] = HW
  cnt[1] = HW                                             # one fully active sample
  cnt[2, :, :16] = 0
  q_t = rng.integers(-127, 128, size=(4, T, T)).astype(np.int8)
  q_c = np.where(rng.uniform(size=(4, C, C)) < 0.6, rng.choice([-127, -126, 126, 127], size=(4, C, C)),
                 rng.integers(-127, 128, size=(4, C, C))).astype(np.int8)
  q_c[:, :, :8] = 127                                     # |acc_c| of a fully active sample passes 2^24 at H W = 1024
  q_c[:, :, 8:16] = -127
  acc_t, acc_c = ar.tcja_acc(cnt, q_t, q_c)
  k = 1e2 if big else 3.0
  st = F32(k / max(1.0, float(np.abs(acc_t).max())) * 4)
  sc = F32(k / max(1.0, float(np.std(acc_c))))
  return cnt, q_t, q_c, st, sc


def spikes_for_counts(rng, cnt, H, W):
  """Un-pooled spikes (T, B, H, W, C) whose per-(b, t, c) count over (h, w) is cnt (B, T, C)."""
  B, T, C = cnt.shape
  r = rng.uniform(size=(T, B, H * W, C)).argsort(axis=2)
  s = (r < np.transpose(cnt, (1, 0, 2))[:, :, None, :]).astype(np.uint8)
  return s.reshape(T, B, H, W, C)


def run_tcja(lib, T, HW, big, route, seed=0):
  """route: "counts" (spikes == NULL, counts given), "spikes" (k_tcja_counts from batch-major spikes with a padded
  sample stride), either with "+misaligned" (counts pointer offset by 4 bytes: the scalar kernel k_tcja_att).
  Returns (att (T, B, C), counts (B, T, C))."""
  H, W = TCJA_HW[HW]
  cnt, q_t, q_c, st, sc = tcja_case(T, HW, big, seed)
  B, C = 3, 128
  buf = torch.zeros(B * T * C + 4, device=DEV, dtype=torch.int32)
  off = 1 if route.endswith("+misaligned") else 0
  cnt_d = buf[off:off + B * T * C]
  sd = None
  p = BlockParams()
  p.T, p.B, p.H, p.W, p.Cin, p.Cout = T, B, H, W, C, C
  if route.startswith("spikes"):
    s = spikes_for_counts(np.random.default_rng(seed), cnt, H, W)
    sbuf = torch.zeros((B, T * H * W * C + 64), device=DEV, dtype=torch.uint8)
    sbuf[:, :T * H * W * C] = dev(np.swapaxes(s, 0, 1).reshape(B, -1))
    sd = sbuf
    p.x_stride_t, p.x_stride_b = H * W * C, sbuf.stride(0)
  else:
    cnt_d.copy_(dev(cnt).reshape(-1))
  attb = torch.full((T, B, C + 4), np.nan, device=DEV)
  att = attb[:, :, :C]
  p.att_stride_t, p.att_stride_b = att.stride(0), att.stride(1)
  qt, qc = dev(q_t), dev(q_c)
  std, scd = dev(np.array([st], F32)), dev(np.array([sc], F32))
  _lib.check(lib.snnqp_tcja_fwd(p, P(sd), P(qt), P(qc), P(std), P(scd), P(cnt_d), P(att), _lib.stream()))
  torch.cuda.synchronize()
  return att.cpu().numpy(), cnt_d.cpu().numpy().reshape(B, T, C)


def tcja_routes():
  out = []
  for T in TCJA_T:
    for HW in TCJA_HW:
      out.append((T, HW, False, "counts"))
      out.append((T, HW, True, "counts"))
  for T, HW in ((2, 64), (17, 256), (32, 1024), (1, 255)):
    out.append((T, HW, False, "spikes"))
  return out


def check_tcja(results, label):
  """results: {(T, HW, big, route): (att, cnt)} -> the largest expf ulp offset needed."""
  worst = 0
  saw0 = saw1 = False
  for (T, HW, big, route), (att, cnt) in results.items():
    cnt_ref, q_t, q_c, st, sc = tcja_case(T, HW, big)
    assert np.array_equal(cnt, cnt_ref), (label, T, HW, route, "counts")
    assert cnt_ref.max() == HW
    acc_t, acc_c = ar.tcja_acc(cnt_ref, q_t, q_c)
    cands, pr = ar.tcja_candidates(acc_t, acc_c, st, sc)
    worst = max(worst, ar.tcja_check(att, cands, (label, T, HW, big, route)))
    if big:
      saw0 |= bool((att == 0).any())
      saw1 |= bool((att == 1).any())
      assert (np.abs(acc_c) > 2 ** 24).any() or HW < 1024 or T == 1
  assert saw0 and saw1, label
  return worst


@gpu
def test_tcja_mma_and_scalar_kernels_candidate_set(cuda_lib, oracle_lib):
  """k_tcja_att_mma (the default) and the scalar k_tcja_att (counts pointer not 16-byte aligned) at T in {1, 2, 16,
  17, 20, 32} (T > 16: the mma kernel's second time tile) and H W in {64, 255, 256, 1024} with fully active channels
  (counts 256 / 1024 use the high count plane): counts exact, att within the expf candidate set."""
  worst = {}
  for misaligned, name in ((False, "k_tcja_att_mma"), (True, "k_tcja_att")):
    res = {}
    for T, HW, big, route in tcja_routes():
      r = route + ("+misaligned" if misaligned else "")
      res[(T, HW, big, route)] = run_tcja(cuda_lib, T, HW, big, r)
    worst[name] = check_tcja(res, name)
  print("largest expf ulp offset needed: " + ", ".join(f"{k} {v}" for k, v in worst.items()))


def _dp4a_worker(path):
  os.environ["SNNQP_TCJA_IMPL"] = "1"                   # read once per process, at the first TCJA launch
  lib = _lib.lib()
  out = {}
  for i, (T, HW, big, route) in enumerate(tcja_routes()):
    att, cnt = run_tcja(lib, T, HW, big, route)
    out[f"att{i}"], out[f"cnt{i}"] = att, cnt
  np.savez(path, **out)


@gpu
def test_tcja_dp4a_kernel_candidate_set(cuda_lib, oracle_lib, tmp_path):
  """k_tcja_att_dp4a (SNNQP_TCJA_IMPL=1, chosen once per process, so run in a child process): the HIGH == false
  instance at H W <= 255 and HIGH == true above, same shapes and checks as the other two kernels."""
  path = str(tmp_path / "dp4a.npz")
  p = multiprocessing.get_context("spawn").Process(target=_dp4a_worker, args=(path,))
  p.start()
  p.join(600)
  assert p.exitcode == 0
  z = np.load(path)
  res = {k: (z[f"att{i}"], z[f"cnt{i}"]) for i, k in enumerate(tcja_routes())}
  print(f"largest expf ulp offset needed: k_tcja_att_dp4a {check_tcja(res, 'k_tcja_att_dp4a')}")
