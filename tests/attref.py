"""Emulation of the attention path's arithmetic (conv5, dense1, TCJA): what each kernel computes, step by step, in numpy.

The tcgen05 kernels (umma_att.cu) take att as 24-bit fixed point (ptx::att_fix24: round to nearest even of att * 2^24,
clamped to 0xFFFFFF), contract the three byte planes exactly on the tensor core and recombine them in fp32
(ptx::att_combine).  The SIMT kernels (simt.cu) run one sequential fp32 fma chain per output.  TCJA's integer
accumulators are exact; its only inexact step is the device expf.  Every function here reproduces one of these bit for
bit (or, for expf, as the set of results its documented error allows), so a GPU test can compare the kernels exactly.

The exact integer sums are taken in float64 matrix products: every sum here is an integer below 2^43, so float64 holds
it exactly whatever the summation order."""
import numpy as np

from oracle import ref_int

F32 = np.float32
EPS = 2.0 ** -24          # unit roundoff of fp32 (round to nearest)
FIX_MAX = 0xFFFFFF


# ------------------------------------------------------------------------------------------------ fixed point ----
def att_fix24(att):
  """ptx::att_fix24: round(att * 2^24) half to even (att * 2^24 is exact), clamped to 0xFFFFFF.  int64."""
  f = np.rint(np.asarray(att, F32).astype(np.float64) * 2.0 ** 24)
  return np.minimum(f, FIX_MAX).astype(np.int64)


def att_bytes(att):
  """The three byte planes (b2, b1, b0) of att_fix24(att), most significant first (the operand plane order)."""
  f = att_fix24(att)
  return (f >> 16) & 255, (f >> 8) & 255, f & 255


def combine(s2, s1, s0):
  """ptx::att_combine: f1 = fma((float)a1, 256, (float)a0), f = fma((float)a2, 65536, f1), f * 2^-24.  The float64
  sums are exact (integers < 2^53), so each astype(F32) is the fma's single rounding."""
  a2, a1, a0 = (np.asarray(s, np.int64).astype(F32).astype(np.float64) for s in (s2, s1, s0))
  f1 = (a1 * 256.0 + a0).astype(F32).astype(np.float64)
  f = (a2 * 65536.0 + f1).astype(F32)
  return (f * F32(2.0 ** -24)).astype(F32)


def fix_bound(att):
  """Bound of |att - att_fix24(att) 2^-24|: 2^-25 (round to nearest), or 2^-24 where the clamp bites (att = 1.0)."""
  a = np.asarray(att, F32).astype(np.float64)
  return np.where(np.rint(a * 2.0 ** 24) > FIX_MAX, 2.0 ** -24, 2.0 ** -25)


# ------------------------------------------------------------------------------------- exact float64 contractions ----
def conv_f64(planes, q):
  """planes (..., H, W, Cin) float64 (any leading axes), q (3, 3, Cin, Cout) -> (..., H, W, Cout) float64, 3x3 SAME
  conv with zero padding, as ref_int.conv3x3_acc.  Exact while every partial sum is an integer below 2^53."""
  lead, (H, W, Cin) = planes.shape[:-3], planes.shape[-3:]
  x = planes.reshape((-1, H, W, Cin))
  xp = np.zeros((x.shape[0], H + 2, W + 2, Cin))
  xp[:, 1:-1, 1:-1] = x
  qf = np.asarray(q).astype(np.float64)
  out = np.zeros((x.shape[0] * H * W, qf.shape[-1]))
  for kh in range(3):
    for kw in range(3):
      out += xp[:, kh:kh + H, kw:kw + W].reshape(-1, Cin) @ qf[kh, kw]
  return out.reshape(lead + (H, W, qf.shape[-1]))


def dense_f64(planes, q):
  """planes (..., K) float64, q (K, N) -> (..., N) float64."""
  return planes @ np.asarray(q).astype(np.float64)


# --------------------------------------------------------------------------------------- tcgen05: byte planes ----
def conv_att_tc_acc(x, att, q, want=False):
  """k_conv_att_umma's fp32 accumulators.  x (T, B, H, W, C) u8 (any non-zero byte is a spike), att (T, B, C) fp32,
  q (3, 3, C, Cout) int8.  With want: also the plane sums S (3, T, B, H, W, Cout) int64."""
  m = (np.asarray(x) != 0).astype(np.float64)
  planes = np.stack([m * b[:, :, None, None, :].astype(np.float64) for b in att_bytes(att)])
  S = conv_f64(planes, q).astype(np.int64)
  acc = combine(S[0], S[1], S[2])
  return (acc, S) if want else acc


def dense_att_tc_acc(x, att_k, q, want=False):
  """k_dense_umma<3>'s fp32 accumulators.  x (T, B, K) u8, att_k (T, B, K) fp32 (att[t, b, k % att_mod]), q (K, N)."""
  x, att_k = np.asarray(x), np.asarray(att_k, F32)
  S = np.empty((3,) + x.shape[:-1] + (np.shape(q)[1],), np.int64)
  for b0 in range(0, x.shape[1], 512):                   # bounded float64 working set at large B
    m = (x[:, b0:b0 + 512] != 0).astype(np.float64)
    planes = np.stack([m * b.astype(np.float64) for b in att_bytes(att_k[:, b0:b0 + 512])])
    S[:, :, b0:b0 + 512] = dense_f64(planes, q).astype(np.int64)
  acc = combine(S[0], S[1], S[2])
  return (acc, S) if want else acc


def tc_acc_bound(fix_term, S):
  """Bound of |tcgen05 accumulator - exact sum att x q|, given fix_term = sum over the spiking inputs of
  |q| fix_bound(att) (the fixed-point term) and the plane sums S: each of the three int -> float conversions and
  the two fmas rounds once, at most EPS times a value bounded by M = 2^-24 (2^16 |S2| + 2^8 |S1| + |S0|) (1 + 2^-20),
  and the final * 2^-24 is exact."""
  M = 2.0 ** -24 * (65536.0 * np.abs(S[0]) + 256.0 * np.abs(S[1]) + np.abs(S[2]))
  return fix_term + 5.0 * EPS * M * (1.0 + 2.0 ** -20)


# ----------------------------------------------------------------------------------------- SIMT: the fma chain ----
def conv_att_simt_acc(x, att, q):
  """k_conv3x3_simt<true>'s fp32 accumulators: acc = fmaf(x != 0 ? att : 0, q, acc) in the order kh, kw, channel
  ascending.  A zero-padding term leaves acc unchanged (acc never holds -0), which is the kernel's skip."""
  T, B, H, W, C = x.shape
  xs = np.where(np.asarray(x) != 0, np.asarray(att, F32)[:, :, None, None, :], F32(0)).astype(F32)
  xp = np.zeros((T * B, H + 2, W + 2, C), F32)
  xp[:, 1:-1, 1:-1] = xs.reshape(T * B, H, W, C)
  qf = np.asarray(q).astype(F32)
  acc = np.zeros((T * B, H, W, qf.shape[-1]), F32)
  for kh in range(3):
    for kw in range(3):
      win = xp[:, kh:kh + H, kw:kw + W]
      for c in range(C):
        acc = ref_int.fmaf(win[..., c:c + 1], qf[kh, kw, c], acc)
  return acc.reshape(T, B, H, W, -1)


def dense_att_simt_acc(x, att_k, q):
  """k_dense_simt<true>'s fp32 accumulators: acc = fmaf(x != 0 ? att_k : 0, q, acc), k ascending."""
  xs = np.where(np.asarray(x) != 0, np.asarray(att_k, F32), F32(0)).astype(F32)
  qf = np.asarray(q).astype(F32)
  acc = np.zeros(xs.shape[:-1] + (qf.shape[1],), F32)
  for k in range(xs.shape[-1]):
    acc = ref_int.fmaf(xs[..., k:k + 1], qf[k], acc)
  return acc


def gamma(n):
  """Bound factor of an n-term sequential fp32 fma chain: |err| <= gamma(n) sum |terms|."""
  return n * EPS / (1.0 - n * EPS)


# ------------------------------------------------------------------------------------------------------- TCJA ----
def tcja_acc(cnt, q_t, q_c):
  """Integer accumulators of TCJA from counts cnt (B, T, C) int32 (k_tcja_counts' layout): acc_t (T, B, C) of the
  conv over the channel axis, acc_c (T, B, C) of the conv over the time axis (ref_int.tcja_att's wiring)."""
  x = np.ascontiguousarray(cnt, dtype=np.int32)
  acc_t = ref_int.conv1d_acc(np.ascontiguousarray(np.transpose(x, (0, 2, 1))), q_t, 1)   # (B, C, T)
  acc_c = ref_int.conv1d_acc(x, q_c, 1)                                                 # (B, T, C)
  return np.transpose(acc_t, (2, 0, 1)), np.transpose(acc_c, (1, 0, 2))


def tcja_candidates(acc_t, acc_c, scale_t, scale_c, ulps=2):
  """Every att the kernels may return: to = fl(fl(acc_t) st), co = fl(fl(acc_c) sc), pr = fl(co to) are exact fp32
  steps; e = expf(-pr) is any fp32 within `ulps` ulp of the correctly rounded exp (CUDA documents <= 2 ulp), up to inf
  on overflow; att = fl(1 / fl(1 + e)).  Returns (cand (2 ulps + 1, ...) fp32 ordered by ulp offset -ulps .. ulps,
  pr)."""
  to = (np.asarray(acc_t).astype(F32) * F32(scale_t)).astype(F32)
  co = (np.asarray(acc_c).astype(F32) * F32(scale_c)).astype(F32)
  pr = (co * to).astype(F32)
  with np.errstate(over="ignore"):
    e0 = np.exp(-pr.astype(np.float64)).astype(F32)            # correctly rounded for all practical purposes
  cands = []
  for k in range(-ulps, ulps + 1):
    e = e0.copy()
    for _ in range(abs(k)):
      e = np.nextafter(e, F32(np.inf) if k > 0 else F32(0)).astype(F32)
    e = np.maximum(e, F32(0))
    with np.errstate(over="ignore"):
      cands.append((F32(1) / (F32(1) + e)).astype(F32))
  return np.stack(cands), pr


def tcja_check(att, cands, label=""):
  """att (T, B, C) must be one of the candidates; returns the largest |ulp offset| of expf needed (the smallest
  offset that explains each value, maximised over the values)."""
  ulps = (cands.shape[0] - 1) // 2
  hit = cands == np.asarray(att, F32)[None]
  ok = hit.any(axis=0)
  assert ok.all(), (label, "att outside the expf candidate set", int((~ok).sum()), np.argwhere(~ok)[:8].tolist())
  off = np.abs(np.arange(-ulps, ulps + 1))[:, None]
  need = np.where(hit.reshape(hit.shape[0], -1), off, ulps + 1).min(axis=0)
  return int(need.max())
