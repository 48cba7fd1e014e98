"""conv1 (Cin = 2, event counts) against a float64 rounding band.

conv1 has no recurrence between neurons: its input is frames, not spikes.  So for every neuron-step a float64
evaluation of the exact LIF (integer accumulator, the folded fp32 scale and bias taken as exact reals) says whether
ANY evaluation whose rounding error stays within a bound derived from the kernel's arithmetic must spike, must not
spike, or may go either way.  Only the last kind may differ from float64, so a correct kernel has zero unexplained
differences -- in LIF_EXACT, LIF_FAST (and lif_mode 101-103) and LIF_TENSOR alike -- and a wrong rounding, a shifted
threshold or a stale carry is a failure, not a budget item.  The bounds are in conv1_band's docstring.

CPU tests check the band against the fp32 reference order (ref_int) and numpy emulations of the single-rounding and
tensor-core arithmetic; gpu tests hold the kernels to it, plus exact threshold ties, dyadic layers on which every mode
is exact, y_popcount and the stride / routing envelope."""
import numpy as np
import pytest
import torch

from oracle import ref_int
from snnquantprune_b200 import _lib, synthetic
from snnquantprune_b200 import pack as pk_mod
from snnquantprune_b200._lib import BlockParams
from test_gpu_parity import DEV, F32, make_layer, run_conv
from test_gpu_persistent_schedules import _edge_layer

gpu = pytest.mark.gpu
EPS = 2.0 ** -24          # unit roundoff of fp32 (round to nearest)
# Accumulation error of LIF_TENSOR's tcgen05.mma chain per step, in units of EPS * M (M = the sum of the magnitudes
# of everything the step adds: see conv1_band).  One step is 5 MMAs (kind::f16, fp32 accumulator).  The rounding mode
# and alignment width of the tensor core's accumulation are not documented, so the bound assumes the worst of what
# fp32 accumulation can do short of dropping bits of the result: every MMA truncates (not rounds) its result to fp32,
# an error below one ulp, 2 * EPS relative, of a partial sum bounded by M -- 5 x 2 = 10.
# test_tensor_accumulation_error_t1 measures the real error directly and holds it to this bound (B200: at most 2.96).
C_ACC = 10.0
MODES = ("exact", "fast", "tensor")


# ----------------------------------------------------------------------------------------------- the band oracle ----
def tensor_domain(scale, bias):
  """LIF_TENSOR's membrane scale dom = 2^(15 - e), e the frexp exponent of max_c max(63.5 |s_c|, 0.5 |b_c|), in the
  kernel's fp32 arithmetic (umma_conv1_tc.cu)."""
  s, b = np.abs(np.asarray(scale, F32)), np.abs(np.asarray(bias, F32))
  mx = max(F32(1e-30), np.max(np.maximum(F32(63.5) * s, F32(0.5) * b)))
  return 2.0 ** (15 - int(np.frexp(np.float32(mx))[1]))


def _f16(x):
  return np.asarray(x, F32).astype(np.float16).astype(np.float64)


def tensor_pieces(scale, bias, dom):
  """What LIF_TENSOR's operands hold, emulated exactly: W' = fl32(q * fl32(s/2 * dom)) as hi + lo fp16 pieces and
  b' = fl32(b/2 * dom) as three fp16 pieces (np.float16 rounds to nearest even and has the subnormals).  Returns
  (w_hi, w_eff (C, 255) float64 for q = -127 .. 127: the hi piece and hi + lo, b_eff (C,),
  rw (C,) = max_q |w_eff - q s dom / 2| / |q|, rb (C,) = |b_eff - b dom / 2|)."""
  s, b = np.asarray(scale, F32), np.asarray(bias, F32)
  sch = (F32(0.5) * s * F32(dom)).astype(F32)
  qv = np.arange(-127, 128, dtype=np.float64)
  p = (qv[None, :].astype(F32) * sch[:, None]).astype(F32)
  hi = _f16(p)
  lo = _f16((p.astype(np.float64) - hi).astype(F32))
  w_eff = hi + lo
  exact = qv[None, :] * (s.astype(np.float64) * 0.5 * dom)[:, None]
  nz = qv != 0
  rw = np.max(np.abs(w_eff - exact)[:, nz] / np.abs(qv[nz])[None, :], axis=1)
  bh = (F32(0.5) * b * F32(dom)).astype(F32)
  p1 = _f16(bh)
  r1 = (bh.astype(np.float64) - p1).astype(F32)
  p2 = _f16(r1)
  p3 = _f16((r1.astype(np.float64) - p2).astype(F32))
  b_eff = p1 + p2 + p3
  return hi, w_eff, b_eff, rw, np.abs(b_eff - b.astype(np.float64) * 0.5 * dom)


def _pool_any(a):
  B, H, W, C = a.shape
  return a.reshape(B, H // 2, 2, W // 2, 2, C).any(axis=(2, 4))


def _pool_all(a):
  B, H, W, C = a.shape
  return a.reshape(B, H // 2, 2, W // 2, 2, C).all(axis=(2, 4))


def conv1_band(x, q, scale, bias, modes=MODES, c_acc=C_ACC, emulate=()):
  """The float64 band of conv1 (pooled, tau 2, threshold 1, reset 0).  x (T, B, H, W, 2) u8, q (3, 3, 2, C) int8.

  Per neuron and step, with acc_t the exact integer accumulator and s = scale, b = bias exact reals:
      h_t = (acc_t s + b) / 2,   U_t = h_t + u_{t-1} / 2,   spike iff U_t >= 1,   u_t = 0 on a spike else U_t.
  float64 is exact enough: acc_t s has at most 20 + 24 = 44 significant bits; the additions round at 2^-53 relative,
  which the band absorbs (the 2^-50 term below).  A_t = sum |q| x (ref_int.conv3x3_acc(x, |q|)) bounds the products.

  Per-step rounding bound e_t of each mode, in membrane (threshold = 1) units, from the kernels' code:
    exact  (reference order, ref_int / LIF_EXACT, k_conv1_umma LIFV 0): v = fma(acc, s, b), d = v - u, un = u + d/2
           round once each:  e_t = EPS (|h_t| + |h_t - u_{t-1}/2| + |U_t|).
    fast   (LIF_FAST, lif_mode 101-103): h = fma(acc, s/2, b/2) and un = fma(u, 0.5, h) round once each:
           e_t = EPS (|h_t| + |U_t|).
    tensor (LIF_TENSOR, k_conv1_tclif), computed in the domain dom (tensor_domain) and divided by it:
           the operand pieces (tensor_pieces) miss the exact weights by at most rw per unit of |q| and the bias by rb,
           and the 5 MMAs accumulate with at most c_acc EPS M, M = A_t |s| dom / 2 + |b'| + |D_{t-1}| / 2:
           e_t = (A_t rw + rb) / dom + c_acc EPS (A_t |s| / 2 + |b| / 2 + |u_{t-1}| / 2).
  Every e_t is multiplied by 1 + 2^-10 (the bounds are taken at the float64 values, not the kernel's) plus 2^-50 (|U_t|
  + 1) for float64 itself.  The compares are exact in every mode (FSET, and sat(x 2^24 + 1 - 2^24) -- exactly 1 at
  the threshold and 0 one ulp below it), the reset is exact.

  Propagation: a synchronised neuron (the kernel's membrane within delta of float64) has delta_t = e_t +
  delta_{t-1} / 2.  Step t is decided fire if U_t - delta_t >= 1, decided silent if U_t + delta_t < 1; a decided fire
  resets both to exactly 0 (delta = 0).  The first undecided step ends the neuron's synchronisation for the rest of
  the sample.  A pooled output is decided if a synchronised neuron of the quad decidedly fires, or all four are
  synchronised and decidedly silent.

  ``emulate``: also run numpy emulations ("fast": the single-rounding chain with ref_int.fmaf; "tensor": the fp16
  pieces accumulated in fp32, round to nearest, three roundings per step).  Computed one step at a time.  Returns a
  dict: "pooled" float64 pooled spikes u8 (T, B, Ho, Wo, C), "ref" the fp32 reference order's pooled spikes (bit-equal
  to ref_int.spiking_conv3x3), "ref_u" its u_T, "u" float64 u_T, "ties" neuron-steps with U_t == 1 exactly, and per
  mode m: "dec_m" decided pooled mask, "delta_m" delta_T, "sync_m" synchronised through T, "excl_m" excluded count;
  per emulation: "emu_m" pooled spikes, "emu_u_m" u_T."""
  T, B, H, W, _ = x.shape
  C = q.shape[-1]
  s32, b32 = np.asarray(scale, F32), np.asarray(bias, F32)
  s, b = s32.astype(np.float64), b32.astype(np.float64)
  qa = np.abs(q.astype(np.int16)).astype(np.int8)
  if "tensor" in modes or "tensor" in emulate:
    dom = tensor_domain(s32, b32)
    w_hi, w_eff, b_eff, rw, rb = tensor_pieces(s32, b32, dom)
  u = np.zeros((B, H, W, C))
  u32 = np.zeros((B, H, W, C), F32)
  st = {m: dict(delta=np.zeros((B, H, W, C)), sync=np.ones((B, H, W, C), bool)) for m in modes}
  out = dict(pooled=np.empty((T, B, H // 2, W // 2, C), np.uint8), ref=np.empty((T, B, H // 2, W // 2, C), np.uint8),
             ties=0)
  for m in modes:
    out["dec_" + m] = np.empty((T, B, H // 2, W // 2, C), bool)
  emu = {}
  if "fast" in emulate:
    emu["fast"] = np.zeros((B, H, W, C), F32)
  if "tensor" in emulate:
    emu["tensor"] = np.zeros((B, H, W, C), F32)
    # the hi / lo pieces of every weight (q -> index q + 127), convolved in float64 (exact: < 2^45 of the finest grain)
    qi = (np.arange(C)[None, None, None, :], q.astype(np.int64) + 127)
    whi, wlo = w_hi[qi], w_eff[qi] - w_hi[qi]
  for m in emulate:
    out["emu_" + m] = np.empty((T, B, H // 2, W // 2, C), np.uint8)
  for t in range(T):
    xt = np.ascontiguousarray(x[t])
    acc = ref_int.conv3x3_acc(xt, q)
    A = ref_int.conv3x3_acc(xt, qa).astype(np.float64)
    h = (acc * s + b) * 0.5
    up = u
    U = h + up * 0.5
    fire = U >= 1.0
    out["ties"] += int(np.count_nonzero(U == 1.0))
    out["pooled"][t] = _pool_any(fire)
    u = np.where(fire, 0.0, U)
    # fp32 reference order (the C oracle's lif_update, restated in numpy: every op IEEE round to nearest)
    v32 = ref_int.fmaf(acc.astype(F32), s32, b32)
    un32 = (u32 + ((v32 - u32) / F32(2.0))).astype(F32)
    f32 = (un32 - F32(1.0)) >= 0
    out["ref"][t] = _pool_any(f32)
    u32 = np.where(f32, F32(0.0), un32)
    for m in modes:
      if m == "exact":
        e = EPS * (np.abs(h) + np.abs(h - up * 0.5) + np.abs(U))
      elif m == "fast":
        e = EPS * (np.abs(h) + np.abs(U))
      else:
        e = (A * rw + rb) / dom + c_acc * EPS * (A * np.abs(s) * 0.5 + np.abs(b) * 0.5 + np.abs(up) * 0.5)
      e = e * (1.0 + 2.0 ** -10) + 2.0 ** -50 * (np.abs(U) + 1.0)
      d = st[m]["delta"] = e + st[m]["delta"] * 0.5
      sync = st[m]["sync"]
      dfire = sync & (U - d >= 1.0)
      dsil = sync & (U + d < 1.0)
      out["dec_" + m][t] = _pool_any(dfire) | _pool_all(dsil)
      sync &= dfire | dsil
      st[m]["delta"] = np.where(dfire, 0.0, d)
    if "fast" in emu:
      hh = ref_int.fmaf(acc.astype(F32), F32(0.5) * s32, F32(0.5) * b32)
      un = ref_int.fmaf(emu["fast"], F32(0.5), hh)
      fe = un >= F32(1.0)
      out["emu_fast"][t] = _pool_any(fe)
      emu["fast"] = np.where(fe, F32(0.0), un)
    if "tensor" in emu:
      Dp = emu["tensor"].astype(np.float64)
      sh = _conv_f64(xt, whi)
      sl = _conv_f64(xt, wlo)
      D = (Dp * 0.5 + sh).astype(F32)
      D = (D.astype(np.float64) + sl).astype(F32)
      D = (D.astype(np.float64) + b_eff).astype(F32)
      fe = D >= F32(dom)
      out["emu_tensor"][t] = _pool_any(fe)
      emu["tensor"] = np.where(fe, F32(0.0), D)
  out["u"], out["ref_u"] = u, u32
  for m in modes:
    out["delta_" + m], out["sync_" + m] = st[m]["delta"], st[m]["sync"]
    out["excl_" + m] = int(out["dec_" + m].size - np.count_nonzero(out["dec_" + m]))
  if "fast" in emu:
    out["emu_u_fast"] = emu["fast"]
  if "tensor" in emu:
    out["emu_u_tensor"] = (emu["tensor"].astype(np.float64) / dom).astype(F32)
  return out


def _conv_f64(x, w):
  """x (B, H, W, 2) u8, w (3, 3, 2, C) float64 -> (B, H, W, C) float64, zero padding (SAME), as ref_int.conv3x3_acc."""
  B, H, W, Cin = x.shape
  xp = np.zeros((B, H + 2, W + 2, Cin))
  xp[:, 1:-1, 1:-1] = x
  out = np.zeros((B, H, W, w.shape[-1]))
  for dy in range(3):
    for dx in range(3):
      out += np.einsum("bhwi,ic->bhwc", xp[:, dy:dy + H, dx:dx + W], w[dy, dx])
  return out


def check_band(band, mode, s, u=None, label=""):
  """Kernel pooled spikes s (T, B, Ho, Wo, C) u8 and (optionally) u_T (B, H, W, C) against the band of ``mode``:
  every decided pooled output equals float64, every synchronised membrane is within delta_T.  Returns the statistics
  the tests report."""
  dec = band["dec_" + mode]
  bad = dec & (s != band["pooled"])
  assert not bad.any(), (label, mode, "decided pooled outputs differ from float64", int(bad.sum()),
                         np.argwhere(bad)[:8].tolist())
  flips = s != band["ref"]
  stats = dict(excluded=band["excl_" + mode] / dec.size, flips_vs_fp32=int(flips.sum()),
               flips_outside_excluded=int((flips & dec).sum()))
  if u is not None:
    sync, delta = band["sync_" + mode], band["delta_" + mode]
    err = np.abs(u.astype(np.float64) - band["u"])
    over = sync & (err > delta)
    assert not over.any(), (label, mode, "synchronised membranes outside delta_T", int(over.sum()),
                            float(err[over].max()), np.argwhere(over)[:8].tolist())
    ratio = np.where(sync & (delta > 0), err / np.where(delta > 0, delta, 1.0), 0.0)
    stats["max_err_over_delta"] = float(ratio.max())
  return stats


# ------------------------------------------------------------------------------------------------ layers / inputs ----
def q_layer(q, bits=8):
  """A layer dict whose DuQ levels are exactly the given int8 q (step a / (2^(bits-1) - 1) = 1)."""
  q = np.asarray(q, np.int8)
  a = F32(2 ** (bits - 1) - 1)
  lay = {"kernel": q.astype(F32), "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)},
         "prune_0": {"mask": np.ones(q.shape, F32)}}
  assert np.array_equal(ref_int.duq_levels_c(lay["kernel"], lay["prune_0"]["mask"], a, bits), q)
  return lay


def random_conv1(seed, bits=8):
  rng = np.random.default_rng(seed)
  lay, q, bn, stt = make_layer(rng, 2, 128, bits, 0.3)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128)
  return rng, lay, q, bn, stt, scale, bias


def frames(rng, shape, lam=0.3):
  x = np.minimum(rng.poisson(lam, size=shape), 255).astype(np.uint8)
  x[0, 0, 0, 0, :] = 255
  x[-1, -1, -1, -1, :] = 200
  return x


def production_conv1():
  """conv1 of the synthetic network the LIF_TENSOR flip rates were measured on, with its frames (T, B, H, W, 2)."""
  v = synthetic.make_variables(bits=8, prune_percentage=0.5, T=20, H=128, seed=1, stable=True)
  P, S = v["params"], v["batch_stats"]
  lay, bn, stt = P["QuantConv_0"], P["BatchNorm_0"], S["BatchNorm_0"]
  q = ref_int.duq_levels_c(lay["kernel"], lay["prune_0"]["mask"], lay["DuQ_0"]["a"][0], 8)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  x = np.ascontiguousarray(np.swapaxes(synthetic.make_frames(5, 20, 128, 128, seed=1, stable=True), 0, 1))
  return lay, bn, stt, q, scale, bias, x


LADDER_BIAS = (2.0, 2.0 - 2.0 ** -22, 1.0, 0.0, -1.0)


def ladder_layer():
  """Zero weights (the frames are zero anyway), every channel's scale 0.1 -- so LIF_TENSOR's domain is fixed by the
  ordinary channels (63.5 * 0.1 > 0.5 * 2: dom = 2^12) -- and biases from LADDER_BIAS by channel mod 5: U_1 = 1 (a
  tie, fires), U_1 = 1 - 2^-23 (silent), U_t = 1 - 2^-t (the ladder), 0 and -1 (silent)."""
  q = np.zeros((3, 3, 2, 128), np.int8)
  q[1, 1, 0, :] = 1                                  # some weights, never met by a count
  scale = np.full(128, 0.1, F32)
  bias = np.array([LADDER_BIAS[c % 5] for c in range(128)], F32)
  assert tensor_domain(scale, bias) == 2.0 ** 12
  return q, scale, bias


# --------------------------------------------------------------------------------------------------- CPU tests ----
@pytest.mark.parametrize("case", ["make_layer", "edges", "outlier_2e16", "outlier_2e20"])
def test_band_contains_reference_order(oracle_lib, case):
  """The band of the reference order contains ref_int's fp32 reference-order LIF: every decided pooled output equals
  it, every synchronised membrane is within delta_T of its u_T; and the numpy fp32 restatement inside conv1_band is
  bit-equal to ref_int.spiking_conv3x3.  The FAST and TENSOR emulations sit inside their bands, the 2^16 / 2^20
  outlier channels included."""
  if case == "make_layer":
    rng, lay, q, bn, stt, scale, bias = random_conv1(17)
  else:
    log2 = {"edges": None, "outlier_2e16": 16, "outlier_2e20": 20}[case]
    rng = np.random.default_rng(5 + (log2 or 0))
    lay, q, bn, stt = _edge_layer(rng, 2, log2)
    scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  x = frames(rng, (6, 2, 8, 128, 2))
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  band = conv1_band(x, q, scale, bias, emulate=("fast", "tensor"))
  assert np.array_equal(band["ref"], s_ref) and np.array_equal(band["ref_u"], info["u"])
  check_band(band, "exact", s_ref, info["u"], case)
  check_band(band, "fast", band["emu_fast"], band["emu_u_fast"], case)
  check_band(band, "tensor", band["emu_tensor"], band["emu_u_tensor"], case)
  assert 0.02 < s_ref.mean() < 0.9
  for m in MODES:
    assert band["excl_" + m] < 1e-2 * s_ref.size, (m, band["excl_" + m])


def test_band_rejects_a_shifted_threshold(oracle_lib):
  """The band is not vacuous: the fp32 reference order with its threshold raised by 2^-16 (or its reset skipped once)
  leaves it."""
  rng, lay, q, bn, stt, scale, bias = random_conv1(23)
  x = frames(rng, (8, 4, 16, 128, 2))
  band = conv1_band(x, q, scale, bias, modes=("exact", "tensor"))
  acc = ref_int.conv3x3_acc(x.reshape(-1, 16, 128, 2), q).reshape(8, 4, 16, 128, 128)
  u = np.zeros(acc.shape[1:], F32)
  sp = []
  for t in range(8):
    un = u + (ref_int.fmaf(acc[t].astype(F32), scale, bias) - u) / F32(2)
    f = un >= F32(1 + 2.0 ** -16)
    sp.append(_pool_any(f))
    u = np.where(f, F32(0), un)
  sp = np.array(sp, np.uint8)
  for m in ("exact", "tensor"):
    with pytest.raises(AssertionError):
      check_band(band, m, sp)


def test_ladder_on_the_fp32_reference(oracle_lib):
  """Bias 1, zero input: U_t = 1 - 2^-t exactly in float64, for t <= 24 also in fp32.  Step 24 (1 - 2^-24, the
  largest fp32 below 1) must not fire; step 25 rounds 1 - 2^-25 to 1.0 (ties to even) and fires, in the reference
  order and in the single-rounding form alike; float64 never fires; the band marks step 25 undecided."""
  q, scale, bias = ladder_layer()
  T = 26
  x = np.zeros((T, 1, 4, 128, 2), np.uint8)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  band = conv1_band(x, q, scale, bias, emulate=("fast", "tensor"))
  ch = 2                                                           # bias 1
  for sp in (s_ref, band["emu_fast"], band["emu_tensor"]):
    col = sp[:, 0, 0, 0, ch]
    assert not col[:24].any() and col[24] == 1 and col[25] == 0, col
  assert not band["pooled"][:, ..., ch].any()
  for m in MODES:
    # the early rungs are decided, step 25 is not (nor is anything after it: the neuron left synchronisation)
    dec = band["dec_" + m][:, 0, 0, 0, ch]
    assert dec[:16].all() and not dec[24:].any(), (m, dec)
  # float64: the tie (bias 2) fires at every step, 1 - 2^-23 (bias 2 - 2^-22) is silent at step 1
  assert band["pooled"][:, 0, 0, 0, 0].all() and band["pooled"][0, 0, 0, 0, 1] == 0
  # ladder membranes after 24 steps: 1 - 2^-24 exactly, in fp32
  x24 = x[:24]
  _, info24 = ref_int.spiking_conv3x3(x24, q, scale, bias, pool=True, want=True)
  assert np.all(info24["u"][..., ch] == F32(1 - 2.0 ** -24))
  assert info24["u"][..., ch].dtype == F32 and F32(1 - 2.0 ** -24) < F32(1)


def test_dyadic_layer_is_exact_in_every_mode(oracle_lib):
  """The dyadic layer of the gpu test is exact in float64, the fp32 reference order and both emulations (see
  dyadic_layer for the arithmetic), and has hundreds of exact threshold ties."""
  q, scale, bias, x = dyadic_layer()
  band = conv1_band(x, q, scale, bias, emulate=("fast", "tensor"))
  assert np.array_equal(band["ref"], band["pooled"]) and np.array_equal(band["ref_u"].astype(np.float64), band["u"])
  for m in ("fast", "tensor"):
    assert np.array_equal(band["emu_" + m], band["pooled"]), m
    assert np.array_equal(band["emu_u_" + m].astype(np.float64), band["u"]), m
  assert band["ties"] >= 300, band["ties"]


def dyadic_layer(T=10, B=2, H=8, W=128, seed=31):
  """Weights q in [-3, 3], counts <= 7 (Poisson 0.3), scales k 2^-6 (k = 1..4) and biases j 2^-6 (j = 96..160, so
  h_1 = U_1 sits on a 2^-7 grid around 1 and about one neuron-step in 64 is an exact tie at t = 1).
  |acc| <= 18 * 3 * 7 = 378, so |acc s + b| < 378 * 4 / 64 + 160 / 64 < 2^5 and |U_t| < 2^5; U_t is a multiple of
  2^-(6 + t), so at T = 10 every value is an integer multiple of 2^-16 below 2^21 of them: exact in fp32 (24 bits),
  whatever the order of the additions, the fma's, the halving, the tensor core's scale-input-d or its alignment.
  LIF_TENSOR's domain: 63.5 * 4/64 < 4 -> dom = 2^13, W' = q k 64 and b' = 64 j are integers below 2^14 (fp16-exact,
  the lo and the further bias pieces are 0)."""
  rng = np.random.default_rng(seed)
  q = rng.integers(-3, 4, size=(3, 3, 2, 128)).astype(np.int8)
  scale = (rng.integers(1, 5, size=128) / 64.0).astype(F32)
  bias = (rng.integers(96, 161, size=128) / 64.0).astype(F32)
  x = np.minimum(rng.poisson(0.3, size=(T, B, H, W, 2)), 7).astype(np.uint8)
  assert tensor_domain(scale, bias) == 2.0 ** 13
  return q, scale, bias, x


# -------------------------------------------------------------------------------------------------- GPU helpers ----
def launch(lib, x, p_shape, wq, scale, bias, *, lif_mode, y_bits, u_final=False, popcount=None, x_strides=None,
           y=None, y_strides=None):
  """snnqp_spiking_conv3x3_fwd for conv1 on device tensors with explicit strides.  x: a uint8 device tensor view whose
  data pointer is element (t = 0, b = 0); x_strides = (stride_t, stride_b) in bytes.  Returns (rc, y, u)."""
  T, B, H, W = p_shape
  if y is None:
    y = torch.full((T, B, H // 2, W // 2, 16 if y_bits else 128), 7, device=DEV, dtype=torch.uint8)
    y_strides = (y.stride(0), y.stride(1))
  u = torch.zeros((B, H, W, 128), device=DEV, dtype=torch.float32) if u_final else None
  p = BlockParams()
  p.T, p.B, p.H, p.W, p.Cin, p.Cout = T, B, H, W, 2, 128
  p.x_stride_t, p.x_stride_b = x_strides
  p.y_stride_t, p.y_stride_b = y_strides
  p.att_mod = 2
  p.tau, p.v_threshold, p.v_reset = 2.0, 1.0, 0.0
  p.pool, p.impl = 1, _lib.IMPL_TCGEN05
  p.x_format, p.y_format, p.lif_mode = 0, int(y_bits), lif_mode
  if popcount is not None:
    p.y_popcount = _lib.ptr(popcount)
  rc = lib.snnqp_spiking_conv3x3_fwd(p, _lib.ptr(x), None, _lib.ptr(wq), _lib.ptr(scale), _lib.ptr(bias), _lib.ptr(y),
                                     _lib.ptr(u), None, _lib.stream())
  torch.cuda.synchronize()
  return rc, y, u


def unbits(y):
  return np.unpackbits(y.cpu().numpy(), axis=-1, bitorder="little")


def packed_q(q, scale, bias):
  packed = pk_mod.pack_conv3x3(q_layer(q), 8, DEV, None, None)
  return packed.wq, torch.as_tensor(np.asarray(scale, F32), device=DEV), torch.as_tensor(np.asarray(bias, F32), device=DEV)


FAST_MODES = (_lib.LIF_FAST, 101, 102, 103)


def _fmt(stats):
  return {k: (round(v, 7) if isinstance(v, float) else v) for k, v in stats.items()}


# --------------------------------------------------------------------------------------------------- GPU tests ----
@gpu
def test_threshold_ladder_and_ties_all_modes(cuda_lib, oracle_lib):
  """Zero frames, T = 26, the LADDER_BIAS channels at every quad position (FSET and FFMA.SAT compares alike).
  EXACT, FAST, 101-103 and TENSOR are bit-exact against the fp32 reference for t <= 24, u_T included where the mode
  exposes it (T = 1: the tie has fired and reset, T = 24: the ladder stands at 1 - 2^-24).  At step 25 the bias-1
  channel sits on 1 - 2^-25: EXACT and FAST round it to 1 and fire (bit-exact vs ref_int); TENSOR may go either way,
  and what it does is reported.  The bias -1 channel meets the same rounding at -(1 - 2^-25)."""
  q, scale, bias = ladder_layer()
  wq, sd, bd = packed_q(q, scale, bias)
  for T in (1, 24, 26):
    x = np.zeros((T, 2, 4, 128, 2), np.uint8)
    s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
    s, u, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps="u", lif_mode=_lib.LIF_EXACT)
    assert np.array_equal(s, s_ref) and np.array_equal(u, info["u"]), ("EXACT", T)
    for lm in (_lib.LIF_EXACT,) + FAST_MODES:
      for yb in (False, True):
        s, _, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps=False, y_bits=yb, lif_mode=lm)
        assert np.array_equal(s, s_ref), (lm, yb, T, np.argwhere(s != s_ref)[:8].tolist())
    tens = {}
    for yb in (False, True):
      s, u, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps="u", y_bits=yb,
                         lif_mode=_lib.LIF_TENSOR)
      s2, _, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps=False, y_bits=yb,
                          lif_mode=_lib.LIF_TENSOR)
      assert np.array_equal(s, s2), ("TENSOR production and u_final variants differ", T, yb)
      tens[yb] = (s, u)
    s, u = tens[False]
    assert np.array_equal(tens[True][0], s) and np.array_equal(tens[True][1], u)
    assert np.array_equal(s[:24], s_ref[:24]), ("TENSOR", T, np.argwhere(s[:24] != s_ref[:24])[:8].tolist())
    if T <= 24:
      assert np.array_equal(u, info["u"]), ("TENSOR u_T", T, np.argwhere(u != info["u"])[:8].tolist())
      continue
    # T = 26: channels 0, 1, 3 exact at every step; the bias 1 / -1 channels show the accumulation's rounding
    ladder, neg = np.arange(2, 128, 5), np.arange(4, 128, 5)
    other = np.setdiff1d(np.arange(128), np.concatenate([ladder, neg]))
    assert np.array_equal(s[..., other], s_ref[..., other]) and np.array_equal(u[..., other], info["u"][..., other])
    assert np.array_equal(s[..., neg], s_ref[..., neg])
    rn = dict(fire25=1, u_ladder=F32(0.5), u_neg=F32(-1.0))                      # round to nearest (= ref_int)
    tz = dict(fire25=0, u_ladder=F32(1 - 2.0 ** -24), u_neg=F32(-(1 - 2.0 ** -24)))   # truncation toward zero
    fire25 = np.unique(s[24][..., ladder])
    assert fire25.size == 1 and not s[25][..., ladder].any(), fire25
    mode = rn if fire25[0] == 1 else tz
    assert np.all(u[..., ladder] == mode["u_ladder"]) and np.all(u[..., neg] == mode["u_neg"]), \
        (np.unique(u[..., ladder]).tolist(), np.unique(u[..., neg]).tolist())
    print(f"\nLIF_TENSOR ladder step 25: {'fires (round to nearest)' if mode is rn else 'silent (truncation)'}")


@gpu
def test_tensor_accumulation_error_t1(cuda_lib, oracle_lib):
  """T = 1 measures LIF_TENSOR's per-step error directly: u_T = U_1 for the silent neurons, so err = |u_T - U_1| minus
  the operand-piece error is the tensor core's accumulation error.  It must stay within C_ACC EPS M, M = A |s| / 2 +
  |b| / 2 (in threshold units).  Reports max err / (EPS M)."""
  ratios = []
  for seed, lam in ((41, 0.3), (42, 2.0), (43, 20.0)):
    rng, lay, q, bn, stt, scale, bias = random_conv1(seed)
    x = np.minimum(rng.poisson(lam, size=(1, 4, 16, 256, 2)), 255).astype(np.uint8)
    packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
    band = conv1_band(x, q, scale, bias, modes=("tensor",), c_acc=0.0)        # delta = the piece errors alone
    s, u, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05, dumps="u",
                       lif_mode=_lib.LIF_TENSOR)
    acc = ref_int.conv3x3_acc(x[0], q).astype(np.float64)
    A = ref_int.conv3x3_acc(x[0], np.abs(q.astype(np.int16)).astype(np.int8)).astype(np.float64)
    U = (acc * scale.astype(np.float64) + bias.astype(np.float64)) * 0.5
    M = A * np.abs(scale.astype(np.float64)) * 0.5 + np.abs(bias.astype(np.float64)) * 0.5
    silent = (U < 1.0) & (u != 0)
    err = np.maximum(np.abs(u.astype(np.float64) - U) - band["delta_tensor"], 0.0)
    r = err[silent] / (EPS * M[silent])
    ratios.append(float(r.max()))
    assert silent.sum() > 1000
  print(f"\nLIF_TENSOR accumulation error per step: max err / (2^-24 M) = {max(ratios):.3f} (C_ACC = {C_ACC})",
        ratios)
  assert max(ratios) <= C_ACC, ratios


@gpu
def test_dyadic_layer_bit_exact_every_mode(cuda_lib, oracle_lib):
  """On dyadic_layer every operation of every mode is exact, so EXACT, FAST (101-103) and TENSOR equal float64 bit
  for bit -- pooled spikes in u8 and bit layouts, u_T for EXACT and TENSOR -- with hundreds of exact ties U == 1."""
  q, scale, bias, x = dyadic_layer()
  band = conv1_band(x, q, scale, bias, modes=())
  assert band["ties"] >= 300
  wq, sd, bd = packed_q(q, scale, bias)
  for bm in (False, True):
    s, u, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps="u", batch_major=bm,
                       lif_mode=_lib.LIF_EXACT)
    assert np.array_equal(s, band["pooled"]) and np.array_equal(u.astype(np.float64), band["u"]), ("EXACT", bm)
    for yb in (False, True):
      for lm in (_lib.LIF_EXACT,) + FAST_MODES:
        s, _, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps=False, batch_major=bm,
                           y_bits=yb, lif_mode=lm)
        assert np.array_equal(s, band["pooled"]), (lm, bm, yb, np.argwhere(s != band["pooled"])[:8].tolist())
      s, u, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps="u", batch_major=bm, y_bits=yb,
                         lif_mode=_lib.LIF_TENSOR)
      assert np.array_equal(s, band["pooled"]), ("TENSOR", bm, yb, np.argwhere(s != band["pooled"])[:8].tolist())
      d = np.argwhere(u.astype(np.float64) != band["u"])
      assert d.size == 0, ("TENSOR u_T", bm, yb, d[:8].tolist())


@pytest.fixture(scope="module")
def production():
  lay, bn, stt, q, scale, bias, x = production_conv1()
  band = conv1_band(x, q, scale, bias, modes=("fast", "tensor"))
  return dict(lay=lay, bn=bn, stt=stt, q=q, x=x, band=band)


@gpu
def test_production_shape_band(cuda_lib, oracle_lib, production):
  """conv1 of the synthetic network (seed 1, stable), H = W = 128, T = 20, B = 5: 160 work items, a full wave of 148
  persistent CTAs plus a ragged one.  Both batch orders, u8 and bit-packed output: TENSOR (with u_T) and FAST / 101-103
  (spikes) decide every decided pooled output as float64 does, TENSOR's synchronised membranes are within delta_T, every
  flip against the fp32 reference is an excluded output, and the excluded fraction stays below 1e-2."""
  pr = production
  band, x = pr["band"], pr["x"]
  packed = pk_mod.pack_conv3x3(pr["lay"], 8, DEV, pr["bn"], pr["stt"])
  report = []
  for bm in (False, True):
    for yb in (False, True):
      s, u, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05, dumps="u",
                         batch_major=bm, y_bits=yb, lif_mode=_lib.LIF_TENSOR)
      st = check_band(band, "tensor", s, u, ("TENSOR", bm, yb))
      assert st["flips_outside_excluded"] == 0 and st["excluded"] < 1e-2, st
      report.append(("TENSOR", bm, yb, _fmt(st)))
      for lm in FAST_MODES:
        s, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05,
                           dumps=False, batch_major=bm, y_bits=yb, lif_mode=lm)
        st = check_band(band, "fast", s, None, (lm, bm, yb))
        assert st["flips_outside_excluded"] == 0 and st["excluded"] < 1e-2, st
        report.append((lm, bm, yb, _fmt(st)))
  print("\n" + "\n".join(map(str, report)))


def _stress_cases():
  """(name, q, scale, bias, x): cancellation (count-255 blocks under mixed-sign weights: A_t large, acc_t near 0) and a
  bias-dominated domain (one channel's 0.5 |b| above every 63.5 |s|)."""
  out = []
  rng, lay, q, bn, stt, scale, bias = random_conv1(51)
  qc = q.copy()
  qc[:, :, 0, :] = np.abs(qc[:, :, 0, :])
  qc[:, :, 1, :] = -qc[:, :, 0, :]                                # each tap's two input channels cancel
  x = frames(rng, (6, 2, 8, 128, 2))
  blk = rng.uniform(size=(6, 2, 4, 64)) < 0.25
  blk = np.repeat(np.repeat(blk, 2, axis=2), 2, axis=3)
  x[blk] = 255                                                    # both channels of the pixel: acc cancels to ~0
  sc = scale * F32(8.0)                                           # so that U sits near the threshold
  out.append(("cancellation", qc, sc.astype(F32), bias, x))
  rng, lay, q, bn, stt, scale, bias = random_conv1(52)
  bias = bias.copy()
  bias[7] = F32(2.0 * 63.5 * np.abs(scale).max() * 3.0)
  assert 0.5 * bias[7] > 63.5 * np.abs(scale).max()
  out.append(("bias_dominated", q, scale, bias, frames(rng, (6, 2, 8, 128, 2))))
  return out


@pytest.mark.parametrize("idx", [0, 1], ids=["cancellation", "bias_dominated"])
def test_stress_cases_in_band_cpu(oracle_lib, idx):
  name, q, scale, bias, x = _stress_cases()[idx]
  band = conv1_band(x, q, scale, bias, emulate=("fast", "tensor"))
  check_band(band, "exact", band["ref"], band["ref_u"], name)
  check_band(band, "fast", band["emu_fast"], band["emu_u_fast"], name)
  check_band(band, "tensor", band["emu_tensor"], band["emu_u_tensor"], name)


@gpu
@pytest.mark.parametrize("idx", [0, 1], ids=["cancellation", "bias_dominated"])
def test_stress_cases_band(cuda_lib, oracle_lib, idx):
  """Cancellation and a bias-dominated domain through EXACT (bit-exact), FAST / 101-103 and TENSOR (band)."""
  name, q, scale, bias, x = _stress_cases()[idx]
  band = conv1_band(x, q, scale, bias)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  wq, sd, bd = packed_q(q, scale, bias)
  s, u, acc = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, lif_mode=_lib.LIF_EXACT)
  assert np.array_equal(acc, info["acc"]) and np.array_equal(s, s_ref) and np.array_equal(u, info["u"])
  for yb in (False, True):
    for lm in FAST_MODES:
      s, _, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps=False, y_bits=yb, lif_mode=lm)
      check_band(band, "fast", s, None, (name, lm, yb))
    s, u, _ = run_conv(cuda_lib, x, wq, sd, bd, 128, True, _lib.IMPL_TCGEN05, dumps="u", y_bits=yb,
                       lif_mode=_lib.LIF_TENSOR)
    print("\n", name, yb, _fmt(check_band(band, "tensor", s, u, (name, yb))))


@gpu
def test_popcount_variants_equal_their_bits(cuda_lib, oracle_lib):
  """y_popcount of k_conv1_tclif<POPC> (LIF_TENSOR) and k_conv1_umma FAST POPC (LIF_FAST, EXACT) equals, per (b, t), the
  popcount of the bits the same launch wrote, and the spikes equal the non-POPC launch's."""
  rng, lay, q, bn, stt, scale, bias = random_conv1(61)
  x = frames(rng, (5, 3, 8, 256, 2))
  T, B = x.shape[:2]
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  band = conv1_band(x, q, scale, bias, modes=("fast", "tensor"))
  for lm in (_lib.LIF_TENSOR, _lib.LIF_FAST, _lib.LIF_EXACT):
    for bm in (False, True):
      cnt = torch.zeros((B, T), device=DEV, dtype=torch.int32)
      s, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05, dumps=False,
                         y_bits=True, lif_mode=lm, batch_major=bm, popcount=cnt)
      s0, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05,
                          dumps=False, y_bits=True, lif_mode=lm, batch_major=bm)
      assert np.array_equal(s, s0), (lm, bm)
      want = s.sum(axis=(2, 3, 4), dtype=np.int64).T
      assert np.array_equal(cnt.cpu().numpy(), want), (lm, bm, cnt.cpu().numpy().tolist(), want.tolist())
      if lm != _lib.LIF_EXACT:
        check_band(band, "tensor" if lm == _lib.LIF_TENSOR else "fast", s, None, (lm, bm))


@gpu
def test_engine_tracked_densities_default_mode(cuda_lib):
  """CextNetEngine(track_densities=True) in its default conv1 mode (LIF_TENSOR): densities() of conv_1 / conv_2 /
  conv_t_0 inputs, counted by the producing epilogues, equal density_stats of the spikes that forward wrote."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet
  from snnquantprune_b200.input_pipeline import density_stats
  bits, T, H, B = 8, 4, 128, 3
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  fr = torch.as_tensor(synthetic.make_frames(B, T, H, H, seed=2)).cuda()
  eng = CextNetEngine(pack_cextnet(v, bits, T, H, device="cuda"), track_densities=True)
  assert eng.lif_mode == _lib.LIF_TENSOR and eng.packed_spikes
  eng.forward(fr)
  d = eng.densities()
  ws = list(eng._ws.values())[-1]
  for key, name in (("conv_1_inpt", "s1"), ("conv_2_inpt", "s2"), ("conv_t_0_inpt", "s3")):
    x = ws[name][:B].contiguous()
    w = density_stats(x, B * T, bits=True)
    assert d[key]["min"] == float(w["min"]) and d[key]["mean"] == float(w["mean"]), (key, d[key], w)
  assert 0.0 < d["conv_1_inpt"]["mean"] < 1.0


@gpu
def test_tensor_layouts_and_routing(cuda_lib, oracle_lib):
  """LIF_TENSOR with padded x / y strides (+16 k bytes) in both batch orders, a sample sub-range (pointer offset, as
  the engine's chunks), T = 1 and B = 1 (the tensor map's stride substitution): the same bits as the contiguous launch,
  inside the band.  Outside the envelope (W = 64, H = 6, an x stride that is not a multiple of 16) the mode means the
  reference order: bit-exact against ref_int, or an error code -- never a different answer."""
  rng, lay, q, bn, stt, scale, bias = random_conv1(71)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  T, B, H, W = 4, 3, 8, 128
  x = frames(rng, (T, B, H, W, 2))
  band = conv1_band(x, q, scale, bias, modes=("tensor",))
  ref, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05, dumps=False,
                       lif_mode=_lib.LIF_TENSOR)
  check_band(band, "tensor", ref, None, "contiguous")
  img = H * W * 2
  for bm in (False, True):
    for pad in (16, 48):
      # x padded: every (t, b) image starts pad bytes after the previous one's end
      n0, n1 = (B, T) if bm else (T, B)
      buf = torch.zeros((n0 * n1 * (img + pad) + 64,), device=DEV, dtype=torch.uint8)
      xv = buf[:n0 * n1 * (img + pad)].view(n0, n1, img + pad)[:, :, :img]
      xv.copy_(torch.as_tensor(np.ascontiguousarray(np.swapaxes(x, 0, 1) if bm else x).reshape(n0, n1, img)))
      xs = (xv.stride(1), xv.stride(0)) if bm else (xv.stride(0), xv.stride(1))
      for yb in (False, True):
        C8 = 16 if yb else 128
        yimg = (H // 2) * (W // 2) * C8
        ybuf = torch.full((n0, n1, yimg + 8 * pad), 7, device=DEV, dtype=torch.uint8)
        yv = ybuf[:, :, :yimg]
        ys = (yv.stride(1), yv.stride(0)) if bm else (yv.stride(0), yv.stride(1))
        rc, _, _ = launch(cuda_lib, xv, (T, B, H, W), packed.wq, packed.scale, packed.bias, lif_mode=_lib.LIF_TENSOR,
                          y_bits=yb, x_strides=xs, y=yv, y_strides=ys)
        _lib.check(rc)
        y = yv.reshape(n0, n1, H // 2, W // 2, C8).cpu().numpy()
        y = np.swapaxes(y, 0, 1) if bm else y
        if yb:
          y = np.unpackbits(y, axis=-1, bitorder="little")
        assert np.array_equal(y, ref), ("padded", bm, pad, yb)
        assert np.all(ybuf[:, :, yimg:].cpu().numpy() == 7), "write past the image"
  # a sample sub-range: samples 1..2 of the batch-major tensor
  xb = torch.as_tensor(np.ascontiguousarray(np.swapaxes(x, 0, 1)), device=DEV)
  rc, y, _ = launch(cuda_lib, xb[1], (T, 2, H, W), packed.wq, packed.scale, packed.bias, lif_mode=_lib.LIF_TENSOR,
                    y_bits=True, x_strides=(xb.stride(1), xb.stride(0)))
  _lib.check(rc)
  assert np.array_equal(unbits(y), ref[:, 1:3]), "sample sub-range"
  # T = 1 and B = 1: the stride substitution (a stride that is meaningless for a single step / sample)
  for Tn, Bn in ((1, B), (T, 1), (1, 1)):
    xs = np.ascontiguousarray(x[:Tn, :Bn])
    bnd = conv1_band(xs, q, scale, bias, modes=("tensor",))
    xd = torch.as_tensor(xs, device=DEV)
    rc, y, u = launch(cuda_lib, xd, (Tn, Bn, H, W), packed.wq, packed.scale, packed.bias, lif_mode=_lib.LIF_TENSOR,
                      y_bits=False, u_final=True, x_strides=(12345 * 16 if Tn == 1 else xd.stride(0),
                                                             777 * 16 if Bn == 1 else xd.stride(1)))
    _lib.check(rc)
    check_band(bnd, "tensor", y.cpu().numpy(), u.cpu().numpy(), ("T/B = 1", Tn, Bn))
    if Tn == T:
      assert np.array_equal(y.cpu().numpy(), ref[:, :Bn])
  # outside the envelope
  for shp in ((2, 2, 8, 64), (2, 2, 6, 128)):
    Tn, Bn, Hn, Wn = shp
    xs = frames(rng, (Tn, Bn, Hn, Wn, 2))
    s_ref, info = ref_int.spiking_conv3x3(xs, q, scale, bias, pool=True, want=True)
    for lm in (_lib.LIF_TENSOR, _lib.LIF_EXACT):
      try:
        s, u, _ = run_conv(cuda_lib, xs, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05,
                           dumps="u", lif_mode=lm)
      except _lib.SnnqpError:
        continue
      assert np.array_equal(s, s_ref) and np.array_equal(u, info["u"]), (shp, lm)
    try:
      s, _, _ = run_conv(cuda_lib, xs, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05,
                         dumps=False, lif_mode=_lib.LIF_TENSOR)
    except _lib.SnnqpError:
      continue
    assert np.array_equal(s, s_ref), shp
  xs = x[:, :1]
  s_ref = ref_int.spiking_conv3x3(xs, q, scale, bias, pool=True)
  buf = torch.zeros((T * (img + 8) + 64,), device=DEV, dtype=torch.uint8)
  xv = buf[:T * (img + 8)].view(T, img + 8)[:, :img]
  xv.copy_(torch.as_tensor(np.ascontiguousarray(xs).reshape(T, img)))
  rc, y, _ = launch(cuda_lib, xv, (T, 1, H, W), packed.wq, packed.scale, packed.bias, lif_mode=_lib.LIF_TENSOR,
                    y_bits=False, x_strides=(xv.stride(0), T * (img + 8)))
  if rc == 0:
    assert np.array_equal(y.cpu().numpy(), s_ref), "x stride not a multiple of 16"
