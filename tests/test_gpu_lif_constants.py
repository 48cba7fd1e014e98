"""Every fused spiking block under multi_step_LIF constants other than (tau = 2, v_threshold = 1, v_reset = 0), and the
128-channel blocks under count-valued u8 input, bit for bit against the integer oracle (oracle/ref_int.py) or the
attention-path emulation (tests/attref.py) run with the same constants.

The constants travel in snnqp_block_params.  The production epilogues hard-code the standard ones (LifParams<true>,
conv1's FAST / TENSOR / 101-103 variants), so every launcher must check all three before it picks one of them, and
must refuse bit-packed output (which only those epilogues emit) otherwise.  Each constant set catches one way this
can go wrong (LIF_SETS).  A layer's bias is shifted by v_threshold - v_reset - 1: under a constant drive v the
membrane settles at v + v_reset, so the shift keeps the firing regime of the standard layer (except for the set that
is meant to fire everywhere); tau > 2 adds 0.2 (tau - 2), since over a few steps a slower membrane stays further
below that level.

CPU tests (unmarked) pin the C oracle's generic LIF to ref_snn.lif_step, which the executed reference pins
(test_from_reference_cpu.py), and build every GPU case's reference to check that it is not vacuous: its spike rate
is inside bounds, and setting any one non-default field back to its default changes its outputs, so a kernel that
ignores tau, v_threshold or v_reset fails."""
import functools
import json
import os

import numpy as np
import pytest
import torch

import attref as ar
import test_gpu_attention_path as tap
from oracle import ref_int, ref_net, ref_snn
from snnquantprune_b200 import _lib, synthetic
from snnquantprune_b200 import pack as pk_mod
from test_gpu_parity import check_free_running_vs_float_path, make_layer, run_conv, run_dense

F32 = np.float32
DEV = "cuda"
gpu = pytest.mark.gpu
P = _lib.ptr
GOLD = os.path.join(os.path.dirname(__file__), "golden")
OPS = np.load(os.path.join(GOLD, "from_reference_ops.npz"))
META = json.loads(str(OPS["meta"]))

DEFAULT = (2.0, 1.0, 0.0)
LIF_SETS = {                                   # (tau, v_threshold, v_reset)
    "ref_case": (1.7, 0.8, 0.1),               # the executed reference's own non-default case
    "tau3": (3.0, 1.0, 0.0),                   # one field off the default at a time: each catches a routing check
    "vth075": (2.0, 0.75, 0.0),                #   that omits that field and lets a hard-coded variant run
    "vreset0125": (2.0, 1.0, 0.125),
    "tau2_vth_vreset": (2.0, 0.5, -0.25),      # tau = 2 with other threshold and reset: the TAU2 specialisations
    "fires_everywhere": (2.0, -0.5, 0.0),      # fires on the constants alone: phantom rows of a partial tile fire
    "ties": (4.0, 0.75, 0.25),                 # exact ties un == v_th on the identity-centre-tap grid
    "reset_above_th": (0.5, 1.0, 1.2),         # reset above the threshold (repeated firing), tau < 1
}
RATE = {"fires_everywhere": (0.5, 1.0)}        # every other set: (0.02, 0.9)
LIF_MODES = (_lib.LIF_EXACT, _lib.LIF_FAST, _lib.LIF_TENSOR, 101, 102, 103)


def lif_kw(name):
  return dict(zip(("tau", "v_th", "v_reset"), LIF_SETS[name]))


def bias_shift(name):
  tau, vth, vr = LIF_SETS[name]
  return 0.0 if name == "fires_everywhere" else vth - vr - 1.0 + 0.2 * max(tau - 2.0, 0.0)


def shifted(bias, name):
  return (np.asarray(bias, np.float64) + bias_shift(name)).astype(F32)


def defaulted(consts):
  """consts with each non-default field set back to its default, one at a time."""
  return [tuple(d if j == i else v for j, v in enumerate(consts)) for i, (c, d) in enumerate(zip(consts, DEFAULT))
          if c != d]


def assert_not_vacuous(name, label, lif_fn, spikes, u):
  """lif_fn(tau, v_th, v_reset) -> (spikes, u_T) of the same case under other constants."""
  lo, hi = RATE.get(name, (0.02, 0.9))
  rate = float(np.mean(spikes != 0))
  assert lo < rate <= hi, (name, label, rate)
  for c in defaulted(LIF_SETS[name]):
    s2, u2 = lif_fn(*c)
    assert not (np.array_equal(s2, spikes) and np.array_equal(np.asarray(u2).view(np.uint32),
                                                              np.asarray(u).view(np.uint32))), (name, label, c)


def dev(a):
  return torch.as_tensor(np.ascontiguousarray(a), device=DEV)


def diffs(**pairs):
  """name=(got, want) -> the names that differ (compared as raw bits)."""
  bad = []
  for k, (g, w) in pairs.items():
    g, w = np.asarray(g), np.asarray(w)
    if g.dtype == np.float32:
      g, w = g.view(np.uint32), w.astype(F32).view(np.uint32)
    if g.shape != w.shape or not np.array_equal(g, w):
      bad.append(k if g.shape != w.shape else f"{k}: {int((g != w).sum())} of {g.size} differ")
  return bad


def counts_of(s_un):
  """un-pooled spikes (T, B, H, W, C) -> spike_counts layout (B, T, C)."""
  return s_un.sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2)


def expect_unsupported(fn):
  with pytest.raises(_lib.SnnqpError) as e:
    fn()
  assert e.value.code == 3, str(e.value)


# ================================================================================ CPU: the oracle's LIF ====
@pytest.mark.parametrize("name", ["default"] + list(LIF_SETS))
def test_oracle_lif_matches_reference_lif_step(oracle_lib, name):
  """orc_lif_from_acc / orc_lif_from_f32 (zero carry, v = fmaf(acc, scale, bias)) equal ref_snn.lif_step on the same
  pre-activations bit for bit: the fixture's lif*_x (fp32 accumulators) and random int32 accumulators, each with
  scale 1 / bias 0 and with a non-trivial scale and bias."""
  tau, vth, vr = DEFAULT if name == "default" else LIF_SETS[name]
  rng = np.random.default_rng(3)
  cases = [(OPS[f"lif{ci}_x"].astype(F32), sb) for ci in range(len(META["lif_cases"]))
           for sb in ((1.0, 0.0), (0.37, 0.11))]
  cases += [(rng.integers(-4, 5, size=(8, 4096)).astype(np.int32), (1.0, 0.0)),
            (rng.integers(-3000, 3000, size=(8, 4096)).astype(np.int32), (2.0 ** -9, 0.3)),
            (rng.integers(-3000, 3000, size=(8, 4096)).astype(np.int32), (3.1e-4, -0.17))]
  fired = 0
  for acc, (sc, bi) in cases:
    scale, bias = np.full(1, sc, F32), np.full(1, bi, F32)
    s, uT = ref_int.lif_from_acc(np.ascontiguousarray(acc[:, :, None]), scale, bias, tau, vth, vr)
    u = np.zeros(acc.shape[1], F32)
    for t in range(acc.shape[0]):
      v = ref_int.fmaf(acc[t].astype(F32), scale[0], bias[0])
      u, st = ref_snn.lif_step(u, v, tau, vth, vr)
      assert np.array_equal(s[t, :, 0] != 0, st != 0), (name, acc.dtype, sc, t)
    assert np.array_equal(uT[:, 0].view(np.uint32), u.view(np.uint32)), (name, acc.dtype, sc)
    fired += int(s.sum())
  assert fired > 0


# ===================================================================================== the cases ====
CONV1_SHAPES = [((3, 2, 8, 64, 2), 8, True), ((2, 1, 6, 128, 2), 4, False), ((5, 3, 128, 128, 2), 8, True)]


@functools.lru_cache(maxsize=None)
def conv1_data(i):
  """The data of test_spiking_conv1_tcgen05_bit_exact (test_gpu_parity.py): Poisson counts with extreme corners."""
  shape, bits, pool = CONV1_SHAPES[i]
  rng = np.random.default_rng(shape[2] * 5 + bits)
  lay, q, bn, stt = make_layer(rng, 2, 128, bits, 0.3)
  x = np.minimum(rng.poisson(0.3, size=shape), 255).astype(np.uint8)
  x[0, 0, 0, 0, :] = 255; x[-1, -1, -1, -1, :] = 200
  T, B, H, W, _ = shape
  acc = ref_int.conv3x3_acc(x.reshape(T * B, H, W, 2), q).reshape(T, B, H, W, 128)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128)
  return lay, bn, stt, bits, pool, x, acc, scale, bias


TILE_SHAPES = [(2, 5, 64, 64), (3, 20, 24, 32), (2, 10, 18, 64)]    # (T, B, H, W): 160 work items each (> 148 SMs)
SIMT_TILE_SHAPE = (3, 2, 16, 16)


@functools.lru_cache(maxsize=None)
def tile_data(shape):
  """conv2-4 geometry; H = 24: whole epilogue warps below the image in the last tile row, H = 18: a thread's second
  row pair (as test_gpu_persistent_schedules.py)."""
  T, B, H, W = shape
  rng = np.random.default_rng(1000 + H + W)
  lay, q, bn, stt = make_layer(rng, 128, 128, 8, 0.5)
  x = (rng.uniform(size=(T, B, H, W, 128)) < 0.25).astype(np.uint8)
  acc = ref_int.conv3x3_acc(x.reshape(T * B, H, W, 128), q).reshape(T, B, H, W, 128)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  return lay, bn, stt, x, acc, scale, bias


def lif_ref(name, label, acc, scale, bias):
  """(spikes, u_T) of the generic LIF with the set's constants on acc (int32 or fp32), checked not to be vacuous."""
  s, u = ref_int.lif_from_acc(acc, scale, bias, *LIF_SETS[name])
  assert_not_vacuous(name, label, lambda *c: ref_int.lif_from_acc(acc, scale, bias, *c), s, u)
  return s, u


CONV5_CASES = [(_lib.IMPL_TCGEN05, 5, 60, 16, "bt", 0), (_lib.IMPL_TCGEN05, 3, 24, 8, "tb", 1),
               (_lib.IMPL_SIMT, 4, 2, 16, "tb", 4)]      # (impl, T, B, H, att layout, att row pad)


@functools.lru_cache(maxsize=None)
def conv5_data(i):
  impl, T, B, H, layout, pad = CONV5_CASES[i]
  rng = np.random.default_rng(300 + i)
  lay, q, bn, stt, scale, bias = tap.conv_layer(310 + i)
  bias = (bias + F32(0.3)).astype(F32)                 # att < 1 scales the drive down: conv5 fires at ~2 % otherwise
  x = (rng.uniform(size=(T, B, H, 8, 128)) < 0.3).astype(np.uint8)
  att = tap.edge_att(rng, T, B)
  emu = ar.conv_att_tc_acc(x, att, q) if impl == _lib.IMPL_TCGEN05 else ar.conv_att_simt_acc(x, att, q)
  return lay, q, bn, stt, scale, bias, x, att, emu


DENSE_BIN_CASES = [(_lib.IMPL_TCGEN05, 5, 4800, 256, 110),     # 150 column tiles of 32 samples: more than the SMs
                   (_lib.IMPL_TCGEN05, 20, 19, 512, 110), (_lib.IMPL_SIMT, 3, 9, 100, 40)]
DENSE_ATT_CASES = [(_lib.IMPL_TCGEN05, 3, 101), (_lib.IMPL_SIMT, 3, 6)]


def dense_binary_layer(rng, K, N, bits=8):
  from oracle import ref_quant
  k = (rng.standard_normal((K, N)) * (5.0 / np.sqrt(K))).astype(F32)
  mask = ref_quant.local_mask(k, 0.5)
  a = ref_quant.gaussian_init(k, bits)
  lay = {"kernel": k, "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)}, "prune_0": {"mask": mask}}
  q = ref_int.duq_levels_c(k, mask, a, bits)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], bits, n=N)
  return lay, q, scale, bias


@functools.lru_cache(maxsize=None)
def dense_bin_data(i):
  impl, T, B, K, N = DENSE_BIN_CASES[i]
  rng = np.random.default_rng(K + N + i)
  lay, q, scale, bias = dense_binary_layer(rng, K, N)
  x = (rng.uniform(size=(T, B, K)) < 0.2).astype(np.uint8)
  return lay, scale, bias, x, ref_int.dense_acc(x, q)


@functools.lru_cache(maxsize=None)
def dense_att_data(i):
  impl, T, B = DENSE_ATT_CASES[i]
  rng = np.random.default_rng(400 + i)
  lay, q, scale, bias = tap.dense_layer(410 + i)
  x = (rng.uniform(size=(T, B, 2048)) < 0.15).astype(np.uint8)
  att = tap.edge_att(rng, T, B)
  att_k = np.tile(att, (1, 1, 16))
  emu = ar.dense_att_tc_acc(x, att_k, q) if impl == _lib.IMPL_TCGEN05 else ar.dense_att_simt_acc(x, att_k, q)
  return lay, q, scale, bias, x, att, emu


def build_refs(name):
  """Every per-block reference of the set (spikes, u_T), each checked not to be vacuous."""
  out = {}
  for i in range(len(CONV1_SHAPES)):
    _, _, _, _, _, _, acc, scale, bias = conv1_data(i)
    out["conv1", i] = lif_ref(name, ("conv1", i), acc, scale, shifted(bias, name))
  for shape in TILE_SHAPES + [SIMT_TILE_SHAPE]:
    *_, acc, scale, bias = tile_data(shape)
    out["tile", shape] = lif_ref(name, ("tile", shape), acc, scale, shifted(bias, name))
  for i in range(len(CONV5_CASES)):
    _, _, _, _, scale, bias, _, _, emu = conv5_data(i)
    out["conv5", i] = lif_ref(name, ("conv5", i), emu, scale, shifted(bias, name))
  for i in range(len(DENSE_BIN_CASES)):
    _, scale, bias, _, acc = dense_bin_data(i)
    out["dense_bin", i] = lif_ref(name, ("dense_bin", i), acc, scale, shifted(bias, name))
  for i in range(len(DENSE_ATT_CASES)):
    _, _, scale, bias, _, _, emu = dense_att_data(i)
    out["dense_att", i] = lif_ref(name, ("dense_att", i), emu, scale, shifted(bias, name))
  return out


@pytest.mark.parametrize("name", list(LIF_SETS))
def test_cases_are_not_vacuous(oracle_lib, name):
  """Reference side of every GPU case below: spike rate inside bounds, outputs sensitive to each non-default field."""
  build_refs(name)


# ======================================================================================= GPU: conv1 ====
def popcount_buf(B, T):
  return torch.zeros((B, T), device=DEV, dtype=torch.int32)


@gpu
@pytest.mark.parametrize("name", list(LIF_SETS))
def test_conv1_lif_constants_bit_exact(cuda_lib, oracle_lib, name):
  """k_conv1_umma (generic epilogue) and the SIMT conv1 under the set's constants, both (t, b) orders: under every
  lif_mode, the call with every dump (accumulators, spikes, u_T), with membranes only, and without dumps (production),
  all bit-exact to the reference order.  Bit-packed output (with or without y_popcount) must be refused (code 3)."""
  lif = lif_kw(name)
  for i, (shape, _, _) in enumerate(CONV1_SHAPES):
    lay, bn, stt, bits, pool, x, acc_ref, scale, bias = conv1_data(i)
    bias_s = shifted(bias, name)
    s_un, u_ref = ref_int.lif_from_acc(acc_ref, scale, bias_s, **lif)
    s_ref = ref_int.maxpool2_u8(s_un) if pool else s_un
    packed = pk_mod.pack_conv3x3(lay, bits, DEV, bn, stt)
    packed.bias.copy_(dev(bias_s))
    T, B = shape[:2]
    for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
      for bm in (True, False):
        run = lambda **kw: run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl,
                                    batch_major=bm, **lif, **kw)
        tag = (name, shape, impl, bm)
        for lm in LIF_MODES if impl == _lib.IMPL_TCGEN05 else (_lib.LIF_EXACT,):
          s, u, acc = run(lif_mode=lm)
          bad = diffs(acc=(acc, acc_ref), spikes=(s, s_ref), u_final=(u, u_ref))
          assert not bad, (tag, "every dump", lm, bad)
          if pool:
            s, u, _ = run(dumps="u", lif_mode=lm)
            assert not diffs(spikes=(s, s_ref), u_final=(u, u_ref)), (tag, "membranes only", lm)
          s, _, _ = run(dumps=False, lif_mode=lm)
          assert np.array_equal(s, s_ref), (tag, "production", lm)
        if pool and impl == _lib.IMPL_TCGEN05:
          for lm in (_lib.LIF_EXACT, _lib.LIF_FAST, _lib.LIF_TENSOR):
            expect_unsupported(lambda: run(dumps=False, y_bits=True, lif_mode=lm))
            expect_unsupported(lambda: run(dumps=False, y_bits=True, lif_mode=lm, popcount=popcount_buf(B, T)))


# ================================================================================= GPU: conv2 - conv4 ====
def check_tile(lib, name, shape, impl, lif):
  lay, bn, stt, x, acc_ref, scale, bias = tile_data(shape)
  T, B, H, W = shape
  bias_s = shifted(bias, name)
  s_un, u_ref = ref_int.lif_from_acc(acc_ref, scale, bias_s, **lif)
  s_pool, cnt_ref = ref_int.maxpool2_u8(s_un), counts_of(s_un)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  packed.bias.copy_(dev(bias_s))
  cnt = torch.zeros((B, T, 128), device=DEV, dtype=torch.int32)
  x_formats = (False, True) if impl == _lib.IMPL_TCGEN05 else (False,)
  for xb in x_formats:
    for bm in (True, False):
      run = lambda pool, **kw: run_conv(lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl, batch_major=bm,
                                        x_bits=xb, counts=cnt, **lif, **kw)
      tag = (name, shape, impl, "x_bits" if xb else "x_u8", "bt" if bm else "tb")
      cnt.zero_()
      s, u, acc = run(pool=False)                                   # instrumented: every dump, un-pooled spikes
      bad = diffs(acc=(acc, acc_ref), spikes=(s, s_un), u_final=(u, u_ref), counts=(cnt.cpu().numpy(), cnt_ref))
      assert not bad, (tag, "instrumented", bad)
      cnt.zero_()
      s, _, _ = run(pool=True, dumps=False)                         # production-shaped: pooled spikes + counts
      bad = diffs(spikes=(s, s_pool), counts=(cnt.cpu().numpy(), cnt_ref))
      assert not bad, (tag, "production", bad)
  if impl == _lib.IMPL_TCGEN05:
    expect_unsupported(lambda: run_conv(lib, x, packed.wq, packed.scale, packed.bias, 128, True, impl, batch_major=True,
                                        x_bits=True, y_bits=True, dumps=False, **lif))


@gpu
@pytest.mark.parametrize("name", list(LIF_SETS))
def test_tile_conv_lif_constants_bit_exact(cuda_lib, oracle_lib, name):
  """k_conv3x3_tile's generic epilogue under the set's constants at three multi-wave shapes, two of them ending in a
  partial tile row: u8 and bit-packed input, both (t, b) orders, the instrumented call (accumulators, un-pooled spikes,
  u_T, spike counts) and the production-shaped call (pool, no dumps, spike counts), bit-exact; bit-packed output
  refused (code 3).  The SIMT kernel at one shape."""
  lif = lif_kw(name)
  for shape in TILE_SHAPES:
    check_tile(cuda_lib, name, shape, _lib.IMPL_TCGEN05, lif)
  check_tile(cuda_lib, name, SIMT_TILE_SHAPE, _lib.IMPL_SIMT, lif)


# ========================================================================================= GPU: conv5 ====
@gpu
@pytest.mark.parametrize("name", list(LIF_SETS))
def test_conv_att_lif_constants_bit_exact(cuda_lib, oracle_lib, name):
  """k_conv_att_umma<true> (tau = 2) / <false> and the SIMT conv5 under the set's constants: accumulators, un-pooled
  spikes, u_T, spike counts and the pooled production spikes equal the emulation followed by the generic LIF."""
  for i, (impl, T, B, H, layout, pad) in enumerate(CONV5_CASES):
    lay, q, bn, stt, scale, bias, x, att, _ = conv5_data(i)
    bias_s = shifted(bias, name)
    packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
    packed.bias.copy_(dev(bias_s))
    tap.check_conv(cuda_lib, x, att, q, packed, scale, bias_s, impl, layout=layout, pad=pad,
                   batch_major=(layout == "bt"), **lif_kw(name))


# ================================================================================= GPU: dense1 / dense2 ====
@gpu
@pytest.mark.parametrize("name", list(LIF_SETS))
def test_dense_lif_constants_bit_exact(cuda_lib, oracle_lib, name):
  """k_dense_umma<1, tau == 2> (binary input, dense2) against the integer oracle, at a shape with more column tiles
  than SMs; k_dense_umma<3, tau == 2> (att input, dense1) against the emulation; the SIMT kernels for both."""
  lif = lif_kw(name)
  for i, (impl, T, B, K, N) in enumerate(DENSE_BIN_CASES):
    lay, scale, bias, x, acc_ref = dense_bin_data(i)
    bias_s = shifted(bias, name)
    s_ref, u_ref = ref_int.lif_from_acc(acc_ref, scale, bias_s, **lif)
    packed = pk_mod.pack_dense(lay, 8, DEV)
    packed.bias.copy_(dev(bias_s))
    s, u, acc = run_dense(cuda_lib, x, packed.wq, packed.scale, packed.bias, N, impl=impl, **lif)
    bad = diffs(acc=(acc, acc_ref), spikes=(s, s_ref), u_final=(u, u_ref))
    assert not bad, (name, "binary", impl, T, B, K, N, bad)
  for i, (impl, T, B) in enumerate(DENSE_ATT_CASES):
    lay, q, scale, bias, x, att, _ = dense_att_data(i)
    bias_s = shifted(bias, name)
    packed = pk_mod.pack_dense(lay, 8, DEV)
    packed.bias.copy_(dev(bias_s))
    tap.check_dense(cuda_lib, x, att, q, packed, scale, bias_s, impl, **lif)


# ========================================================================================== GPU: ties ====
def identity_grid_ref(consts):
  """test_lif_bit_exact_vs_reference_multi_step_lif's grid: identity centre tap, scale 2^-6, bias -0.25, so the
  pre-activation is exactly x = count 2^-6 - 0.25.  ref_snn.lif_step over it -> (spikes, u_T, number of exact ties
  un == v_th)."""
  cnt = OPS["lifgrid_counts"]                          # (T, 1, H, W, C)
  tau, vth, vr = (F32(c) for c in consts)
  x = (cnt.astype(F32) * F32(2.0 ** -6) - F32(0.25)).astype(F32)
  u = np.zeros(cnt.shape[1:], F32)
  spikes, ties = [], 0
  for t in range(cnt.shape[0]):
    un = (u + ((x[t] - (u - vr)).astype(F32) / tau).astype(F32)).astype(F32)
    ties += int((un == vth).sum())
    u, s = ref_snn.lif_step(u, x[t], *consts)
    spikes.append((s != 0).astype(np.uint8))
  return np.stack(spikes), u, ties


def test_identity_grid_has_exact_ties():
  s, u, ties = identity_grid_ref(LIF_SETS["ties"])
  assert ties >= 100, ties
  assert 0.02 < s.mean() < 0.9
  for c in defaulted(LIF_SETS["ties"]):
    s2, u2, _ = identity_grid_ref(c)
    assert not (np.array_equal(s2, s) and np.array_equal(u2.view(np.uint32), u.view(np.uint32))), c


@gpu
@pytest.mark.parametrize("impl", [_lib.IMPL_TCGEN05, _lib.IMPL_SIMT])
def test_exact_ties_bit_exact_vs_lif_step(cuda_lib, impl):
  """(tau, v_th, v_reset) = (4, 0.75, 0.25) on the identity-centre-tap grid: u_1 = count 2^-8, so count 192 gives
  un == v_th exactly (>= fires).  Un-pooled spikes and u_T (as uint32) bit for bit, pooled spikes of the call without
  dumps."""
  consts = LIF_SETS["ties"]
  s_ref, u_ref, ties = identity_grid_ref(consts)
  assert ties > 0
  cnt = OPS["lifgrid_counts"]
  T, B, H, W, C = cnt.shape
  wq = np.zeros((9, C, C), np.int8)
  wq[4] = np.eye(C, dtype=np.int8)                     # centre tap, [tap][cout][cin]
  blob = torch.zeros((int(cuda_lib.snnqp_conv3x3_blob_bytes(C, C)),), device=DEV, dtype=torch.int8)
  blob[:9 * C * C] = dev(wq).reshape(-1)
  nz = torch.empty((36,), device=DEV, dtype=torch.uint8)
  _lib.check(cuda_lib.snnqp_conv3x3_slab_bitmap(P(blob), C, C, P(nz), _lib.stream()))
  blob[9 * C * C:9 * C * C + 36] = nz.view(torch.int8)
  scale, bias = dev(np.full(C, 2.0 ** -6, F32)), dev(np.full(C, -0.25, F32))
  lif = dict(zip(("tau", "v_th", "v_reset"), consts))
  for bm in (True, False):
    s, u, _ = run_conv(cuda_lib, cnt, blob, scale, bias, C, False, impl, batch_major=bm, **lif)
    assert np.array_equal(s, s_ref), (impl, bm)
    assert np.array_equal(u.view(np.uint32), u_ref.view(np.uint32)), (impl, bm)
    s, _, _ = run_conv(cuda_lib, cnt, blob, scale, bias, C, True, impl, batch_major=bm, dumps=False, **lif)
    assert np.array_equal(s, ref_int.maxpool2_u8(s_ref)), (impl, bm)


# ======================================================================================= GPU: network ====
def tb(c, k):
  return np.ascontiguousarray(np.swapaxes(c[k].cpu().numpy(), 0, 1))


def engine(pk, consts, **kw):
  from snnquantprune_b200 import CextNetEngine
  tau, vth, vr = consts
  return CextNetEngine(pk, tau=tau, v_threshold=vth, v_reset=vr, **kw)


def teacher_forced(c, v, bits, H, fr, consts, b=slice(None)):
  """The oracle fed the GPU's own attention-path outputs (samples b) -> (oracle collect, logits)."""
  forced = {k: tb(c, k)[:, b] for k in ("att4", "s5", "att5", "d1")}
  co = {}
  tau, vth, vr = consts
  lo = ref_net.forward(ref_net.pack_network(v, bits, H), fr[b], collect=co, forced=forced, tau=tau, v_th=vth,
                       v_reset=vr)
  return co, lo


@gpu
def test_network_lif_constants_small(cuda_lib, oracle_lib):
  """(1.7, 0.8, 0.1) at H = 32, T = 4, B = 3: teacher-forced, s1-s4 with their accumulators and membranes, d2 and
  the logits bit-exact; the default lif_mode gives the logits of LIF_EXACT; free-running against the reference-order
  float path within the flip and logit budget of test_network_layerwise_teacher_forced_and_float_path."""
  from snnquantprune_b200 import pack_cextnet
  consts = LIF_SETS["ref_case"]
  bits, T, H, B = 8, 4, 32, 3
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=81)
  fr = synthetic.make_frames(B, T, H, H, seed=82)
  pk = pack_cextnet(v, bits, T, H, device=DEV)
  c = {}
  logits = engine(pk, consts, lif_mode=_lib.LIF_EXACT).forward(dev(fr), collect=c).cpu().numpy()
  co, lo = teacher_forced(c, v, bits, H, fr, consts)
  for i, k in enumerate(("s1", "s2", "s3", "s4"), 1):
    assert np.array_equal(tb(c, k), co[k]), k
    assert np.array_equal(c[f"conv{i}_acc"].cpu().numpy(), co[f"conv{i}_acc"]), f"conv{i} accumulators"
    assert np.array_equal(c[f"conv{i}_u"].cpu().numpy(), co[f"conv{i}_u"]), f"conv{i} membrane"
  assert np.array_equal(c["dense2_acc"].cpu().numpy(), co["dense2_acc"])
  assert np.array_equal(tb(c, "d2"), co["d2"]) and np.array_equal(logits, lo)
  rates = {k: float(tb(c, k).mean()) for k in ("s1", "s2", "s3", "s4", "s5", "d1", "d2")}
  assert min(rates.values()) > 0.01, rates
  co_std, _ = teacher_forced(c, v, bits, H, fr, DEFAULT)
  assert not np.array_equal(co_std["s1"], co["s1"])                 # the constants matter from the first block on
  assert np.array_equal(engine(pk, consts).forward(dev(fr)).cpu().numpy(), logits)      # default lif_mode
  check_free_running_vs_float_path(c, logits, v, fr, bits, *consts)


@gpu
def test_network_lif_constants_reference_geometry(cuda_lib, oracle_lib):
  """(1.7, 0.8, 0.1) at H = 128, T = 20, B = 2 -- where the engine would otherwise exchange bit-packed spikes, which
  only the standard constants' epilogues emit: the production forward runs and equals the instrumented forward; one
  sample teacher-forced is bit-exact on s1-s4 and the logits; CextNet with that neuron_dynamics gives the same logits."""
  from snnquantprune_b200 import pack_cextnet
  from snnquantprune_b200.models import CextNet, ModelConfig
  from snnquantprune_b200.quant import QuantConfig
  from snnquantprune_b200.spiking_learning import atan, multi_step_LIF
  consts = LIF_SETS["ref_case"]
  bits, T, H, B = 8, 20, 128, 2
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=91)
  fr = synthetic.make_frames(B, T, H, H, seed=92)
  frd = dev(fr)
  eng = engine(pack_cextnet(v, bits, T, H, device=DEV), consts)
  logits = eng.forward(frd).cpu().numpy()
  c = {}
  assert np.array_equal(eng.forward(frd, collect=c).cpu().numpy(), logits)
  co, lo = teacher_forced(c, v, bits, H, fr, consts, b=slice(0, 1))
  for i, k in enumerate(("s1", "s2", "s3", "s4"), 1):
    assert np.array_equal(tb(c, k)[:, :1], co[k]), k
    assert np.array_equal(c[f"conv{i}_u"].cpu().numpy()[:1], co[f"conv{i}_u"]), f"conv{i} membrane"
  assert np.array_equal(logits[:1], lo)
  assert min(float(tb(c, k).mean()) for k in ("s1", "s2", "s3", "s4", "s5", "d1", "d2")) > 0.01
  tau, vth, vr = consts
  cfg = ModelConfig(num_frames=T, quant=QuantConfig(bits=bits),
                    neuron_dynamics=lambda **kw: multi_step_LIF(tau=tau, spike_fn=atan, v_threshold=vth, v_reset=vr,
                                                                **kw))
  got, _ = CextNet(config=cfg).apply(v, frd)
  assert np.array_equal(got.cpu().numpy(), logits)


# ============================================================================ GPU: count-valued inputs ====
COUNT_TILE_SHAPE = (3, 20, 32, 32)     # (T, B, H, W): 160 work items, H % 16 == 0 (the production epilogue)
SAT = slice(5, 13)                     # the output channels whose levels are all +127


def saturate_channels(lay, scale, bias):
  """Every level of the SAT output channels at +127 (the kernel at the clip 2 a, unpruned), their folded scale 2^-25
  and bias 0.25 ... 0.53, so that v = acc 2^-25 + bias sits near the threshold where acc passes 2^24: the power-of-two
  scale carries one ulp of float(acc) (2 or 4 there) into v exactly, so spikes and u_T depend on how the int32 -> fp32
  conversion rounds.  The biases differ so that the channels are not copies of one another."""
  a = float(lay["DuQ_0"]["a"][0])
  lay["kernel"][..., SAT] = F32(2 * a)
  lay["prune_0"]["mask"][..., SAT] = 1.0
  n = SAT.stop - SAT.start
  scale[SAT] = F32(2.0 ** -25)
  bias[SAT] = (0.25 + 0.04 * np.arange(n)).astype(F32)


def bytes_summing_to(rng, n, total, K=128):
  """n rows of K u8 bytes (255s, one remainder byte, zeros, shuffled), each row summing to total."""
  full, rest = divmod(total, 255)
  row = np.zeros(K, np.uint8)
  row[:full] = 255
  row[full] = rest
  return np.stack([rng.permutation(row) for _ in range(n)])


def tie_bias(f, scale):
  """The bias that puts v = fma(f, scale, bias) at exactly 2.0, so that the first step's un = v / 2 meets the
  threshold 1 exactly (and fires) for float(acc) = f rounded to nearest; a conversion that rounds below f falls short."""
  b = F32(2.0 - float(f) * float(scale))
  assert float(f) * float(scale) + float(b) == 2.0
  return b


def round_toward_zero(acc):
  """int32 -> fp32 rounded toward zero (what a truncating conversion gives), as fp32 accumulators."""
  f = acc.astype(F32)
  over = np.abs(f.astype(np.float64)) > np.abs(acc.astype(np.float64))
  return np.where(over, np.nextafter(f, F32(0)), f).astype(F32)


@functools.lru_cache(maxsize=None)
def count_tile_data():
  T, B, H, W = COUNT_TILE_SHAPE
  rng = np.random.default_rng(501)
  lay, _, bn, stt = make_layer(rng, 128, 128, 8, 0.5)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  saturate_channels(lay, scale, bias)
  q = ref_int.duq_levels_c(lay["kernel"], lay["prune_0"]["mask"], lay["DuQ_0"]["a"][0], 8)
  assert (q[..., SAT] == 127).all()
  x = np.minimum(rng.poisson(0.8, size=(T, B, H, W, 128)), 255).astype(np.uint8)
  x[0, 0, 8:16, 8:16] = 255                            # saturated patches: interior, edge, corner
  x[1, 3, :6, 10:20] = 255
  x[-1, -1, -5:, -5:] = 255
  x[:, 6:10, 4:12, 4:12] = rng.integers(128, 256, size=(T, 4, 8, 8, 128))     # bytes >= 128 everywhere in patches
  # a patch whose every pixel sums to TIE_SUM over the channels: each interior output of a SAT channel sees
  # acc = 127 * 9 * TIE_SUM = TIE_ACC_T = 3 mod 4 in [2^25, 2^26), which rounds up to nearest; with channel SAT.start's
  # bias at tie_bias its first step fires exactly at the threshold, and would not for a truncated conversion
  x[0, 11, 16:24, 16:24] = bytes_summing_to(rng, 64, TIE_SUM_T).reshape(8, 8, 128)
  bias[SAT.start] = tie_bias(F32(TIE_ACC_T), scale[SAT.start])
  acc = ref_int.conv3x3_acc(x.reshape(T * B, H, W, 128), q).reshape(T, B, H, W, 128)
  assert (acc[0, 11, 17:23, 17:23, SAT] == TIE_ACC_T).all()
  return lay, bn, stt, x, acc, scale, bias


TIE_SUM_T = 29361                      # 127 * 9 * 29361 = 33559623 = 3 mod 4: in [2^25, 2^26) fp32 rounds it up by 1
TIE_ACC_T = 127 * 9 * TIE_SUM_T
COUNT_DENSE = (5, 40, 1024, 110)       # (T, B, K, N)
TIE_SUM_D = 132105                     # 127 * 132105 = 16777335 = 3 mod 4: in [2^24, 2^25) the tie rounds up to even
TIE_ACC_D = 127 * TIE_SUM_D


@functools.lru_cache(maxsize=None)
def count_dense_data():
  T, B, K, N = COUNT_DENSE
  rng = np.random.default_rng(502)
  lay, _, scale, bias = dense_binary_layer(rng, K, N)
  saturate_channels(lay, scale, bias)
  q = ref_int.duq_levels_c(lay["kernel"], lay["prune_0"]["mask"], lay["DuQ_0"]["a"][0], 8)
  assert (q[:, SAT] == 127).all()
  x = np.minimum(rng.poisson(1.0, size=(T, B, K)), 255).astype(np.uint8)
  x[0, 0] = 255; x[2, 5] = 255; x[-1, -1, ::2] = 255
  x[1, 9] = rng.integers(128, 256, size=K)
  x[:, 10:20] = rng.integers(128, 256, size=(T, 10, K))
  # rows summing to TIE_SUM_D: the SAT channels see acc = TIE_ACC_D exactly; channel SAT.start (scale 2^-24 here, so
  # that the ulp of float(acc) is one ulp of v below 2) fires at the threshold on their step only when it rounds up
  x[0, 20:30] = bytes_summing_to(rng, 10, TIE_SUM_D, K)
  scale[SAT.start] = F32(2.0 ** -24)
  bias[SAT.start] = tie_bias(F32(TIE_ACC_D), scale[SAT.start])
  acc = ref_int.dense_acc(x, q)
  assert (acc[0, 20:30, SAT] == TIE_ACC_D).all()
  return lay, x, acc, scale, bias


def check_conversion_matters(acc, scale, bias, min_u, min_s, pool=False):
  """The outputs depend on rounding float(acc) to nearest: rounding toward zero instead changes u_T of the SAT
  channels at >= min_u neurons and their spikes at >= min_s neuron-steps (pooled spikes and counts too, for the conv
  case, which is all its production epilogue emits).  Also: the spike rate is inside (0.02, 0.9)."""
  s, u = ref_int.lif_from_acc(acc, scale, bias)
  assert 0.02 < s.mean() < 0.9
  s_rz, u_rz = ref_int.lif_from_acc(round_toward_zero(acc), scale, bias)
  du = int((u[..., SAT].view(np.uint32) != u_rz[..., SAT].view(np.uint32)).sum())
  ds = int((s != s_rz).sum())
  assert du >= min_u and ds >= min_s, (du, ds)
  if pool:
    assert int((ref_int.maxpool2_u8(s) != ref_int.maxpool2_u8(s_rz)).sum()) >= min_s // 4
    assert not np.array_equal(counts_of(s), counts_of(s_rz))


def test_count_inputs_reach_rounding_accumulators(oracle_lib):
  """Oracle side of the count-valued cases: bytes >= 128 occur, the SAT channels' |acc| passes 2^24 where the
  int32 -> fp32 conversion rounds, and their u_T depends on that rounding (a truncating conversion changes it), for
  the tile case and the dense case."""
  _, _, _, x, acc, scale, bias = count_tile_data()
  assert (x >= 128).sum() > 10000 and np.abs(acc).max() > 3.7e7 > 2 ** 24
  assert (np.abs(acc[..., SAT]) > 2 ** 24).sum() >= 512
  check_conversion_matters(acc, scale, bias, 128, 36, pool=True)
  _, x, acc, scale, bias = count_dense_data()
  assert (x >= 128).sum() > 1000 and np.abs(acc).max() > 3.3e7 > 2 ** 24
  assert (np.abs(acc[..., SAT]) > 2 ** 24).sum() >= 256
  check_conversion_matters(acc, scale, bias, 8, 10)


@gpu
def test_count_inputs_bit_exact(cuda_lib, oracle_lib):
  """u8 counts 0..255 (Poisson, saturated patches, bytes >= 128) into k_conv3x3_tile -- instrumented, and the
  production epilogue (pool, spike counts; u8 and bit-packed output) -- and the SIMT conv; into k_dense_umma<1> and
  the SIMT dense.  Accumulators up to 3.7e7 > 2^24, where the SAT channels' u_T depends on the int32 -> fp32 conversion
  rounding to nearest like (float)acc (test_count_inputs_reach_rounding_accumulators).  Everything bit-exact against
  ref_int."""
  lay, bn, stt, x, acc_ref, scale, bias = count_tile_data()
  T, B, H, W = COUNT_TILE_SHAPE
  s_un, u_ref = ref_int.lif_from_acc(acc_ref, scale, bias)
  s_pool, cnt_ref = ref_int.maxpool2_u8(s_un), counts_of(s_un)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  packed.scale.copy_(dev(scale)); packed.bias.copy_(dev(bias))
  cnt = torch.zeros((B, T, 128), device=DEV, dtype=torch.int32)
  for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
    for bm in (True, False):
      run = lambda pool, **kw: run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, pool, impl,
                                        batch_major=bm, **kw)
      cnt.zero_()
      s, u, acc = run(False, counts=cnt)
      bad = diffs(acc=(acc, acc_ref), spikes=(s, s_un), u_final=(u, u_ref), counts=(cnt.cpu().numpy(), cnt_ref))
      assert not bad, (impl, bm, "instrumented", bad)
      cnt.zero_()
      s, _, _ = run(True, counts=cnt, dumps=False)
      bad = diffs(spikes=(s, s_pool), counts=(cnt.cpu().numpy(), cnt_ref))
      assert not bad, (impl, bm, "production", bad)
      if impl == _lib.IMPL_TCGEN05:
        s, _, _ = run(True, dumps=False, y_bits=True)
        assert np.array_equal(s, s_pool), (bm, "production, bit-packed output")
  lay, x, acc_ref, scale, bias = count_dense_data()
  s_ref, u_ref = ref_int.lif_from_acc(acc_ref, scale, bias)
  packed = pk_mod.pack_dense(lay, 8, DEV)
  packed.scale.copy_(dev(scale)); packed.bias.copy_(dev(bias))
  for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
    s, u, acc = run_dense(cuda_lib, x, packed.wq, packed.scale, packed.bias, COUNT_DENSE[3], impl=impl)
    bad = diffs(acc=(acc, acc_ref), spikes=(s, s_ref), u_final=(u, u_ref))
    assert not bad, (impl, "dense", bad)
