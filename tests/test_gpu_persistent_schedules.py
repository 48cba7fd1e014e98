"""The persistent tcgen05 kernels against the integer oracle at production work-item counts and skip patterns.

Every fused tcgen05 kernel runs min(items, #SMs) CTAs that loop over work items; the accumulator buffer and MMA issuer
(step & 1), the mbarrier phases, the input ring, the zacc skip flag, the slab list and the per-item zero carry of the
membranes all carry from one item to the next.  These tests give every CTA several items (a ragged last wave, odd and
even T), build bit-packed inputs whose all-zero boxes follow chosen per-(b, t, tile) patterns, reach the block-sparse
branches with structured masks, and feed the kernels BatchNorm statistics at their edges.  Every comparison is against
the C oracle (oracle/ref_int.py): bit-exact where the kernel's arithmetic is integer, otherwise under the bars of the
existing parity tests (pre-activation <= 1e-5 in membrane units, spike flips <= 1e-4).

A failing bit-exact comparison names the layer and the first differing (t, b, tile), the tile's work item, which item of
its CTA that is, and the accumulator buffer / MMA issuer of the step."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ref_int, ref_quant
from snnquantprune_b200 import _lib
from snnquantprune_b200 import pack as pk_mod
from test_gpu_parity import DEV, F32, make_layer, preact_err, run_conv, run_dense

gpu = pytest.mark.gpu
TILE_H, TILE_W = 16, 8            # output tile of k_conv3x3_tile: one work item per (b, tile) for all T steps


# ------------------------------------------------------------------ helpers ----
def sm_count():
  return torch.cuda.get_device_properties(0).multi_processor_count


def tile_rows(H):
  return -(-H // TILE_H)            # the last tile row of an image may be partial


def tile_items(B, H, W):
  return B * tile_rows(H) * (W // TILE_W)


def box_empty(x):
  """Geometry model of the spike-tile skip: x (T,B,H,W,C) -> bool (T,B,ceil(H/16),W/8), True where the input box of
  the tile is all zero.  Tile (ty, tx) reads rows 16ty-1 .. 16ty+16 and columns 8tx-1 .. 8tx+8, clipped at the image."""
  T, B, H, W, _ = x.shape
  nz = np.zeros((T, B, H + 2, W + 2), bool)
  nz[:, :, 1:-1, 1:-1] = x.any(axis=-1)
  out = np.empty((T, B, tile_rows(H), W // TILE_W), bool)
  for ty in range(tile_rows(H)):
    for tx in range(W // TILE_W):
      out[:, :, ty, tx] = ~nz[:, :, TILE_H * ty:TILE_H * ty + TILE_H + 2, TILE_W * tx:TILE_W * tx + TILE_W + 2].any(axis=(2, 3))
  return out


def where_differs(layer, got, want, tile, tiles_x, tiles_per_img, T, B):
  """Empty string if got == want, else which (t, b, tile) differ and where those steps sit in the persistent schedule.
  got / want: (T, B, rows, cols, C) or (B, rows, cols, C) (final membranes); tile = (rows, cols) of a tile in them."""
  if np.array_equal(got, want):
    return ""
  d = got != want
  if d.ndim == 4:
    d = d[None]
  pos = np.argwhere(d.any(axis=-1))
  grid = min(B * tiles_per_img, sm_count())
  lines = [f"{layer}: {len(pos)} positions differ (grid {grid} CTAs, {B * tiles_per_img} items, T = {T})"]
  for t, b, h, w in pos[:6]:
    ty, tx = h // tile[0], w // tile[1]
    item = b * tiles_per_img + ty * tiles_x + tx
    nth = item // grid
    if got.ndim == 5:
      step = nth * T + t
      lines.append(f"  t={t} b={b} tile=({ty},{tx}) item={item}: item {nth} of CTA {item % grid}, CTA step {step}, "
                   f"buffer / issuer {step & 1}")
    else:
      lines.append(f"  final membrane b={b} tile=({ty},{tx}) item={item}: item {nth} of CTA {item % grid}")
  return "\n".join(lines)


def tile_check(layer, got, want, H, W, T, B, pooled):
  tiles_x = W // TILE_W
  tile = (TILE_H // 2, TILE_W // 2) if pooled else (TILE_H, TILE_W)
  msg = where_differs(layer, got, want, tile, tiles_x, tiles_x * tile_rows(H), T, B)
  assert not msg, msg


def skip_stats(lib, reset):
  sk, tot = ctypes.c_int64(0), ctypes.c_int64(0)
  _lib.check(lib.snnqp_tile_skip_stats(ctypes.byref(sk), ctypes.byref(tot), int(reset)))
  return sk.value, tot.value


def structured_mask(lay, rng, keep_slabs):
  """Zero all but `keep_slabs` of the 36 K-slabs (tap x 32 input channels x all outputs) of a 128 -> 128 layer."""
  keep = np.zeros(36, bool)
  keep[rng.permutation(36)[:keep_slabs]] = True
  mask = lay["prune_0"]["mask"].reshape(9, 4, 32, 128).copy()
  mask[~keep.reshape(9, 4)] = 0
  lay["prune_0"]["mask"] = mask.reshape(3, 3, 128, 128)
  return ref_int.duq_levels_c(lay["kernel"], lay["prune_0"]["mask"], lay["DuQ_0"]["a"][0], 8)


# ------------------------------------------- 1. k_conv3x3_tile, multi-wave ----
@gpu
@pytest.mark.parametrize("T,B,H,W", [(3, 5, 64, 64), (5, 19, 32, 32), (2, 20, 64, 64), (1, 150, 16, 16),
                                     (3, 40, 24, 32), (2, 30, 18, 64)])
def test_tile_conv_multi_wave_bit_exact(cuda_lib, oracle_lib, T, B, H, W):
  """160 / 152 / 640 / 300 / 320 / 480 work items over the SMs (a ragged last wave; more than 4 items per CTA; T = 1,
  where every step starts a new item), odd and even T: accumulators, spikes, membranes, spike counts and y_popcount
  bit-exact, u8 and bit-packed input and output, both (t, b) stride orders.  H = 24 and 18 end in a partial tile row:
  whole epilogue warps (24) or the second row pair of a thread (18) fall below the image, and the channels raised by
  _skip_bias_layer fire there on the bias alone, so a phantom row leaking into any output or count fails."""
  items = tile_items(B, H, W)
  assert items > sm_count() and items % sm_count() != 0
  rng = np.random.default_rng(1000 * T + B)
  lay, q, bn, stt = _skip_bias_layer(rng, None)
  x = (rng.uniform(size=(T, B, H, W, 128)) < 0.25).astype(np.uint8)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  assert 0.02 < info["spikes"].mean() < 0.9
  cnt_ref = info["spikes"].sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2)
  pc_ref = s_ref.sum(axis=(2, 3, 4), dtype=np.int32).T                       # [B][T] pooled spikes
  run = lambda **kw: run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05, **kw)
  chk = lambda name, got, want, pooled=True: tile_check(name, got, want, H, W, T, B, pooled)
  for bm in (True, False):
    for xb in (False, True):
      tag = f"k_conv3x3_tile instrumented ({'b,t' if bm else 't,b'} order, {'bit-packed' if xb else 'u8'} input)"
      s, u, acc = run(batch_major=bm, x_bits=xb)
      chk(tag + " accumulators", acc, info["acc"], pooled=False)
      chk(tag + " spikes", s, s_ref)
      chk(tag + " final membranes", u, info["u"], pooled=False)
    cnt = torch.zeros((B, T, 128), device=DEV, dtype=torch.int32)
    s, _, _ = run(batch_major=bm, dumps=False, counts=cnt)
    chk("k_conv3x3_tile production u8 spikes", s, s_ref)
    assert np.array_equal(cnt.cpu().numpy(), cnt_ref), "production u8 spike counts"
    cnt.zero_()
    s, _, _ = run(batch_major=bm, dumps=False, counts=cnt, x_bits=True, y_bits=True)
    chk("k_conv3x3_tile production bit-packed spikes", s, s_ref)
    assert np.array_equal(cnt.cpu().numpy(), cnt_ref), "production bit-packed spike counts"
    pc = torch.zeros((B, T), device=DEV, dtype=torch.int32)
    s, _, _ = run(batch_major=bm, dumps=False, x_bits=True, y_bits=True, popcount=pc)
    chk("k_conv3x3_tile y_popcount variant spikes", s, s_ref)
    assert np.array_equal(pc.cpu().numpy(), pc_ref), "y_popcount != popcount of the oracle's pooled spikes"


# ------------------------------------------------- 2. spike-tile skip ----
def test_box_geometry_model_matches_oracle_conv(oracle_lib):
  """The skip model: a tile's input box is empty iff the oracle's 3x3 convolution with all-ones weights is zero on all
  128 outputs of the tile -- random sparse inputs and single spikes on every halo position, at image edges too."""
  rng = np.random.default_rng(5)
  T, B, H, W, C = 2, 6, 48, 40, 8
  x = (rng.uniform(size=(T, B, H, W, C)) < 1e-3).astype(np.uint8)
  for k, (r, c) in enumerate([(15, 7), (15, 12), (15, 16), (23, 7), (23, 16), (32, 7), (32, 12), (32, 16),
                              (0, 0), (H - 1, W - 1), (16, 8)]):
    x[k % T, k // T] = 0
    x[k % T, k // T, r, c, k % C] = 1
  acc = ref_int.conv3x3_acc(x.reshape(T * B, H, W, C), np.ones((3, 3, C, 1), np.int8)).reshape(T, B, H, W)
  quiet = ~acc.reshape(T, B, H // TILE_H, TILE_H, W // TILE_W, TILE_W).any(axis=(3, 5))
  model = box_empty(x)
  assert np.array_equal(model, quiet)
  assert 0.2 < model.mean() < 0.8                  # both verdicts well represented


def _skip_bias_layer(rng, keep_slabs):
  lay, q, bn, stt = make_layer(rng, 128, 128, 8, 0.5)
  bn["bias"][:8] += 3.0           # these channels fire on the bias alone every step, the next 8 every other step:
  bn["bias"][8:16] += 1.0         # a skipped step (acc = 0) still runs the LIF
  if keep_slabs is not None:
    q = structured_mask(lay, rng, keep_slabs)
  return lay, q, bn, stt


def _patterned_input(rng, T, B, H, W, empty_step, density=0.1):
  """Bernoulli spikes; whole images empty where empty_step(t) and, elsewhere, a quarter of the tiles' boxes zeroed."""
  x = rng.uniform(size=(T, B, H, W, 128)) < density
  for t in range(T):
    if empty_step(t):
      x[t] = False
      continue
    for b in range(B):
      for ty in range(H // TILE_H):
        for tx in range(W // TILE_W):
          if rng.uniform() < 0.25:
            x[t, b, max(TILE_H * ty - 1, 0):TILE_H * ty + TILE_H + 1, max(TILE_W * tx - 1, 0):TILE_W * tx + TILE_W + 1] = False
  return x.astype(np.uint8)


def _halo_input(rng, T, B):
  """48 x 24 images (3 x 3 tiles): at step t a single spike on halo position t % 8 of the centre tile (corners and edge
  midpoints of its box), nothing else -- the centre tile's interior is empty, its box is not."""
  H, W = 48, 24
  halo = [(15, 7), (15, 16), (32, 7), (32, 16), (15, 11), (32, 11), (23, 7), (23, 16)]
  x = np.zeros((T, B, H, W, 128), np.uint8)
  for t in range(T):
    for b in range(B):
      r, c = halo[(t + b) % 8]
      x[t, b, r, c, rng.integers(128)] = 1
  return x


SKIP_PATTERNS = {
    "all_empty": lambda t: True,
    "alternate": lambda t: t % 2 == 0,          # T even: one issuer always skips, the other never does
    "period3": lambda t: t % 3 == 0,            # both issuers mix skipped and computed steps on their buffer
    "first": lambda t: t == 0,
    "last": lambda t: t == 5,
    "halo": None,
}


@gpu
@pytest.mark.parametrize("slabs", [None, 10], ids=["dense_mma", "slab_list"])
@pytest.mark.parametrize("pattern", list(SKIP_PATTERNS))
def test_spike_tile_skip_patterns(cuda_lib, oracle_lib, pattern, slabs):
  """Bit-packed input with chosen all-zero boxes over 160+ work items: outputs bit-exact, and the kernel's skip counter
  (snnqp_tile_skip_stats) equals the geometry model's count of empty boxes exactly, both with the dense MMA sequence
  and with the block-sparse slab list (10 of 36 non-zero slabs)."""
  rng = np.random.default_rng(list(SKIP_PATTERNS).index(pattern) * 100 + (slabs or 0))
  lay, q, bn, stt = _skip_bias_layer(rng, slabs)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  nz = int(packed.slab_nz.cpu().numpy().astype(bool).sum())
  assert (nz == 36) if slabs is None else (0 < nz <= 12)
  if pattern == "halo":
    T, B, H, W = 8, 17, 48, 24
    x = _halo_input(rng, T, B)
  else:
    T, B, H, W = 6, 80, 16, 16
    x = _patterned_input(rng, T, B, H, W, SKIP_PATTERNS[pattern])
  assert tile_items(B, H, W) > sm_count()
  empty = box_empty(x)
  if pattern == "halo":
    assert not empty[:, :, 1, 1].any()            # the centre tile must be computed
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  if pattern == "all_empty":
    assert not info["acc"].any() and info["spikes"].any()     # acc = 0 everywhere, the LIF still fires on the bias
  run = lambda **kw: run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05,
                              x_bits=True, **kw)
  want_stats = (int(empty.sum()), empty.size)
  for bm in (True, False):
    skip_stats(cuda_lib, reset=True)
    s, u, acc = run(batch_major=bm)
    assert skip_stats(cuda_lib, reset=True) == want_stats, "instrumented variant: (skipped, total) != model"
    tile_check(f"k_conv3x3_tile skip[{pattern}] accumulators", acc, info["acc"], H, W, T, B, False)
    tile_check(f"k_conv3x3_tile skip[{pattern}] spikes", s, s_ref, H, W, T, B, True)
    tile_check(f"k_conv3x3_tile skip[{pattern}] final membranes", u, info["u"], H, W, T, B, False)
    cnt = torch.zeros((B, T, 128), device=DEV, dtype=torch.int32)
    s, _, _ = run(batch_major=bm, dumps=False, y_bits=True, counts=cnt)
    assert skip_stats(cuda_lib, reset=True) == want_stats, "production variant: (skipped, total) != model"
    tile_check(f"k_conv3x3_tile skip[{pattern}] production spikes", s, s_ref, H, W, T, B, True)
    assert np.array_equal(cnt.cpu().numpy(), info["spikes"].sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2))


# -------------------------------------------- 3. k_conv_att_umma (conv5) ----
def _att_check(lib, x, att, q, packed, scale, bias, pool, outside_envelope=()):
  """conv5 under the bars of the attention-weighted layers.  Channels in ``outside_envelope`` are left out of the
  pre-activation bar (only): the accumulator is fp32 (24-bit fixed-point attention, as documented in umma_att.cu), so a
  channel whose |scale| and |bias| are 2^16+ times the others' and cancel in v = acc * scale + bias carries that
  accumulator error, times |scale|, into v.  Their spikes, membranes and counts are still checked."""
  T, B = x.shape[:2]
  accf = ref_int.conv3x3_att_accf(x, att, q)
  s_ref, u_ref = ref_int.lif_from_acc(accf, scale, bias)
  cnt = torch.zeros((B, T, 128), device=DEV, dtype=torch.int32)
  s, u, acc = run_conv(lib, x, packed.wq, packed.scale, packed.bias, 128, pool, _lib.IMPL_TCGEN05, att=att,
                       batch_major=True, counts=cnt)
  ch = np.setdiff1d(np.arange(128), outside_envelope)
  assert preact_err(acc[..., ch], accf[..., ch], scale[ch], bias[ch]) <= 1e-5
  # given the kernel's own accumulators the epilogue (LIF, pool, counts) is bit-exact
  s2, u2 = ref_int.lif_from_acc(acc, scale, bias)
  msg = where_differs("k_conv_att_umma membranes", u, u2, (8, 8), 1, 1, T, B)
  assert not msg, msg
  msg = where_differs("k_conv_att_umma spikes", s, ref_int.maxpool2_u8(s2) if pool else s2, (4, 4) if pool else (8, 8),
                      1, 1, T, B)
  assert not msg, msg
  assert np.array_equal(cnt.cpu().numpy(), s2.sum(axis=(2, 3), dtype=np.int32).transpose(1, 0, 2))
  assert np.mean(s2 != s_ref) <= 1e-4
  same = (s2 == s_ref).all(axis=0)
  same[..., list(outside_envelope)] = False
  assert np.max((np.abs(u - u_ref) / np.maximum(np.abs(u_ref), 1.0))[same]) <= 1e-5
  return s2


@gpu
@pytest.mark.parametrize("B", [3, 300])
@pytest.mark.parametrize("removed", [0, 18, 27, 36])
def test_conv_att_multi_item_and_block_sparse(cuda_lib, oracle_lib, B, removed):
  """conv5 (W = H = 8, one work item per image) at T = 5: B = 300 gives two or three items per CTA and odd T moves
  every later item to the other accumulator buffer.  Structured masks removing 50 / 75 / 100 % of the 36 K-slabs take
  the kernel's block-sparse branch (the dense sequence needs all 36)."""
  T, H = 5, 8
  rng = np.random.default_rng(B + removed)
  lay, q, bn, stt = make_layer(rng, 128, 128, 8, 0.5)
  if removed:
    q = structured_mask(lay, rng, 36 - removed)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  nz = packed.slab_nz.cpu().numpy().astype(bool)
  assert nz.sum() == 36 - removed
  x = (rng.uniform(size=(T, B, H, H, 128)) < 0.3).astype(np.uint8)
  att = rng.uniform(0.0, 1.0, size=(T, B, 128)).astype(F32)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  s2 = _att_check(cuda_lib, x, att, q, packed, scale, bias, pool=(B == 300))
  if removed == 36:
    assert not q.any()                 # a fully pruned layer: acc = 0, the bias alone drives the LIF
  else:
    assert s2.any() and not s2.all()


# ------------------------------------------------------ 4. k_dense_umma ----
@gpu
def test_dense_more_column_tiles_than_sms(cuda_lib, oracle_lib):
  """T = 20 puts NB = 8 samples in a column tile: B = 1200 is 150 items for N = 128, so two CTAs take a second item
  and the weight prefetch crosses from one item to the next.  Binary input bit-exact, attention input under the bars
  of the attention-weighted layers."""
  T, B, K, N = 20, 1200, 2048, 128
  rng = np.random.default_rng(77)
  k = (rng.standard_normal((K, N)) * (5.0 / np.sqrt(K))).astype(F32)
  a = ref_quant.gaussian_init(k, 8)
  lay = {"kernel": k, "DuQ_0": {"a": np.array([a], F32), "c": np.array([a], F32)},
         "prune_0": {"mask": ref_quant.local_mask(k, 0.5)}}
  packed = pk_mod.pack_dense(lay, 8, DEV)
  q = ref_int.duq_levels_c(k, lay["prune_0"]["mask"], a, 8)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, n=N)
  x = (rng.uniform(size=(T, B, K)) < 0.2).astype(np.uint8)
  acc_ref = ref_int.dense_acc(x, q)
  s_ref, u_ref = ref_int.lif_from_acc(acc_ref, scale, bias)
  s, u, acc = run_dense(cuda_lib, x, packed.wq, packed.scale, packed.bias, N, impl=_lib.IMPL_TCGEN05)
  bad = np.argwhere((acc != acc_ref).any(axis=(0, 2)))[:, 0]
  assert bad.size == 0, f"k_dense_umma: samples {bad[:8].tolist()} differ (column tiles {sorted(set((bad // 8).tolist()))[:8]})"
  assert np.array_equal(s, s_ref) and np.array_equal(u, u_ref)
  assert 0.01 < s_ref.mean() < 0.9
  # attention-weighted input (dense1): att[t, b, k % 128]
  att = rng.uniform(0.05, 1, size=(T, B, 128)).astype(F32)
  accf = np.concatenate([ref_int.dense_att_accf(x[:, b:b + 200], np.tile(att[:, b:b + 200], (1, 1, K // 128)), q)
                         for b in range(0, B, 200)], axis=1)
  sf_ref, _ = ref_int.lif_from_acc(accf, scale, bias)
  s, u, acc = run_dense(cuda_lib, x, packed.wq, packed.scale, packed.bias, N, att=att, att_mod=128,
                        impl=_lib.IMPL_TCGEN05)
  assert preact_err(acc, accf, scale, bias) <= 1e-5
  assert np.mean(s != sf_ref) <= 1e-4
  s2, u2 = ref_int.lif_from_acc(acc, scale, bias)
  assert np.array_equal(s, s2) and np.array_equal(u, u2)


# ------------------------------------------- 5. BatchNorm statistics at their edges ----
def _edge_layer(rng, cin, outlier_log2=None):
  """make_layer plus the channels trained checkpoints contain: 0 all weights pruned with running var = mean = 0 (scale
  gamma * (c / L) / sqrt(eps), hundreds of times the others), 1 gamma = 0, 2 negative gamma, 3 a bias that always
  fires, 4 a bias that never fires; optionally 5 an outlier whose |scale| is 2^outlier_log2 times the others'."""
  lay, _, bn, stt = make_layer(rng, cin, 128, 8, 0.3)
  mask = lay["prune_0"]["mask"].copy()
  mask[..., 0] = 0
  lay["prune_0"]["mask"] = mask
  stt["var"][0] = 0.0
  stt["mean"][0] = 0.0
  bn["scale"][1] = 0.0
  bn["scale"][2] = -bn["scale"][2]
  bn["bias"][3] = 40.0
  bn["bias"][4] = -40.0
  if outlier_log2 is not None:
    bn["scale"][5] *= F32(2.0 ** outlier_log2)
  q = ref_int.duq_levels_c(lay["kernel"], mask, lay["DuQ_0"]["a"][0], 8)
  assert not q[..., 0].any() and q[..., 5].any()
  return lay, q, bn, stt


@gpu
def test_fold_affine_bn_edges_bit_exact(cuda_lib):
  """snnqp_fold_affine with var = 0, gamma = 0, negative gamma, huge |gamma|: bit-exact against ref_int.fold_affine."""
  rng = np.random.default_rng(12)
  for log2 in (None, 16, 20):
    lay, _, bn, stt = _edge_layer(rng, 128, log2)
    for bits in (2, 4, 8):
      s_ref, b_ref = ref_int.fold_affine(lay["DuQ_0"]["c"], bits, bn, stt, 128)
      s, b = pk_mod.fold_affine(lay["DuQ_0"]["c"], bits, 128, DEV, bn, stt)
      assert np.array_equal(s.cpu().numpy(), s_ref) and np.array_equal(b.cpu().numpy(), b_ref), (log2, bits)
      assert s_ref[1] == 0 and s_ref[2] < 0


EDGE_CASES = pytest.mark.parametrize("outlier_log2", [None, 16, 20], ids=["trained_edges", "outlier_2e16", "outlier_2e20"])


def _edge_case(outlier_log2, cin):
  rng = np.random.default_rng((21 if outlier_log2 is None else outlier_log2) + cin)
  lay, q, bn, stt = _edge_layer(rng, cin, outlier_log2)
  packed = pk_mod.pack_conv3x3(lay, 8, DEV, bn, stt)
  scale, bias = ref_int.fold_affine(lay["DuQ_0"]["c"], 8, bn, stt, 128)
  if outlier_log2 is None:
    assert abs(scale[0]) > 100 * np.median(np.abs(scale[6:]))      # the all-pruned, var = 0 channel
  return rng, q, packed, scale, bias


@gpu
@EDGE_CASES
def test_bn_edges_tile_kernel(cuda_lib, oracle_lib, outlier_log2):
  """The edge channels through the 3x3 tile kernel (conv2-4): integer accumulators, so bit-exact whatever the scales."""
  rng, q, packed, scale, bias = _edge_case(outlier_log2, 128)
  T, B, H = 3, 3, 32
  x = (rng.uniform(size=(T, B, H, H, 128)) < 0.25).astype(np.uint8)
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  assert info["spikes"][..., 3].all() and not info["spikes"][..., 4].any()
  for xb in (False, True):
    s, u, acc = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05, x_bits=xb)
    assert np.array_equal(acc, info["acc"]) and np.array_equal(s, s_ref) and np.array_equal(u, info["u"]), xb
  s, _, _ = run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05, dumps=False,
                     x_bits=True, y_bits=True)
  assert np.array_equal(s, s_ref)


@gpu
@EDGE_CASES
def test_bn_edges_conv5(cuda_lib, oracle_lib, outlier_log2):
  """The edge channels through k_conv_att_umma under the attention-weighted bars; the stress outlier channel's
  pre-activation is outside the fp32 accumulator's envelope (see _att_check)."""
  rng, q, packed, scale, bias = _edge_case(outlier_log2, 128)
  x = (rng.uniform(size=(4, 3, 8, 8, 128)) < 0.3).astype(np.uint8)
  att = rng.uniform(0.0, 1.0, size=(4, 3, 128)).astype(F32)
  _att_check(cuda_lib, x, att, q, packed, scale, bias, pool=True, outside_envelope=() if outlier_log2 is None else (5,))


@gpu
@EDGE_CASES
def test_bn_edges_conv1(cuda_lib, oracle_lib, outlier_log2):
  """The edge channels through conv1 (Cin = 2, event counts up to 255): the reference-order LIF bit-exact, LIF_FAST
  within the flip budget and the float64 rounding band, LIF_TENSOR within the flip budget and the band (spikes and
  membranes, tests/test_gpu_conv1_rounding_band.py).  LIF_TENSOR scales its whole membrane domain by one power of two
  fitted to the largest channel, so an outlier channel costs every other channel precision: with the all-pruned
  var = 0 channel (~100x the others) the membranes also meet 1e-5; with a 2^16 / 2^20 stress outlier the band, which
  charges the fp16 pieces' subnormal floor, is what bounds them (include/snnqp.h)."""
  from test_gpu_conv1_rounding_band import check_band, conv1_band
  rng, q, packed, scale, bias = _edge_case(outlier_log2, 2)
  x = np.minimum(rng.poisson(0.3, size=(6, 4, 32, 128, 2)), 255).astype(np.uint8)
  x[0, 0, 0, 0, :] = 255
  x[-1, -1, -1, -1, :] = 200
  s_ref, info = ref_int.spiking_conv3x3(x, q, scale, bias, pool=True, want=True)
  band = conv1_band(x, q, scale, bias, modes=("fast", "tensor"))
  run1 = lambda **kw: run_conv(cuda_lib, x, packed.wq, packed.scale, packed.bias, 128, True, _lib.IMPL_TCGEN05, **kw)
  s, u, acc = run1(lif_mode=_lib.LIF_EXACT)
  assert np.array_equal(acc, info["acc"]) and np.array_equal(s, s_ref) and np.array_equal(u, info["u"])
  fails = []
  for yb in (False, True):
    s, _, _ = run1(dumps=False, y_bits=yb, lif_mode=_lib.LIF_EXACT)
    if not np.array_equal(s, s_ref):
      fails.append(("LIF_EXACT production", yb, int((s != s_ref).sum())))
    s, _, _ = run1(dumps=False, y_bits=yb, lif_mode=_lib.LIF_FAST)
    if np.mean(s != s_ref) > 1e-4:
      fails.append(("LIF_FAST flips", yb, int((s != s_ref).sum())))
    check_band(band, "fast", s, None, ("LIF_FAST", yb))
    s, u, _ = run1(dumps="u", y_bits=yb, lif_mode=_lib.LIF_TENSOR)
    print("\nLIF_TENSOR", outlier_log2, yb, check_band(band, "tensor", s, u, ("LIF_TENSOR", yb)),
          "max rel membrane error", float(np.max(np.abs(u - info["u"]) / np.maximum(1.0, np.abs(info["u"])))))
    flips = int((s != s_ref).sum())
    rel = np.abs(u - info["u"]) / np.maximum(1.0, np.abs(info["u"]))
    bad = rel > 1e-5
    if flips > 1e-4 * s_ref.size or (outlier_log2 is None and bad.sum() > 4 + 4 * flips):
      fails.append(("LIF_TENSOR", yb, flips, int(bad.sum()), np.unique(np.argwhere(bad)[:, -1]).tolist()[:16],
                    float(rel.max())))
  assert not fails, fails
