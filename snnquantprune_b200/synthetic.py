"""Synthetic TCJA-SNN parameters and event frames (host-side numpy, no device
work).

There is no dataset and no checkpoint in this environment (BASELINE.md section
1), so benchmarks and tests run on random-init weights of the reference
architecture and synthetic event-count frames (SURVEY.md section 8d):

* kernels ~ N(0, gain^2 / fan_in)  (the layers' default ``lecun_normal`` scale,
  /root/reference/flax_qconv.py:86, flax_qdense.py:51; ``gain`` > 1 on the
  BatchNorm-free layers so that they actually fire);
* DuQ ``a = c = gaussian_init(kernel)``
  (/root/reference/examples/train_inpt_spikingjelly.py:159-172);
* ``prune_0/mask`` from global (or local) magnitude pruning (same file,
  147-223);
* BatchNorm gamma/beta/mean/var drawn around fixed per-layer constants chosen
  so that every block fires at a healthy rate (a dead network would make parity
  checks vacuous);
* frames: uint8 event counts ``min(Poisson(0.15), 15)``, layout (B,T,H,W,2)
  (/root/reference/examples/train_inpt_spikingjelly.py:300-305).

The variable tree mirrors the reference's Flax tree (names ``QuantConv_0..8``,
``QuantDense_0..1``, ``BatchNorm_0..4``;
/root/reference/examples/tcja/tcja_load_pretrained_weights.py:19-36).
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict

import numpy as np

from . import quant as hq

F32 = np.float32

# Gains bring every kernel to a comparable magnitude (std ~0.15-0.3) so that
# GLOBAL magnitude pruning removes a similar share of every layer instead of
# wiping out the 3x3x128x128 kernels (whose lecun std is 0.03); BatchNorm makes
# the conv gains irrelevant to the function, the BN-free layers need > 1 to fire.
_GAIN = {"QuantConv_1": 7.0, "QuantConv_2": 7.0, "QuantConv_3": 7.0, "QuantConv_6": 7.0,
         "QuantDense_0": 7.0, "QuantDense_1": 5.0,
         "QuantConv_4": 3.0, "QuantConv_5": 6.0,
         "QuantConv_7": 3.0, "QuantConv_8": 6.0}
# assumed second moment E[x^2] of each conv block's input (counts, then spike
# rates, then att^2 * rate), used to centre the synthetic running variance
_IN_M2 = (0.1725, 0.27, 0.36, 0.32, 0.06)
_CONV_NAMES = ("QuantConv_0", "QuantConv_1", "QuantConv_2", "QuantConv_3", "QuantConv_6")


class StableRNG:
  """Counter-based generator built from integer arithmetic only (splitmix64 over
  a running counter), so its streams are identical on every numpy / libm:
  fixtures keyed on it can FAIL (not skip) on a digest mismatch.  `uniform`
  is exact 53-bit; `standard_normal` is Irwin-Hall(4) of 16-bit lanes (unit
  variance, support +-3.46 sigma) -- enough for synthetic weights; `poisson15`
  inverts a fixed 4-entry CDF table of Poisson(0.15) (counts >= 4, P = 2e-5,
  are reported as 4)."""

  def __init__(self, seed: int):
    self.ctr = np.uint64((int(seed) * 0x9E3779B97F4A7C15 + 0x632BE59BD9B4E019) & 0xFFFFFFFFFFFFFFFF)

  def _u64(self, n: int) -> np.ndarray:
    with np.errstate(over="ignore"):
      z = self.ctr + (np.arange(1, n + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15))
      self.ctr = z[-1] if n else self.ctr
      z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
      z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
      return z ^ (z >> np.uint64(31))

  def uniform(self, lo=0.0, hi=1.0, size=()) -> np.ndarray:
    n = int(np.prod(size)) if size != () else 1
    u = (self._u64(n) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    return (lo + (hi - lo) * u).reshape(size)

  def standard_normal(self, size=()) -> np.ndarray:
    n = int(np.prod(size)) if size != () else 1
    z = self._u64(n)
    s = np.zeros(n, np.int64)
    for k in range(4):
      s += ((z >> np.uint64(16 * k)) & np.uint64(0xFFFF)).astype(np.int64)
    # sum of four U{0..65535}: mean 131070, variance 4 * (65536^2 - 1) / 12
    return ((s - 131070).astype(np.float64) / 37837.22713327866).reshape(size)

  def poisson15(self, size=()) -> np.ndarray:
    n = int(np.prod(size)) if size != () else 1
    r = self._u64(n) >> np.uint64(11)                     # 53-bit
    # floor(CDF_Poisson(0.15)(k) * 2^53), k = 0..3
    t = np.array([7752568243805408, 8915453480376219, 9002669873119030, 9007030692756171], np.uint64)
    k = (r >= t[0]).astype(np.uint8) + (r >= t[1]) + (r >= t[2]) + (r >= t[3])
    return k.astype(np.uint8).reshape(size)

  def integers(self, lo: int, hi: int, size=()) -> np.ndarray:
    n = int(np.prod(size)) if size != () else 1
    return (lo + (self._u64(n) >> np.uint64(33)).astype(np.int64) % (hi - lo)).reshape(size)


def _effective_energy(kernel, a, mask, bits):
  """sum_k w_eff[k, n]^2 per output channel of the quantized + masked kernel
  (synthetic-statistics helper only; the product quantizes on the device)."""
  L = F32(2 ** (bits - 1) - 1)
  q = np.round(np.clip(kernel / F32(a), -1, 1) * L) / L * F32(a) * mask
  return np.sum(q.reshape(-1, q.shape[-1]).astype(np.float64) ** 2, axis=0)


def kernel_shapes(T: int, channels: int, num_classes: int, H: int
                  ) -> "OrderedDict[str, tuple]":
  """Kernel shapes of CextNet in param-tree order
  (/root/reference/examples/tcja/models.py:111-246; HWIO / (in,out))."""
  C = channels
  side = H // 32
  return OrderedDict([
      ("QuantConv_0", (3, 3, 2, C)),
      ("QuantConv_1", (3, 3, C, C)),
      ("QuantConv_2", (3, 3, C, C)),
      ("QuantConv_3", (3, 3, C, C)),
      ("QuantConv_4", (4, T, T)),       # TCJA-0 conv_t (features = T)
      ("QuantConv_5", (4, C, C)),       # TCJA-0 conv_c
      ("QuantConv_6", (3, 3, C, C)),
      ("QuantConv_7", (4, T, T)),
      ("QuantConv_8", (4, C, C)),
      ("QuantDense_0", (C * side * side, C * 2 * 2)),
      ("QuantDense_1", (C * 2 * 2, num_classes * 10)),
  ])


def make_variables(bits: int = 8, prune_percentage: float = 0.5, T: int = 20,
                   channels: int = 128, num_classes: int = 11, H: int = 128,
                   seed: int = 1, prune_global: bool = True, stable: bool = False) -> Dict:
  """``stable=True`` draws from :class:`StableRNG` (version-independent streams; used by
  the from-reference fixtures), otherwise from ``np.random.default_rng``."""
  rng = StableRNG(seed) if stable else np.random.default_rng(seed)
  shapes = kernel_shapes(T, channels, num_classes, H)
  kernels = OrderedDict()
  for name, shp in shapes.items():
    fan_in = int(np.prod(shp[:-1]))
    g = _GAIN.get(name, 1.0)
    kernels[name] = (rng.standard_normal(shp) * (g / np.sqrt(fan_in))).astype(F32)

  if prune_percentage > 0:
    if prune_global:
      masks = hq.global_masks(kernels, prune_percentage)
    else:
      masks = OrderedDict((n, hq.local_mask(k, prune_percentage))
                          for n, k in kernels.items())
  else:
    masks = OrderedDict((n, np.ones(k.shape, F32)) for n, k in kernels.items())

  params = OrderedDict()
  for name, k in kernels.items():
    ac = hq.gaussian_init(k, bits=bits, sign=True)
    params[name] = {"kernel": k,
                    "DuQ_0": {"a": np.array([ac], F32), "c": np.array([ac], F32)},
                    "prune_0": {"mask": masks[name].astype(F32)}}
  stats = OrderedDict()
  for i in range(5):
    C = channels
    lay = params[_CONV_NAMES[i]]
    energy = _effective_energy(lay["kernel"], lay["DuQ_0"]["a"][0], lay["prune_0"]["mask"], bits)
    var = np.maximum(_IN_M2[i] * energy, 1e-6) * rng.uniform(0.8, 1.25, (C,))
    params[f"BatchNorm_{i}"] = {
        "scale": rng.uniform(0.8, 1.2, (C,)).astype(F32),
        "bias": (0.5 + 0.1 * rng.standard_normal((C,))).astype(F32)}
    stats[f"BatchNorm_{i}"] = {
        "mean": (0.05 * np.sqrt(var) * rng.standard_normal((C,))).astype(F32),
        "var": var.astype(F32)}
  return {"params": params, "batch_stats": stats}


def make_frames(B: int, T: int = 20, H: int = 128, W: int = 128, seed: int = 0,
                rate: float = 0.15, stable: bool = False) -> np.ndarray:
  """uint8 event-count frames (B,T,H,W,2)."""
  if stable:
    assert rate == 0.15
    return StableRNG(seed).poisson15((B, T, H, W, 2))
  rng = np.random.default_rng(seed)
  return np.minimum(rng.poisson(rate, size=(B, T, H, W, 2)), 15).astype(np.uint8)


def make_events(B: int, T: int = 20, H: int = 128, seed: int = 0, rate: float = 0.15):
  """Synthetic event recordings: a list of B int32 (N_b, 3) (x, y, p) arrays, x, y uniform on the H x H sensor, p
  uniform in {0, 1}.  N_b is uniform within +-25 % of ``rate * T * H * H * 2`` (so each cell of the T frames gets
  about ``rate`` events, as in :func:`make_frames`), so sizes vary and N_b % T is mostly non-zero.  Drawn from
  :class:`StableRNG`: identical on every numpy."""
  rng = StableRNG(seed)
  mean = int(round(rate * T * H * H * 2))
  spread = mean // 4
  sizes = rng.integers(mean - spread, mean + spread + 1, (B,))
  out = []
  for n in sizes:
    n = int(n)
    xy = rng.integers(0, H, (n, 2))
    p = rng.integers(0, 2, (n, 1))
    out.append(np.concatenate([xy, p], 1).astype(np.int32))
  return out


def make_labels(B: int, num_classes: int = 11, seed: int = 3) -> np.ndarray:
  return np.random.default_rng(seed).integers(0, num_classes, size=(B,)).astype(np.int32)


def make_frames_blob(B: int, T: int = 20, H: int = 128, W: int = 128, seed: int = 0, radius: float = 18.0,
                     rate: float = 0.6) -> np.ndarray:
  """Spatially structured synthetic DVS frames (B,T,H,W,2): a blob of activity (a moving hand, say) drifts across an
  otherwise silent sensor -- the structure real recordings have and i.i.d. frames lack.  Inside the blob (soft disc
  of ``radius`` pixels) counts are Poisson-like with mean ``rate``; everywhere else exactly zero, so most strips of
  every layer see all-zero input boxes (the spike-tile skip path)."""
  rng = StableRNG(seed)
  yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
  out = np.zeros((B, T, H, W, 2), np.uint8)
  for b in range(B):
    p0 = rng.uniform(0.2, 0.8, (2,)) * np.array([H, W])
    vel = (rng.uniform(-1.0, 1.0, (2,))) * np.array([H, W]) * 0.5 / max(T, 1)
    for t in range(T):
      cy, cx = p0 + vel * t
      inside = ((yy - cy) ** 2 + (xx - cx) ** 2) <= radius ** 2
      u = rng.uniform(0.0, 1.0, (H, W, 2))
      cnt = (u < rate * 0.6).astype(np.uint8) + (u < rate * 0.2) + (u < rate * 0.05)
      out[b, t] = cnt * inside[:, :, None]
  return out
