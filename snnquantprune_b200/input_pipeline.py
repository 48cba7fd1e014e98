"""Event -> frame integration in front of the hot path, with the reference's
entry-point name and argument meaning
(/root/reference/examples/input_pipeline.py:142-219 ``preprocess_data_number``;
``split_by == "number"`` only -- the reference raises NotImplementedError for
"time" too), on the GPU: the frames are produced directly in HBM in the hot
path's input layout (B,T,H,W,2) uint8, so real event streams never touch a CPU
histogram.  No CPU fallback.

Three host -> device wire formats feed the end-to-end host calls of
``CextNetEngine``: dense uint8 frames (``forward_host``), zero-suppressed frames
(``ZsfBatch``, ``forward_host_zsf``) and packed event words (``EventBatch``,
``forward_host_events``): the recordings as the reference's loader holds them,
one 16- or 32-bit word per event, integrated into frames on the GPU chunk by
chunk."""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib


def concat_events(samples: Sequence[np.ndarray]) -> Tuple[torch.Tensor, torch.Tensor]:
  """Host side of a ragged batch: list of (N_b, 3) integer (x, y, p) arrays in time order ->
  (pinned int32 [N_total, 3], pinned int64 [B+1] offsets)."""
  sizes = [int(np.shape(a)[0]) for a in samples]
  offsets = torch.zeros(len(samples) + 1, dtype=torch.int64)
  offsets[1:] = torch.as_tensor(np.cumsum(sizes))
  flat = np.concatenate([np.asarray(a).reshape(-1, 3) for a in samples], 0).astype(np.int32, copy=False) \
      if sum(sizes) else np.zeros((0, 3), np.int32)
  addrs = torch.as_tensor(np.ascontiguousarray(flat))
  if torch.cuda.is_available():
    addrs, offsets = addrs.pin_memory(), offsets.pin_memory()
  return addrs, offsets


def events_to_frames(addrs: torch.Tensor, offsets: torch.Tensor, num_frames: int, wh: int,
                     resolution_scale: int = 1, exact_int32: bool = False,
                     out: Optional[torch.Tensor] = None, max_events_per_sample: int = 0
                     ) -> Tuple[torch.Tensor, torch.Tensor]:
  """Device tensors in, device frames out: (B, T, wh', wh', 2) uint8 (saturating at 255) or int32.
  Returns (frames, n_saturated) with n_saturated a device int64 scalar (no host sync).
  ``max_events_per_sample``: the largest sample size if the caller knows it (``concat_events`` does);
  lets the kernel use 16-bit shared-memory counters (3x the frames in flight), same results."""
  if int(resolution_scale) != resolution_scale or resolution_scale < 1:
    raise NotImplementedError("resolution_scale must be a positive integer")
  if addrs.dtype != torch.int32 or offsets.dtype != torch.int64:
    raise ValueError("addrs must be int32 (N,3) and offsets int64 (B+1,)")
  B = offsets.numel() - 1
  whs = int(wh // resolution_scale)
  dt = torch.int32 if exact_int32 else torch.uint8
  if out is None:
    out = torch.empty((B, num_frames, whs, whs, 2), device=addrs.device, dtype=dt)
  sat = torch.zeros((), device=addrs.device, dtype=torch.int64)
  if B == 0:
    return out, sat
  _lib.check(_lib.lib().snnqp_events_to_frames(_lib.ptr(addrs), _lib.ptr(offsets), B, num_frames, int(wh),
                                               int(resolution_scale), int(max_events_per_sample), _lib.ptr(out),
                                               1 if exact_int32 else 0,
                                               _lib.ptr(sat), _lib.stream()))
  return out, sat


def preprocess_data_number(addrs, times, config, wh, device="cuda") -> torch.Tensor:
  """One sample, reference signature: addrs (N,3) (x,y,p), ``times`` unused by the
  number split (as in the reference), config.num_frames / config.resolution_scale /
  config.split_by.  Returns (T, wh', wh', 2) uint8 on ``device``."""
  if getattr(config, "split_by", "number") != "number":
    raise NotImplementedError
  a, off = concat_events([np.asarray(addrs)])
  fr, _ = events_to_frames(a.to(device, non_blocking=True), off.to(device, non_blocking=True),
                           int(config.num_frames), int(wh), int(getattr(config, "resolution_scale", 1)),
                           max_events_per_sample=int(a.shape[0]))
  return fr[0]


def density_stats(x: torch.Tensor, n_slices: int, bits: bool = False) -> dict:
  """The densities the reference sows per layer (examples/tcja/models.py:128-142): ``x`` is a
  contiguous uint8 device tensor whose leading ``n_slices`` = T*B (or B*T) slices are the
  (t, b) units.  Returns device tensors {"counts" int32 [n_slices], "min", "mean"} ('_min' is
  the max density, as in the reference's naming).  ``bits``: ``x`` is bit-packed spikes
  (SNNQP_SPIKES_BITS): set bits over 8 * bytes."""
  if x.dtype != torch.uint8 or not x.is_contiguous():
    raise ValueError("density_stats takes a contiguous uint8 tensor")
  slice_bytes = x.numel() // n_slices
  counts = torch.empty(n_slices, device=x.device, dtype=torch.int32)
  fn = _lib.lib().snnqp_slice_popcount if bits else _lib.lib().snnqp_slice_nonzeros
  _lib.check(fn(_lib.ptr(x), n_slices, slice_bytes, slice_bytes, _lib.ptr(counts), _lib.stream()))
  frac = counts.to(torch.float64) / float(slice_bytes * (8 if bits else 1))
  return {"counts": counts, "min": frac.max(), "mean": frac.mean()}


# ---- zero-suppressed frames: the host -> device wire format of the end-to-end path --------------------------
class ZsfBatch:
  """A batch of uint8 event-count frames (B, T, H, W, 2) in the zero-suppressed wire format of
  ``snnqp_expand_frames_zsf`` (include/snnqp.h): cell bitmap + running offsets per 1024-cell block + the non-zero
  counts (4 or 8 bits each).  Every sample's value stream starts on a 16-byte boundary, so any sample range
  [b0, b1) is three contiguous slices (``chunk``).  Tensors are pinned CPU tensors when CUDA is available."""

  def __init__(self, shape, bitmap, block_off, values, value_bits, sample_value_start):
    self.shape = tuple(shape)
    self.bitmap, self.block_off, self.values = bitmap, block_off, values
    self.value_bits = int(value_bits)
    self.sample_value_start = sample_value_start          # element index of each sample's first value, [B + 1]
    self.blocks_per_sample = int(np.prod(shape[1:])) // 1024

  @property
  def nbytes(self) -> int:
    return self.bitmap.numel() * 4 + self.block_off.numel() * 4 + self.values.numel()

  def chunk(self, b0: int, b1: int):
    """(bitmap, block_off, values, value_base, n_blocks) slices for samples [b0, b1)."""
    k = self.blocks_per_sample
    v0, v1 = int(self.sample_value_start[b0]), int(self.sample_value_start[b1])
    per_byte = 8 // self.value_bits
    return (self.bitmap[b0 * k * 32:b1 * k * 32], self.block_off[b0 * k:b1 * k + 1],
            self.values[v0 // per_byte:(v1 + per_byte - 1) // per_byte], v0, (b1 - b0) * k)


def zsf_encode(frames: np.ndarray) -> ZsfBatch:
  """Host-side encoder (data-loader side, numpy): uint8 frames (B, T, H, W, 2) -> :class:`ZsfBatch`.  Exact for any
  counts: 4-bit values when every count <= 15, else 8-bit."""
  frames = np.ascontiguousarray(frames, dtype=np.uint8)
  B = frames.shape[0]
  cells = int(np.prod(frames.shape[1:]))
  if cells % 1024:
    raise ValueError("zsf_encode: T*H*W*2 must be a multiple of 1024")
  flat = frames.reshape(B, cells)
  nz = flat != 0
  value_bits = 4 if (flat.max(initial=0) <= 15) else 8
  per_byte = 8 // value_bits
  bitmap = np.packbits(nz.reshape(B, cells // 32, 32), axis=-1, bitorder="little").view(np.uint32).reshape(B, cells // 32)
  per_block = nz.reshape(B, cells // 1024, 1024).sum(-1, dtype=np.int64)            # (B, blocks)
  per_sample = per_block.sum(-1)
  align = 16 * per_byte                                                              # values per 16 bytes
  padded = (per_sample + align - 1) // align * align
  sample_start = np.zeros(B + 1, np.int64)
  sample_start[1:] = np.cumsum(padded)
  if sample_start[-1] >= 2 ** 32:
    raise ValueError("zsf_encode: more than 2^32 values in one batch; encode smaller batches")
  block_off = np.zeros(B * (cells // 1024) + 1, np.int64)
  inner = np.cumsum(per_block, axis=1) - per_block                                   # exclusive, per sample
  block_off[:-1] = (inner + sample_start[:B, None]).reshape(-1)
  block_off[-1] = sample_start[B - 1] + per_sample[B - 1] if B else 0
  vals = np.zeros(int(sample_start[-1]), np.uint8)
  for b in range(B):
    vals[sample_start[b]:sample_start[b] + per_sample[b]] = flat[b][nz[b]]
  if value_bits == 4:
    vals = (vals[0::2] | (vals[1::2] << 4)).astype(np.uint8)
  t = lambda a: torch.as_tensor(np.ascontiguousarray(a))
  # torch has no general uint32 support: the words travel as int32 (same bits)
  ts = [t(bitmap.reshape(-1).view(np.int32)), t(block_off.astype(np.uint32).view(np.int32)), t(vals)]
  if torch.cuda.is_available():
    ts = [x.pin_memory() for x in ts]
  return ZsfBatch(frames.shape, ts[0], ts[1], ts[2], value_bits, sample_start)


def zsf_expand(bitmap: torch.Tensor, block_off: torch.Tensor, values: torch.Tensor, value_base: int, n_blocks: int,
               value_bits: int, out: torch.Tensor) -> torch.Tensor:
  """Device slices of a :class:`ZsfBatch` -> dense uint8 frames in ``out`` (n_blocks * 1024 bytes), on the current
  stream, no host sync."""
  _lib.check(_lib.lib().snnqp_expand_frames_zsf(_lib.ptr(bitmap), _lib.ptr(block_off), _lib.ptr(values),
                                                int(value_base), int(n_blocks), int(value_bits), _lib.ptr(out),
                                                _lib.stream()))
  return out


# ---- packed events: the event-list wire format of the end-to-end path -------------------------------------------
class EventBatch:
  """A batch of event recordings as packed words (``snnqp_events_to_frames_packed``, include/snnqp.h): ``events`` holds
  one word per event, all samples back to back in time order (int16 carrying the SNNQP_EVENTS_U16 bits, or int32
  carrying the SNNQP_EVENTS_U32 bits); ``offsets`` int64 [B+1] index sample b's words as
  ``events[offsets[b]:offsets[b+1]]``.  Tensors are pinned CPU tensors when CUDA is available.  ``eb[lo:hi]`` is a view
  of samples [lo, hi) (it shares ``events``); ``chunk(b0, b1)`` is what one host -> device copy of that range ships."""

  def __init__(self, events: torch.Tensor, offsets: torch.Tensor, format: int, sensor_wh: int,
               max_events_per_sample: int):
    self.events, self.offsets = events, offsets
    self.format = int(format)
    self.sensor_wh = int(sensor_wh)
    self.max_events_per_sample = int(max_events_per_sample)        # an upper bound of every sample's event count

  @property
  def shape(self):
    return (self.offsets.numel() - 1,)

  @property
  def nbytes(self) -> int:
    """Wire bytes of the batch: its words plus its offsets."""
    o0, o1 = int(self.offsets[0]), int(self.offsets[-1])
    return (o1 - o0) * self.events.element_size() + self.offsets.numel() * 8

  def __len__(self):
    return self.shape[0]

  def __getitem__(self, key):
    if not isinstance(key, slice) or key.step not in (None, 1):
      raise TypeError("EventBatch supports contiguous slices only")
    lo, hi, _ = key.indices(self.shape[0])
    hi = max(hi, lo)
    return EventBatch(self.events, self.offsets[lo:hi + 1], self.format, self.sensor_wh, self.max_events_per_sample)

  def chunk(self, b0: int, b1: int):
    """(events slice, offsets slice, event_base) for samples [b0, b1): the words of those samples, their offsets
    ``offsets[b0:b1+1]`` unchanged, and ``event_base = offsets[b0]``."""
    e0, e1 = int(self.offsets[b0]), int(self.offsets[b1])
    return self.events[e0:e1], self.offsets[b0:b1 + 1], e0


def encode_events(samples: Sequence[np.ndarray], sensor_wh: int) -> EventBatch:
  """Host-side encoder (data-loader side, numpy): list of (N_b, 3) integer (x, y, p) arrays in time order ->
  :class:`EventBatch`.  SNNQP_EVENTS_U16 when every x, y < 128, else SNNQP_EVENTS_U32 (every x, y < 2^15); p != 0
  becomes the polarity bit.  No event is dropped: every event counts toward the split of its sample, and an x beyond
  the sensor row is histogrammed at its flat position, as in ``events_to_frames``."""
  sizes = np.array([int(np.shape(a)[0]) for a in samples], np.int64)
  off = np.zeros(len(samples) + 1, np.int64)
  off[1:] = np.cumsum(sizes)
  flat = np.concatenate([np.asarray(a).reshape(-1, 3) for a in samples], 0) if off[-1] else np.zeros((0, 3), np.int64)
  if flat.dtype.kind not in "iu":
    raise ValueError("encode_events takes integer (x, y, p) records")
  xy = flat[:, :2]
  lo, hi = (int(xy.min()), int(xy.max())) if xy.size else (0, 0)
  if lo < 0 or hi >= 2 ** 15:
    bad = np.flatnonzero(((xy < 0) | (xy >= 2 ** 15)).any(1))
    b = int(np.searchsorted(off, bad[0], side="right") - 1)
    raise ValueError(f"encode_events: sample {b} has an event at (x, y) = {tuple(int(v) for v in xy[bad[0]])}, "
                     "outside [0, 32768); integrate such recordings with concat_events + events_to_frames")
  x, y = xy[:, 0].astype(np.uint32), xy[:, 1].astype(np.uint32)
  p = (flat[:, 2] != 0).astype(np.uint32)
  if hi < 128:
    fmt = _lib.EVENTS_U16
    words = (x | (y << 7) | (p << 15)).astype(np.uint16).view(np.int16)
  else:
    fmt = _lib.EVENTS_U32
    words = (x | (y << 15) | (p << 31)).view(np.int32)
  ev, offsets = torch.as_tensor(np.ascontiguousarray(words)), torch.as_tensor(off)
  if torch.cuda.is_available():
    ev, offsets = ev.pin_memory(), offsets.pin_memory()
  return EventBatch(ev, offsets, fmt, sensor_wh, int(sizes.max(initial=0)))


def events_to_frames_packed(events: torch.Tensor, offsets: torch.Tensor, event_format: int, num_frames: int, wh: int,
                            resolution_scale: int = 1, exact_int32: bool = False, out: Optional[torch.Tensor] = None,
                            max_events_per_sample: int = 0, event_base: int = 0,
                            n_saturated: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
  """:func:`events_to_frames` on packed event words (device tensors: ``events`` int16 for SNNQP_EVENTS_U16 or int32
  for SNNQP_EVENTS_U32, 16-byte aligned; ``offsets`` int64 [B+1], sample b's words at ``offsets[b] - event_base``).
  Returns (frames, n_saturated); a given ``n_saturated`` (device int64 scalar) is accumulated into, no host sync."""
  if int(resolution_scale) != resolution_scale or resolution_scale < 1:
    raise NotImplementedError("resolution_scale must be a positive integer")
  want = {_lib.EVENTS_U16: torch.int16, _lib.EVENTS_U32: torch.int32}.get(int(event_format))
  if want is None or events.dtype != want or offsets.dtype != torch.int64:
    raise ValueError("events must be int16 (EVENTS_U16) or int32 (EVENTS_U32) words and offsets int64 (B+1,)")
  B = offsets.numel() - 1
  whs = int(wh // resolution_scale)
  dt = torch.int32 if exact_int32 else torch.uint8
  if out is None:
    out = torch.empty((B, num_frames, whs, whs, 2), device=events.device, dtype=dt)
  if n_saturated is None:
    n_saturated = torch.zeros((), device=events.device, dtype=torch.int64)
  elif not n_saturated.is_cuda or n_saturated.dtype != torch.int64 or n_saturated.numel() != 1:
    raise ValueError("n_saturated must be a device int64 scalar")
  if B == 0:
    return out, n_saturated
  _lib.check(_lib.lib().snnqp_events_to_frames_packed(
      _lib.ptr(events), int(event_format), _lib.ptr(offsets), int(event_base), B, num_frames, int(wh),
      int(resolution_scale), int(max_events_per_sample), _lib.ptr(out), 1 if exact_int32 else 0,
      _lib.ptr(n_saturated), _lib.stream()))
  return out, n_saturated
