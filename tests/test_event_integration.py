"""The event front end -- packed event words, their integration into frames on the GPU, and
CextNetEngine.forward_host_events -- against a plain reference written in this file from the documented definition
(include/snnqp.h), not from the CUDA code:

* unpack: SNNQP_EVENTS_U16  x = w & 0x7F,   y = (w >> 7) & 0x7F,   p = w >> 15 (bit 14 zero);
          SNNQP_EVENTS_U32  x = w & 0x7FFF, y = (w >> 15) & 0x7FFF, p = w >> 31 (bit 30 zero).
* integrate ("split by number", the reference's preprocess_data_number): the N events of a sample, in order, fall in
  T groups; with di = N // T, event i belongs to group min(i // di, T - 1) (every event to the last group when
  di = 0).  So group t is the half-open index range [t di, (t + 1) di), and the last group also takes the remainder.
  An event adds one to frame t, cell (floor(y / rs) * wh + floor(x / rs), p != 0) of a (wh, wh, 2) frame,
  wh = sensor_wh // rs.  Flat positions outside [0, wh * wh) are dropped.  int32 output is exact; uint8 output
  saturates at 255 and n_saturated counts the cells above 255.

These words carry no timestamps: an event's frame is fixed by its index within its sample.  So the bin edges here are
the group bounds t * di, and the chunk edges are the sample ranges [b0, b1) that a batch is shipped in
(EventBatch.chunk, CextNetEngine.host_chunks).  A sample is never split between chunks.

Event counts are integers, so every GPU comparison is exact (torch.equal).  The reference itself is checked on the CPU
against hand-computed cases and against oracle/ref_events.py, the restatement of the original loader."""
import numpy as np
import pytest
import torch

from oracle import ref_events
from snnquantprune_b200 import _lib
from snnquantprune_b200 import input_pipeline as ip

U16, U32 = 1, 2           # SNNQP_EVENTS_U16, SNNQP_EVENTS_U32 (include/snnqp.h)
XY_MAX = {U16: 127, U32: 32767}
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ the reference ----
def pack_words(xyp, fmt) -> np.ndarray:
  """(N, 3) (x, y, p), every x, y in [0, XY_MAX[fmt]] -> the wire words (uint16 / uint32), from the header's layout."""
  a = np.asarray(xyp, np.int64).reshape(-1, 3)
  assert ((a[:, :2] >= 0) & (a[:, :2] <= XY_MAX[fmt])).all()
  p = (a[:, 2] != 0).astype(np.int64)
  if fmt == U16:
    return (a[:, 0] | (a[:, 1] << 7) | (p << 15)).astype(np.uint16)
  return (a[:, 0] | (a[:, 1] << 15) | (p << 31)).astype(np.uint32)


def unpack_words(words, fmt) -> np.ndarray:
  """Wire words (any signedness: only the bits count) -> int64 (N, 3) (x, y, p), field by field."""
  if fmt == U16:
    w = np.asarray(words).view(np.uint16).astype(np.int64)
    assert not (w & (1 << 14)).any()
    return np.stack([w & 0x7F, (w >> 7) & 0x7F, (w >> 15) & 1], 1)
  w = np.asarray(words).view(np.uint32).astype(np.int64)
  assert not (w & (1 << 30)).any()
  return np.stack([w & 0x7FFF, (w >> 15) & 0x7FFF, (w >> 31) & 1], 1)


def frame_of_event(n: int, T: int) -> np.ndarray:
  """Group (frame) index of each of the n events of a sample."""
  di = n // T
  return np.minimum(np.arange(n) // di, T - 1) if di else np.full(n, T - 1, np.int64)


def integrate(samples, T: int, sensor_wh: int, rs: int = 1) -> np.ndarray:
  """List of (N_b, 3) integer (x, y, p) -> int64 (B, T, wh, wh, 2) event counts."""
  wh = sensor_wh // rs
  out = np.zeros((len(samples), T, wh * wh, 2), np.int64)
  for b, a in enumerate(samples):
    a = np.asarray(a, np.int64).reshape(-1, 3)
    pos = (a[:, 1] // rs) * wh + a[:, 0] // rs          # numpy's // on integers floors
    keep = (pos >= 0) & (pos < wh * wh)
    np.add.at(out[b], (frame_of_event(len(a), T)[keep], pos[keep], (a[keep, 2] != 0).astype(np.int64)), 1)
  return out.reshape(len(samples), T, wh, wh, 2)


def saturate_u8(frames: np.ndarray):
  """The uint8 output and its n_saturated."""
  return np.minimum(frames, 255).astype(np.uint8), int((frames > 255).sum())


# -------------------------------------------------------------------------------------------- stream builders ----
def _rand(rng, n, hi_xy, p_vals=(0, 1)):
  return np.concatenate([rng.integers(0, hi_xy, (n, 2)), rng.choice(np.asarray(p_vals), (n, 1))], 1).astype(np.int64)


def _tagged(n: int, first: int = 0, wh: int = 128) -> np.ndarray:
  """n events on n distinct cells: event i on cell (first + i) of a wh x wh x 2 frame (pixel c >> 1, polarity c & 1).
  An event counted in the wrong frame, twice or not at all changes the frames wherever it sits."""
  c = (first + np.arange(n)) % (2 * wh * wh)
  return np.stack([(c >> 1) % wh, (c >> 1) // wh, c & 1], 1).astype(np.int64)


def _one_pixel(n: int, x: int, y: int, p) -> np.ndarray:
  """n events on pixel (x, y); p is a polarity, or "alt" for 0, 1, 0, 1, ..."""
  pol = np.arange(n) & 1 if p == "alt" else np.full(n, p)
  return np.stack([np.full(n, x), np.full(n, y), pol], 1).astype(np.int64)


# -------------------------------------------------------------------------------------------------- the kernel ----
def _offsets(samples) -> np.ndarray:
  return np.concatenate([[0], np.cumsum([len(s) for s in samples])]).astype(np.int64)


def _words(samples, fmt) -> np.ndarray:
  parts = [pack_words(s, fmt) for s in samples if len(s)]
  return np.concatenate(parts) if parts else np.zeros(0, np.uint16 if fmt == U16 else np.uint32)


def _kernel(words, fmt, offsets, T, sensor_wh, rs=1, exact_int32=True, bound=0, event_base=0):
  """One snnqp_events_to_frames_packed call on a fresh (16-byte aligned) device copy of ``words``.  Returns the frames
  on the host and n_saturated."""
  dt = torch.int16 if fmt == U16 else torch.int32
  w = torch.from_numpy(np.ascontiguousarray(words).view(np.int16 if fmt == U16 else np.int32))
  d = torch.zeros(max(w.numel(), 1), dtype=dt, device="cuda")
  d[:w.numel()].copy_(w)
  f, sat = ip.events_to_frames_packed(d, torch.as_tensor(offsets, dtype=torch.int64).cuda(), fmt, T, sensor_wh, rs,
                                      exact_int32=exact_int32, max_events_per_sample=bound, event_base=event_base)
  return f.cpu(), int(sat.item())


def _where(got: torch.Tensor, want: torch.Tensor) -> str:
  """The first few differing cells, (b, t, y, x, p): got / want."""
  bad = (got.to(torch.int64) != want.to(torch.int64)).nonzero()[:4].tolist()
  return "; ".join(f"{tuple(i)}: {int(got[tuple(i)])} / {int(want[tuple(i)])}" for i in bad)


def check_kernel(samples, fmt, T, sensor_wh, rs=1, ranges=(), bounds=None):
  """The kernel on ``samples`` packed as ``fmt``, against the reference, exactly: int32 and uint8 output, with 32-bit
  counters (bound 0), the 16-bit counters the exact bound allows, and a bound too large for them; then each sample
  range [b0, b1) of ``ranges`` shipped as its own words slice with event_base = offsets[b0]."""
  words, off = _words(samples, fmt), _offsets(samples)
  want = integrate(samples, T, sensor_wh, rs)
  want32 = torch.from_numpy(want.astype(np.int32))
  w8, nsat = saturate_u8(want)
  want8 = torch.from_numpy(w8)
  nmax = int(np.diff(off).max(initial=0))
  for bound in (bounds if bounds is not None else (0, nmax, 10 ** 9)):
    got, _ = _kernel(words, fmt, off, T, sensor_wh, rs, True, bound)
    assert torch.equal(got, want32), f"int32, bound {bound}: {_where(got, want32)}"
    got, sat = _kernel(words, fmt, off, T, sensor_wh, rs, False, bound)
    assert torch.equal(got, want8), f"uint8, bound {bound}: {_where(got, want8)}"
    assert sat == nsat, (bound, sat, nsat)
  for b0, b1 in ranges:
    got, _ = _kernel(words[off[b0]:off[b1]], fmt, off[b0:b1 + 1], T, sensor_wh, rs, True, nmax, int(off[b0]))
    assert torch.equal(got, want32[b0:b1]), f"samples [{b0}, {b1}): {_where(got, want32[b0:b1])}"
  return want


# ------------------------------------------------------------------------------------ CPU: the reference itself ----
def test_reference_hand_case():
  # 7 events, T = 3: di = 2, frames take events [0, 2), [2, 4), [4, 7)
  a = np.array([[0, 0, 1], [1, 0, 0], [1, 1, 1], [1, 1, 1], [0, 1, 0], [0, 1, 0], [3, 3, 5]])
  f = integrate([a], 3, 4)[0]
  assert f.sum() == 7 and f[0].sum() == 2 and f[1].sum() == 2 and f[2].sum() == 3
  assert f[0, 0, 0, 1] == 1 and f[0, 0, 1, 0] == 1 and f[1, 1, 1, 1] == 2
  assert f[2, 1, 0, 0] == 2 and f[2, 3, 3, 1] == 1
  # rs = 2 on a 4 x 4 sensor: wh = 2; negative coordinates floor (-1 // 2 = -1): (x, y) = (-1, 2) -> flat position
  # 1 * 2 - 1 = 1, i.e. pixel (1, 0); (1, -1) -> position -2 + 0, dropped
  g = integrate([np.array([[3, 3, 0], [-1, 2, 1], [1, -1, 0], [2, 1, 0]])], 1, 4, 2)[0, 0]
  assert g[1, 1, 0] == 1 and g[0, 1, 1] == 1 and g[0, 1, 0] == 1 and g.sum() == 3


@pytest.mark.parametrize("T", [1, 3, 7, 20])
def test_reference_group_edges(T):
  """One index either side of every group bound t * di: event t di - 1 is in frame t - 1, event t di in frame t;
  the last frame holds di + N % T events; N < T puts every event in the last frame."""
  for n in (0, 1, T - 1, T, T + 1, 5 * T - 1, 5 * T, 5 * T + 1, 37 * T + T // 2):
    g = frame_of_event(n, T)
    di = n // T
    assert len(g) == n and (np.diff(g) >= 0).all()
    if di == 0:
      assert (g == T - 1).all()
      continue
    for t in range(1, T):
      assert g[t * di - 1] == t - 1 and g[t * di] == t
    assert np.bincount(g, minlength=T).tolist() == [di] * (T - 1) + [n - (T - 1) * di]


def test_reference_matches_oracle():
  """The reference here and oracle/ref_events.py (a line-by-line restatement of the original loader: slices,
  float floor-division, bincount) agree on every shape of input: negative coordinates, flat-position overflow,
  N < T, empty samples, polarity values other than 0 and 1."""
  rng = np.random.default_rng(7)
  T = 5
  samples = [_rand(rng, n, 140, (0, 1, 2, -1)) for n in (0, 1, 4, 5, 6, 999, 2000)]
  samples[5][:, :2] -= 9                    # coordinates in [-9, 131)
  samples[6][:100] = [127, 127, 1]
  for wh, rs in ((128, 1), (128, 2), (128, 3), (64, 4)):
    assert np.array_equal(integrate(samples, T, wh, rs), ref_events.batch_to_frames(samples, T, wh, rs)), (wh, rs)
    w8, nsat = saturate_u8(integrate(samples, T, wh, rs))
    r8, rsat = ref_events.batch_to_frames(samples, T, wh, rs, saturate_u8=True)
    assert np.array_equal(w8, r8) and nsat == rsat


# ------------------------------------------------------------------------------------ CPU: pack and unpack ----
def _field_edges(fmt):
  m = XY_MAX[fmt]
  v = [0, 1, m // 2, (m + 1) // 2, m - 1, m]
  return np.array([[x, y, p] for x in v for y in v for p in (0, 1)], np.int64)


@pytest.mark.parametrize("fmt", [U16, U32])
def test_pack_layout_at_field_edges(fmt):
  """Every field at zero, one, its middle bits and its maximum: the encoder's words are the header's layout, bit for
  bit, and unpack back to the records."""
  a = _field_edges(fmt)
  eb = ip.encode_events([a[:5], a[5:]], 128)
  assert eb.format == fmt
  words = eb.events.numpy()
  ref = pack_words(a, fmt)
  assert np.array_equal(words.view(ref.dtype), ref)
  assert np.array_equal(unpack_words(words, fmt), a)
  # the top bit of each field, alone
  if fmt == U16:
    top = {(127, 0, 0): 0x007F, (64, 0, 0): 0x0040, (0, 127, 0): 0x3F80, (0, 64, 0): 0x2000, (0, 0, 1): 0x8000,
           (127, 127, 1): 0xBFFF}
  else:
    top = {(32767, 0, 0): 0x00007FFF, (16384, 0, 0): 0x00004000, (0, 32767, 0): 0x3FFF8000,
           (0, 16384, 0): 0x20000000, (0, 0, 1): 0x80000000, (32767, 32767, 1): 0xBFFFFFFF}
  for rec, word in top.items():
    got = ip.encode_events([np.array([rec]), np.array([[0, 0, 0], [XY_MAX[fmt], 0, 0]])], 128).events.numpy()
    assert int(got.view(ref.dtype)[0]) == word, (rec, hex(word))
    assert unpack_words(np.array([word], ref.dtype), fmt)[0].tolist() == list(rec)


@pytest.mark.parametrize("fmt", [U16, U32])
def test_pack_round_trip_full_range(fmt):
  """Random records over each field's whole legal range (the maxima included) and polarity values far from {0, 1}:
  encode then unpack is the identity, with p != 0 as the polarity bit."""
  rng = np.random.default_rng(fmt)
  m = XY_MAX[fmt]
  sizes = (0, 1, 2, 7, 8, 9, 4095, 0, 30001)
  samples = [np.concatenate([rng.integers(0, m + 1, (n, 2)),
                             rng.choice(np.array([0, 1, 2, 256, -1, -2 ** 31, 2 ** 40]), (n, 1))], 1)
             for n in sizes]
  samples[-1][:4] = [[m, m, 0], [m, m, 256], [0, 0, 0], [0, 0, 2 ** 40]]
  eb = ip.encode_events(samples, 128)
  assert eb.format == fmt and eb.max_events_per_sample == 30001
  want = np.concatenate(samples)
  want[:, 2] = want[:, 2] != 0
  assert np.array_equal(unpack_words(eb.events.numpy(), fmt), want)
  assert eb.offsets.tolist() == _offsets(samples).tolist()


def test_pack_rejects_out_of_range():
  """A coordinate outside [0, 2^15) is rejected with a ValueError naming the sample, never truncated to a field; so
  is a record that is not integer."""
  ok = np.array([[1, 2, 0]])
  for bad in ((32768, 0), (0, 32768), (-1, 0), (0, -1), (65535, 0), (2 ** 31 - 1, 5), (-2 ** 31, 5), (2 ** 40, 0),
              (0, 2 ** 47 + 3)):
    rec = np.array([[bad[0], bad[1], 1]], np.int64)
    with pytest.raises(ValueError, match=r"sample 2 has an event at"):
      ip.encode_events([ok, ok, np.concatenate([ok, rec])], 128)
  with pytest.raises(ValueError, match="integer"):
    ip.encode_events([np.array([[1.0, 2.0, 0.0]])], 128)
  # 127 / 128 is the U16 / U32 boundary; 32767 is the largest U32 coordinate
  assert ip.encode_events([np.array([[127, 127, 1]])], 128).format == U16
  assert ip.encode_events([np.array([[128, 0, 1]])], 128).format == U32
  eb = ip.encode_events([np.array([[32767, 32767, 1]])], 128)
  assert eb.format == U32 and unpack_words(eb.events.numpy(), U32).tolist() == [[32767, 32767, 1]]


# --------------------------------------------------------------------------------- GPU: the integration kernel ----
@gpu
@pytest.mark.parametrize("fmt,sensor,rs", [(U16, 128, 1), (U32, 128, 1), (U32, 256, 2)])
def test_kernel_random_streams_production_geometry(cuda_lib, fmt, sensor, rs):
  """Synthetic recordings at the production bin count (T = 20) and sensor (128 x 128; 256 x 256 at rs = 2), both
  packed formats."""
  from snnquantprune_b200 import synthetic
  samples = synthetic.make_events(5, 20, sensor, seed=fmt + sensor)
  samples[2][:3000] = [sensor - 1, sensor - 1, 1]          # a saturating pixel
  want = check_kernel(samples, fmt, 20, sensor, rs, ranges=((1, 5), (4, 5)))
  assert want.max() > 255


@gpu
@pytest.mark.parametrize("fmt", [U16, U32])
def test_kernel_group_edges(cuda_lib, fmt):
  """Every event on its own cell, so an event on the wrong side of a group bound shows.  Sample sizes are one below,
  at and one above a multiple of T (and N < T), for T = 1, 7 and 20; the samples sit back to back and are shipped
  from every start sample, so the group bounds fall at many word positions of a 16-byte vector."""
  for T in (1, 7, 20):
    sizes = [T - 1, T, T + 1, 1, 13 * T - 1, 13 * T, 13 * T + 1, 0, 257 * T - 1, 257 * T + 7, 3, 64 * T]
    samples, first = [], 0
    for n in sizes:
      samples.append(_tagged(n, first))
      first += 977
    check_kernel(samples, fmt, T, 128, ranges=[(b0, len(sizes)) for b0 in range(1, len(sizes))] + [(0, 5), (4, 5)],
                 bounds=(0, max(sizes)))


@gpu
@pytest.mark.parametrize("fmt", [U16, U32])
def test_kernel_one_pixel_collisions(cuda_lib, fmt):
  """Every event of a group on one pixel -- the corners (0, 0) and (127, 127), one polarity and alternating -- so all
  512 threads of a block add to the same counter (with 16-bit counters, alternating polarities hit both halves of one
  word).  Groups of 25 000 events also take several passes of each thread over the group."""
  samples = [_one_pixel(50001, 0, 0, 0), _one_pixel(50001, 127, 127, 1), _one_pixel(4099, 127, 127, "alt"),
             _one_pixel(777, 0, 0, "alt")]
  samples.append(np.concatenate([_one_pixel(20000, 0, 0, 1), _one_pixel(20001, 127, 127, 0)]))
  check_kernel(samples, fmt, 2, 128, ranges=((2, 5),))


@gpu
@pytest.mark.parametrize("fmt", [U16, U32])
def test_kernel_long_groups(cuda_lib, fmt):
  """Random groups far longer than one pass of the block over them (512 threads; 4096 U16 / 2048 U32 words a pass)."""
  rng = np.random.default_rng(20 + fmt)
  samples = [_rand(rng, n, 128) for n in (120001, 9, 65537)]
  check_kernel(samples, fmt, 3, 128, ranges=((1, 3),))


@gpu
def test_kernel_count_limits(cuda_lib):
  """The largest count each output and counter holds, and one more.  uint8: 254, 255 and 256 events on one cell give
  254, 255, 255 and one saturated cell.  Shared-memory counters: 16 bits are used only while a frame provably holds
  fewer than 65536 events (N // T + T < 65536).  A last frame of 65534 events (the most that bound admits) is exact in
  16-bit counters; frames of 65535 and 65536 events (the latter past any 16-bit counter) must take the 32-bit
  counters and stay exact, including a last group made that large by the remainder (T = 2, N = 2 * 65535 + 1)."""
  s = [np.concatenate([_one_pixel(254, 5, 6, 0), _one_pixel(255, 127, 0, 1), _one_pixel(256, 0, 127, 0)])]
  want = check_kernel(s, U16, 1, 128)
  assert sorted(want[want > 0].tolist()) == [254, 255, 256]
  assert saturate_u8(want)[1] == 1
  for fmt in (U16, U32):
    for T, n, xy, p in ((1, 65534, (127, 127), 0), (2, 2 * 65533 + 1, (0, 0), 1), (1, 65535, (0, 0), 0),
                        (1, 65536, (127, 127), 0), (1, 65536, (3, 3), 1), (2, 2 * 65535 + 1, (0, 0), 0)):
      samples = [_one_pixel(n, *xy, p), _one_pixel(7, *xy, p)]
      want = check_kernel(samples, fmt, T, 128)
      assert want[0, -1, xy[1], xy[0], p] == n - (T - 1) * (n // T), (T, n)


@gpu
@pytest.mark.parametrize("fmt", [U16, U32])
def test_kernel_empty_short_and_partial(cuda_lib, fmt):
  """An all-empty batch, an empty batch (B = 0), empty samples in the middle, one-event samples (the event lands in
  the last frame), N < T, and a last group holding T - 1 remainder events; then every sample range of the batch."""
  T = 20
  got, sat = _kernel(_words([], fmt), fmt, np.zeros(4, np.int64), T, 128)
  assert got.shape == (3, T, 128, 128, 2) and not got.any() and sat == 0
  empty, _ = ip.events_to_frames_packed(torch.zeros(8, dtype=torch.int16 if fmt == U16 else torch.int32,
                                                    device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"),
                                        fmt, T, 128)
  assert empty.shape == (0, T, 128, 128, 2)
  rng = np.random.default_rng(5)
  sizes = (0, 1, 0, 0, T - 1, 1, 2 * T + T - 1, 0, 1)
  samples = [_rand(rng, n, 128) for n in sizes]
  B = len(sizes)
  want = check_kernel(samples, fmt, T, 128, ranges=[(b0, b1) for b0 in range(B) for b1 in range(b0 + 1, B + 1)])
  assert want[1, :-1].sum() == 0 and want[1, -1].sum() == 1


@gpu
@pytest.mark.parametrize("rs", [1, 2, 4])
def test_kernel_polarity_and_corners(cuda_lib, rs):
  """Each corner pixel and polarity gets its own count (1 .. 8 events, in shuffled order): a swap of the polarity
  channels or of x and y, or a lost corner, changes the frame."""
  rng = np.random.default_rng(rs)
  for fmt, sensor in ((U16, 128), (U32, 128), (U32, 256)):
    if sensor // rs > 128:                    # the largest frame the shared-memory histogram holds is 128 x 128
      continue
    m = sensor - 1
    cells = [(x, y, p) for x in (0, m) for y in (0, m) for p in (0, 1)]
    ev = np.concatenate([np.tile(np.array([c]), (k + 1, 1)) for k, c in enumerate(cells)])
    ev = ev[rng.permutation(len(ev))]
    want = check_kernel([ev, ev[::-1]], fmt, 1, sensor, rs)
    for k, (x, y, p) in enumerate(cells):
      assert want[0, 0, y // rs, x // rs, p] == k + 1, (fmt, sensor, x, y, p)
    assert want.sum() == 2 * len(ev)


@gpu
@pytest.mark.parametrize("rs", [1, 2, 4])
def test_int32_records_floor_negative_coordinates(cuda_lib, rs):
  """The int32-record entry point (the route encode_events names for coordinates outside the packed range) floors
  x / rs and y / rs like the reference's float floor-division: (-1, y) at rs = 2 is x = -1, the last pixel of the
  previous row, and y in (-rs, 0) is a row above the frame, dropped -- not row 0."""
  rng = np.random.default_rng(30 + rs)
  T, wh = 3, 128
  samples = [_rand(rng, n, 150, (0, 1)) - np.array([11, 11, 0]) for n in (5000, 17, 0, 3001)]
  samples[1][:, :2] = [[-1, 5], [-2, 5], [-3, 5], [5, -1], [5, -2], [-1, -1], [0, 0], [127, 127], [-rs, 4],
                       [-rs - 1, 4], [4, -rs], [128, 3], [-128, 9], [3, 127 + rs], [-7, 1], [1, -7], [130, 0]]
  want = integrate(samples, T, wh, rs)
  assert np.array_equal(want, ref_events.batch_to_frames(samples, T, wh, rs))
  addrs, off = ip.concat_events(samples)
  for bound in (0, 5000):
    got, _ = ip.events_to_frames(addrs.cuda(), off.cuda(), T, wh, rs, exact_int32=True, max_events_per_sample=bound)
    want32 = torch.from_numpy(want.astype(np.int32))
    assert torch.equal(got.cpu(), want32), f"bound {bound}: {_where(got.cpu(), want32)}"


# ----------------------------------------------------------------------------------------------- GPU: the engine ----
def _engine_stream(B, T, H, seed):
  from snnquantprune_b200 import synthetic
  samples = synthetic.make_events(B, T, H, seed=seed, rate=0.05)
  samples[3] = samples[3][:0]                                 # an empty sample
  samples[5] = samples[5][:1]                                 # a one-event sample
  samples[B - 1][:2000, :2] = [H - 1, 0]                      # a saturating pixel in the last sample
  return samples


@gpu
def test_chunking_invariance(cuda_lib):
  """One batch of recordings, split into sample ranges several ways -- one sample per call, ragged ranges, the whole
  batch -- integrates to the same frames; and forward_host_events gives the same logits at chunk = 1, 2, 4 and B
  (the dense kernels are deterministic at a fixed input), equal to forward on the reference's frames."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic
  bits, T, H, B = 8, 20, 128, 9
  samples = _engine_stream(B, T, H, seed=8)
  eb = ip.encode_events(samples, H)
  assert eb.format == U16
  want8 = torch.from_numpy(saturate_u8(integrate(samples, T, H))[0])
  words, off = eb.events.numpy(), eb.offsets.numpy()
  for cuts in ([0, B], list(range(B + 1)), [0, 2, 3, 7, B], [0, 1, B - 1, B], [0, 4, 5, 6, B]):
    parts = []
    for b0, b1 in zip(cuts[:-1], cuts[1:]):
      ev, o, base = eb.chunk(b0, b1)
      parts.append(_kernel(ev.numpy(), U16, o.numpy(), T, H, 1, False, eb.max_events_per_sample, base)[0])
    got = torch.cat(parts)
    assert torch.equal(got, want8), f"cuts {cuts}: {_where(got, want8)}"
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  pk = pack_cextnet(v, bits, T, H, device="cuda")
  ref = CextNetEngine(pk, chunk=B).forward(want8.cuda()).cpu()
  for chunk in (1, 2, 4, B):
    eng = CextNetEngine(pk, chunk=chunk)
    got = eng.forward_host_events(eb).cpu()
    assert torch.equal(got, ref), chunk
    assert torch.equal(eng.forward(want8.cuda()).cpu(), ref), chunk


@gpu
def test_end_to_end_small_stream(cuda_lib):
  """A short synthetic recording through forward_host_events, one sample per chunk, against the reference integration
  followed by the per-stage oracles chained (as smoke() chains them): both staged frame buffers hold the reference's
  frames, conv1 .. conv4 spikes equal the integer oracle's on those frames, the logits equal the oracle's with the
  attention path's own values forced (tests/test_gpu_attention_path.py holds those to their emulation), and
  forward_host_events returns the same logits."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic
  from oracle import ref_net
  bits, T, H, B = 8, 4, 128, 2
  samples = synthetic.make_events(B, T, H, seed=12)
  samples[1][::8] = [0, 127, 0]                             # one saturated cell per frame of sample 1
  frames8, nsat = saturate_u8(integrate(samples, T, H))
  assert nsat == T
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  eng = CextNetEngine(pack_cextnet(v, bits, T, H, device="cuda"), chunk=1, lif_mode=_lib.LIF_EXACT)
  n_sat = torch.zeros((), dtype=torch.int64, device="cuda")
  got = eng.forward_host_events(ip.encode_events(samples, H), n_saturated=n_sat).cpu().numpy()
  stage = eng._workspace(B, 1)["stage"]
  for b in range(B):                                        # chunk b was integrated into staging buffer b & 1
    assert np.array_equal(stage[b & 1][0].cpu().numpy(), frames8[b]), b
  assert int(n_sat.item()) == nsat
  c = {}                                                    # the instrumented pass takes the batch as one chunk
  logits = CextNetEngine(eng.pk, chunk=B, lif_mode=_lib.LIF_EXACT).forward(torch.from_numpy(frames8).cuda(),
                                                                           collect=c).cpu().numpy()
  tb = lambda k: np.ascontiguousarray(np.swapaxes(c[k].cpu().numpy(), 0, 1))
  forced = {"att4": tb("att4"), "s5": tb("s5"), "att5": tb("att5"), "d1": tb("d1")}
  co = {}
  lo = ref_net.forward(ref_net.pack_network(v, bits, H), frames8, collect=co, forced=forced)
  for k in ("s1", "s2", "s3", "s4"):
    assert np.array_equal(tb(k), co[k]), k
  assert np.array_equal(logits, lo)
  assert np.array_equal(got, logits)
