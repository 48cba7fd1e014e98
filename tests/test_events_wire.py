"""Packed event words (SNNQP_EVENTS_U16 / _U32): the host encoder and EventBatch on the CPU, the packed integration
kernel bit-exact against the oracle and the int32-record kernel on the GPU (through the C-ABI), and
CextNetEngine.forward_host_events against the device-resident forward."""
import os
import re

import numpy as np
import pytest
import torch

import eventsref
from oracle import ref_events
from snnquantprune_b200 import _lib
from snnquantprune_b200 import input_pipeline as ip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rand(rng, n, lo_xy, hi_xy, p_vals=(0, 1)):
  xy = rng.integers(lo_xy, hi_xy, (n, 2))
  p = rng.choice(np.asarray(p_vals), n)
  return np.concatenate([xy, p[:, None]], 1).astype(np.int64)


def _decoded(eb):
  return eventsref.decode_events(eb.events.numpy(), eb.format)


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hi_xy,fmt", [(128, _lib.EVENTS_U16), (2 ** 15, _lib.EVENTS_U32)])
def test_encode_decode_round_trip(hi_xy, fmt):
  rng = np.random.default_rng(hi_xy)
  samples = [_rand(rng, n, 0, hi_xy, (0, 1, 2, -3, 255)) for n in (0, 1, 17, 1000, 0, 333)]
  eb = ip.encode_events(samples, 128)
  assert eb.format == fmt and eb.events.dtype == (torch.int16 if fmt == _lib.EVENTS_U16 else torch.int32)
  assert eb.shape == (6,) and eb.max_events_per_sample == 1000 and eb.sensor_wh == 128
  got = _decoded(eb)
  want = np.concatenate(samples, 0)
  want[:, 2] = want[:, 2] != 0
  assert np.array_equal(got, want)
  assert eb.offsets.tolist() == np.concatenate([[0], np.cumsum([len(s) for s in samples])]).tolist()
  assert eb.nbytes == want.shape[0] * eb.events.element_size() + 7 * 8


def test_encode_format_selection_and_range():
  one = lambda x, y: [np.array([[3, 4, 1]]), np.array([[x, y, 0]])]
  assert ip.encode_events(one(127, 127), 128).format == _lib.EVENTS_U16
  assert ip.encode_events(one(128, 0), 128).format == _lib.EVENTS_U32
  assert ip.encode_events(one(0, 128), 128).format == _lib.EVENTS_U32
  eb = ip.encode_events(one(32767, 32767), 128)
  assert eb.format == _lib.EVENTS_U32 and _decoded(eb)[1].tolist() == [32767, 32767, 0]
  assert ip.encode_events([np.zeros((0, 3), np.int64)], 128).format == _lib.EVENTS_U16
  for x, y in ((32768, 0), (0, 32768), (-1, 5), (5, -1)):
    with pytest.raises(ValueError, match=r"sample 1 .*concat_events \+ events_to_frames"):
      ip.encode_events(one(x, y), 128)


def test_event_batch_chunk_and_slicing():
  rng = np.random.default_rng(4)
  sizes = (5, 0, 9, 1, 0, 0, 16, 3)
  samples = [_rand(rng, n, 0, 128) for n in sizes]
  eb = ip.encode_events(samples, 128)
  words = eb.events.numpy()
  off = np.concatenate([[0], np.cumsum(sizes)])
  B = len(sizes)
  for b0 in range(B + 1):
    for b1 in range(b0, B + 1):
      ev, o, base = eb.chunk(b0, b1)
      assert base == off[b0] and o.tolist() == off[b0:b1 + 1].tolist()
      assert np.array_equal(ev.numpy(), words[off[b0]:off[b1]])
      v = eb[b0:b1]
      assert v.shape == (b1 - b0,) and v.events is eb.events and v.format == eb.format
      for c0 in range(b1 - b0 + 1):            # a chunk of the view is the same chunk of the parent
        for c1 in range(c0, b1 - b0 + 1):
          ev2, o2, base2 = v.chunk(c0, c1)
          ev1, o1, base1 = eb.chunk(b0 + c0, b0 + c1)
          assert base2 == base1 and torch.equal(o2, o1) and torch.equal(ev2, ev1)
      # the words of sample b of the view, rebased
      for k in range(b1 - b0):
        sl = ev.numpy()[int(o[k]) - base:int(o[k + 1]) - base]
        assert np.array_equal(eventsref.decode_events(sl, eb.format)[:, :2], samples[b0 + k][:, :2])


def test_lib_constants_and_signature_match_header():
  header = open(os.path.join(ROOT, "include", "snnqp.h")).read()
  val = lambda name: int(re.search(rf"#define {name} (-?\d+)", header).group(1))
  assert (_lib.EVENTS_U16, _lib.EVENTS_U32) == (val("SNNQP_EVENTS_U16"), val("SNNQP_EVENTS_U32"))
  assert (eventsref.U16, eventsref.U32) == (_lib.EVENTS_U16, _lib.EVENTS_U32)
  decl = re.search(r"int snnqp_events_to_frames_packed\((.*?)\);", header, re.S).group(1)
  kinds = {"int": _lib.C.c_int, "int64_t": _lib.C.c_int64}
  args = [_lib.C.c_void_p if "*" in a else kinds[a.split()[0]] for a in decl.split(",")]
  res, want = _lib.SIGNATURES["snnqp_events_to_frames_packed"]
  assert res is _lib.C.c_int and want == args and len(args) == 13


# ---- GPU: the kernel --------------------------------------------------------------------------------------------------
def _dev_aligned(t: torch.Tensor) -> torch.Tensor:
  """A fresh (16-byte aligned) device copy with at least one element."""
  d = torch.zeros(max(t.numel(), 1), dtype=t.dtype, device="cuda")
  d[:t.numel()].copy_(t)
  return d


def _packed(eb, b0, b1, T, wh, rs, **kw):
  ev, off, base = eb.chunk(b0, b1)
  kw.setdefault("max_events_per_sample", eb.max_events_per_sample)
  return ip.events_to_frames_packed(_dev_aligned(ev), off.cuda(), eb.format, T, wh, rs, event_base=base, **kw)


def _kernel_cases():
  rng = np.random.default_rng(11)
  T = 7
  # U16 on a 128 sensor: empty samples, N < T, N % T != 0, p outside {0, 1}, one hot pixel that saturates
  s = [_rand(rng, n, 0, 128, (0, 1, 7, -1)) for n in (3000, 0, 5, T, 20001, 1, 0, 777)]
  s[4][:4000, :2] = [9, 5]
  yield "u16", s, 128, T
  # U16 words on a 64 sensor: x up to 127 spills into the next row, y >= 64 falls outside the frame
  yield "u16_overflow", [_rand(rng, n, 0, 128) for n in (2000, 13, 0, 901)], 64, T
  # U32 words on a 128 sensor (the largest frame the shared-memory histogram holds at rs = 1), coordinates up to 2x
  # the sensor and far beyond it: flat-position overflow into the next row(s) and drops
  s = [_rand(rng, n, 0, 256, (0, 1, 3)) for n in (5000, 0, 6, 12345, 2)]
  s[0][:500, 0] = rng.integers(256, 4000, 500)           # x beyond the row -> a later row, or outside the frame
  s[3][:300, 1] = rng.integers(256, 2 ** 15, 300)        # y beyond the sensor -> dropped
  s[3][300:2300, :2] = [17, 100]                         # hot pixel
  yield "u32", s, 128, T


@pytest.mark.gpu
@pytest.mark.parametrize("rs", [1, 2, 4])
@pytest.mark.parametrize("case", ["u16", "u16_overflow", "u32"])
def test_packed_kernel_bit_exact(cuda_lib, case, rs):
  name, samples, wh, T = next(c for c in _kernel_cases() if c[0] == case)
  eb = ip.encode_events(samples, wh)
  assert eb.format == (_lib.EVENTS_U32 if name == "u32" else _lib.EVENTS_U16)
  rec = [eventsref.decode_events(eb.chunk(b, b + 1)[0].numpy(), eb.format) for b in range(eb.shape[0])]
  want32 = ref_events.batch_to_frames(rec, T, wh, rs)
  want8, nsat = ref_events.batch_to_frames(rec, T, wh, rs, saturate_u8=True)
  assert nsat > 0 or name == "u16_overflow"
  addrs, off = ip.concat_events(rec)
  B = eb.shape[0]
  for bound in (0, eb.max_events_per_sample, 10 ** 9):   # 32-bit counters / 16-bit packed counters / bound too large
    got32, _ = _packed(eb, 0, B, T, wh, rs, exact_int32=True, max_events_per_sample=bound)
    assert np.array_equal(got32.cpu().numpy(), want32), bound
    i32, _ = ip.events_to_frames(addrs.cuda(), off.cuda(), T, wh, rs, exact_int32=True, max_events_per_sample=bound)
    assert torch.equal(got32, i32), bound
    got8, sat = _packed(eb, 0, B, T, wh, rs, max_events_per_sample=bound)
    assert got8.dtype == torch.uint8 and np.array_equal(got8.cpu().numpy(), want8), bound
    assert int(sat.item()) == nsat, bound
  # any sample range, shipped as (words slice, offsets slice, event_base = offsets[b0])
  for b0, b1 in ((1, B), (2, 4), (B - 1, B), (1, B - 1)):
    got8, sat = _packed(eb, b0, b1, T, wh, rs)
    assert np.array_equal(got8.cpu().numpy(), want8[b0:b1]), (b0, b1)
    assert int(sat.item()) == ref_events.batch_to_frames(rec[b0:b1], T, wh, rs, saturate_u8=True)[1]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt_hi", [128, 512])
def test_packed_kernel_alignment_sweep(cuda_lib, fmt_hi):
  """Sample sizes 1 .. 40 back to back (and shifted by every start word): group bounds fall at every word index mod 8
  (U16) / mod 4 (U32), so every head / vector interior / tail split occurs."""
  rng = np.random.default_rng(fmt_hi)
  T, wh = 3, 128 if fmt_hi == 128 else 512
  samples = [_rand(rng, n, 0, fmt_hi) for n in range(1, 41)]
  eb = ip.encode_events(samples, wh)
  rec = [eventsref.decode_events(eb.chunk(b, b + 1)[0].numpy(), eb.format) for b in range(40)]
  rs = 1 if wh == 128 else 4
  want = ref_events.batch_to_frames(rec, T, wh, rs)
  for b0 in range(0, 9):
    got, _ = _packed(eb, b0, 40, T, wh, rs, exact_int32=True)
    assert np.array_equal(got.cpu().numpy(), want[b0:]), b0


@pytest.mark.gpu
def test_packed_entry_point_errors(cuda_lib):
  L = _lib.lib()
  ev = torch.zeros(64, dtype=torch.int16, device="cuda")
  off = torch.tensor([0, 64], dtype=torch.int64, device="cuda")
  fr = torch.empty((1, 2, 32, 32, 2), dtype=torch.uint8, device="cuda")
  call = lambda e, fmt, f, o=off: L.snnqp_events_to_frames_packed(e, fmt, _lib.ptr(o) if o is not None else None, 0, 1, 2,
                                                                  32, 1, 64, f, 0, None, None)
  assert call(ev.data_ptr(), _lib.EVENTS_U16, fr.data_ptr()) == 0
  torch.cuda.synchronize()
  for args, msg in (((None, _lib.EVENTS_U16, fr.data_ptr()), b"null pointer"),
                    ((ev.data_ptr(), _lib.EVENTS_U16, None), b"null pointer"),
                    ((ev.data_ptr(), 0, fr.data_ptr()), b"event_format"),
                    ((ev.data_ptr(), 3, fr.data_ptr()), b"event_format"),
                    ((ev.data_ptr() + 2, _lib.EVENTS_U16, fr.data_ptr()), b"events must be 16-byte aligned"),
                    ((ev.data_ptr(), _lib.EVENTS_U32, fr.data_ptr() + 8), b"frames must be 16-byte aligned")):
    assert call(*args) == 1 and msg in L.snnqp_last_error(), msg
  assert call(ev.data_ptr(), _lib.EVENTS_U16, fr.data_ptr(), None) == 1
  big = L.snnqp_events_to_frames_packed(ev.data_ptr(), _lib.EVENTS_U16, off.data_ptr(), 0, 1, 2, 512, 1, 64,
                                        fr.data_ptr(), 0, None, None)
  assert big == 3 and b"shared-memory histogram" in L.snnqp_last_error()
  with pytest.raises(ValueError):
    ip.events_to_frames_packed(ev.to(torch.int32), off, _lib.EVENTS_U16, 2, 32)


# ---- GPU: the engine --------------------------------------------------------------------------------------------------
def _device_frames(samples, T, wh, rs=1):
  addrs, off = ip.concat_events(samples)
  return ip.events_to_frames(addrs.cuda(), off.cuda(), T, wh, rs, exact_int32=True)[0]


@pytest.mark.gpu
def test_forward_host_events_equals_device_forward(cuda_lib):
  """Reference geometry, ragged chunk schedule (B = 45, chunk 37), one empty sample, a hot pixel, and a second call
  whose chunks need a larger events staging buffer than the first call's."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic
  bits, T, H, B = 8, 20, 128, 45
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  eng = CextNetEngine(pack_cextnet(v, bits, T, H, device="cuda"), chunk=37)
  host_out = torch.empty((B, 11), dtype=torch.float32).pin_memory()
  small = synthetic.make_events(B, T, H, seed=3, rate=0.03)
  big = synthetic.make_events(B, T, H, seed=4)
  big[7] = big[7][:0]                                   # an empty sample
  big[20][:6000, :2] = [64, 3]                          # a hot pixel: saturated cells
  for samples in (small, big):
    eb = ip.encode_events(samples, H)
    assert eb.format == _lib.EVENTS_U16
    f32 = _device_frames(samples, T, H)
    nsat_want = int((f32 > 255).sum())
    want = eng.forward(f32.clamp(max=255).to(torch.uint8)).cpu()
    nsat = torch.zeros((), dtype=torch.int64, device="cuda")
    eng.forward_host_events(eb, out_host=host_out, n_saturated=nsat)
    torch.cuda.synchronize()
    assert torch.equal(host_out, want)
    assert int(nsat.item()) == nsat_want
    assert torch.equal(eng.forward_host_events(eb).cpu(), want)
  assert nsat_want > 0
  cap = max(int(eb.offsets[b0 + n] - eb.offsets[b0]) for b0, n in eng.host_chunks(B))
  assert eng._workspace(B, 37)["ev"][0][0].numel() == cap
  with pytest.raises(ValueError):
    eng.forward_host_events(eb, resolution_scale=2)


@pytest.mark.gpu
def test_forward_host_events_u32_sensor256_rs2(cuda_lib):
  from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic
  bits, T, H, B = 8, 6, 128, 9
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=2)
  eng = CextNetEngine(pack_cextnet(v, bits, T, H, device="cuda"), chunk=4)
  samples = synthetic.make_events(B, T, 256, seed=5, rate=0.05)
  eb = ip.encode_events(samples, 256)
  assert eb.format == _lib.EVENTS_U32
  f32 = _device_frames(samples, T, 256, 2)
  want = eng.forward(f32.clamp(max=255).to(torch.uint8)).cpu()
  nsat = torch.zeros((), dtype=torch.int64, device="cuda")
  got = eng.forward_host_events(eb, resolution_scale=2, n_saturated=nsat).cpu()
  assert torch.equal(got, want) and int(nsat.item()) == int((f32 > 255).sum())


@pytest.mark.gpu
def test_evaluate_on_event_batches(cuda_lib):
  """eval.evaluate shards an EventBatch like a frames tensor (shape[0] and slicing)."""
  from snnquantprune_b200 import CextNetEngine, pack_cextnet, synthetic
  from snnquantprune_b200.eval import evaluate
  bits, T, H, B = 8, 4, 128, 10
  v = synthetic.make_variables(bits=bits, prune_percentage=0.5, T=T, H=H, seed=1)
  eng = CextNetEngine(pack_cextnet(v, bits, T, H, device="cuda"), chunk=4)
  samples = synthetic.make_events(B, T, H, seed=6)
  y = torch.as_tensor(synthetic.make_labels(B))
  frames = _device_frames(samples, T, H).clamp(max=255).to(torch.uint8)
  want = evaluate(eng.forward, [{"dvs_matrix": frames, "label": y}])
  got = evaluate(eng.forward_host_events, [{"dvs_matrix": ip.encode_events(samples, H), "label": y}])
  assert got == want and got["samples"] == B
