"""Plain-numpy decoder of the packed event words (include/snnqp.h, SNNQP_EVENTS_U16 / SNNQP_EVENTS_U32), written from
the header's bit layouts and independent of the product's encoder: the tests decode what
``input_pipeline.encode_events`` produced and integrate it with ``oracle/ref_events.py``."""
import numpy as np

U16, U32 = 1, 2          # SNNQP_EVENTS_U16, SNNQP_EVENTS_U32


def decode_events(words: np.ndarray, format: int) -> np.ndarray:
  """words (N,) of 16- or 32-bit event words (any signedness: only the bits count) -> int64 (N, 3) (x, y, p)."""
  if format == U16:
    w = np.asarray(words).view(np.uint16).astype(np.int64)
    assert not (w & (1 << 14)).any(), "bit 14 of a U16 word is zero"
    return np.stack([w & 0x7F, (w >> 7) & 0x7F, w >> 15], 1)
  if format == U32:
    w = np.asarray(words).view(np.uint32).astype(np.int64)
    assert not (w & (1 << 30)).any(), "bit 30 of a U32 word is zero"
    return np.stack([w & 0x7FFF, (w >> 15) & 0x7FFF, w >> 31], 1)
  raise ValueError(f"unknown event format {format}")
