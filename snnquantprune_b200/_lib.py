"""ctypes binding of the C-ABI in include/snnqp.h (libsnnqp.so, built in-tree by
``snnquantprune_b200/csrc/build.py``).  There is no CPU fallback: importing the
package works without a GPU, but every compute entry point fails loudly when
the library or an sm_100 device is missing."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SNNQP_LIB: developer switch for same-box A/B timing of two builds (tools/); the product path is the in-tree .so
LIB_PATH = os.environ.get("SNNQP_LIB") or os.path.join(_HERE, "libsnnqp.so")

ABI_VERSION = 4          # include/snnqp.h SNNQP_ABI_VERSION (block params carry x_format / y_format / lif_mode)
IMPL_AUTO, IMPL_SIMT, IMPL_TCGEN05 = 0, 1, 2
SPIKES_U8, SPIKES_BITS = 0, 1
LIF_EXACT, LIF_FAST, LIF_TENSOR = 0, 1, 2
EVENTS_U16, EVENTS_U32 = 1, 2     # packed event words (snnqp_events_to_frames_packed)


class SnnqpError(RuntimeError):
  def __init__(self, code: int, msg: str):
    super().__init__(f"snnqp error {code}: {msg}")
    self.code = code


class BlockParams(C.Structure):
  _fields_ = [
      ("T", C.c_int32), ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
      ("Cin", C.c_int32), ("Cout", C.c_int32),
      ("x_stride_t", C.c_int64), ("x_stride_b", C.c_int64),
      ("y_stride_t", C.c_int64), ("y_stride_b", C.c_int64),
      ("att_stride_t", C.c_int64), ("att_stride_b", C.c_int64),
      ("att_mod", C.c_int32),
      ("tau", C.c_float), ("v_threshold", C.c_float), ("v_reset", C.c_float),
      ("pool", C.c_int32), ("impl", C.c_int32),
      ("x_format", C.c_int32), ("y_format", C.c_int32), ("lif_mode", C.c_int32),
      ("y_popcount", C.c_void_p),
  ]


_vp, _i, _i64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
_BP = C.POINTER(BlockParams)

# name -> (restype, argtypes); every symbol include/snnqp.h declares
SIGNATURES = {
    "snnqp_abi_version": (_i, []),
    "snnqp_last_error": (C.c_char_p, []),
    "snnqp_device_ok": (_i, []),
    "snnqp_launch_count": (_i64, [_i]),
    "snnqp_duq_forward": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _vp, _vp]),
    "snnqp_pack_levels": (_i, [_vp, _vp, _vp, _i, _i64, _vp, _vp]),
    "snnqp_conv3x3_blob_bytes": (_i64, [_i, _i]),
    "snnqp_pack_conv1": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "snnqp_pack_conv3x3": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "snnqp_pack_matrix": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp, _vp]),
    "snnqp_fold_affine": (_i, [_vp, _i, _d, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp, _vp]),
    "snnqp_conv3x3_slab_bitmap": (_i, [_vp, _i, _i, _vp, _vp]),
    "snnqp_spiking_conv3x3_fwd": (_i, [_BP, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "snnqp_spiking_conv3x3_counts_fwd": (_i, [_BP, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "snnqp_spiking_dense_fwd": (_i, [_BP, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "snnqp_qconv3x3_fwd": (_i, [_BP, _vp, _vp, _vp, _vp, _vp, _vp]),
    "snnqp_tcja_fwd": (_i, [_BP, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "snnqp_maxpool2_fwd": (_i, [_BP, _vp, _vp, _vp]),
    "snnqp_vote_fwd": (_i, [_vp, _i, _i, _i, _i, _i64, _i64, _vp, _vp]),
    "snnqp_eval_metrics": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "snnqp_events_to_frames": (_i, [_vp, _vp, _i, _i, _i, _i, _i64, _vp, _i, _vp, _vp]),
    "snnqp_events_to_frames_packed": (_i, [_vp, _i, _vp, _i64, _i, _i, _i, _i, _i64, _vp, _i, _vp, _vp]),
    "snnqp_slice_nonzeros": (_i, [_vp, _i, _i64, _i64, _vp, _vp]),
    "snnqp_slice_popcount": (_i, [_vp, _i, _i64, _i64, _vp, _vp]),
    "snnqp_tile_skip_stats": (_i, [_vp, _vp, _i]),
    "snnqp_qlinear_fwd": (_i, [_vp, _i, _vp, _vp, _i64, _i, _i, _vp, _vp]),
    "snnqp_expand_frames_zsf": (_i, [_vp, _vp, _vp, C.c_uint32, _i64, _i, _vp, _vp]),
    "snnqp_diag_imma_peak": (_i, [_i, _i, C.POINTER(C.c_double), _vp]),
}

_lib = None


def lib() -> C.CDLL:
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      raise RuntimeError(
          f"{LIB_PATH} is missing: build it with "
          "`python snnquantprune_b200/csrc/build.py` (there is no CPU fallback)")
    l = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
      fn = getattr(l, name)
      fn.restype = res
      fn.argtypes = args
    if l.snnqp_abi_version() != ABI_VERSION:
      raise RuntimeError("libsnnqp.so ABI version mismatch")
    _lib = l
  return _lib


def check(rc: int) -> None:
  if rc != 0:
    raise SnnqpError(rc, lib().snnqp_last_error().decode())


def ptr(t) -> int:
  """Device pointer of a torch CUDA tensor (None -> NULL)."""
  if t is None:
    return None
  if not t.is_cuda:
    raise ValueError("snnqp entry points take CUDA tensors only (no CPU fallback)")
  return t.data_ptr()


def stream() -> int:
  import torch
  return torch.cuda.current_stream().cuda_stream
