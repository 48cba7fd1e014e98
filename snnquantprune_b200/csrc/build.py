"""Build libsnnqp.so (the C-ABI library) in-tree with nvcc for sm_100a.

    python snnquantprune_b200/csrc/build.py [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(os.path.dirname(HERE), os.environ.get("SNNQP_BUILD_NAME", "libsnnqp.so"))
SOURCES = ["runtime.cu", "pack.cu", "simt.cu", "umma_conv_t.cu", "umma_conv1.cu", "umma_conv1_tc.cu", "umma_att.cu", "diag.cu", "frames.cu", "plain.cu", "api.cu", "xla_ffi_shim.cc"]
HEADERS = ["common.cuh", "ptx.cuh", "tmap.cuh", "epilogue.cuh", os.path.join(ROOT, "include", "snnqp.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
# XLA FFI handlers (xla_ffi_shim.cc) compile for real where jaxlib's headers are: SNNQP_XLA_INCLUDE=<dir holding xla/ffi/api/ffi.h>
XLA_INC = ["-I", os.environ["SNNQP_XLA_INCLUDE"]] if os.environ.get("SNNQP_XLA_INCLUDE") else []
if os.environ.get("SNNQP_MMA_WARPS"):       # experiment: MMA-issuing warps of the 3x3 tile kernel (1 or 2)
  FLAGS.append("-DSNNQP_MMA_WARPS=" + os.environ["SNNQP_MMA_WARPS"])
if os.environ.get("SNNQP_T_TAPS"):          # experiment: weight taps of the 3x3 tile kernel resident in TMEM
  FLAGS.append("-DSNNQP_T_TAPS=" + os.environ["SNNQP_T_TAPS"])
if os.environ.get("SNNQP_C1_SUSPEND"):      # experiment: hardware-suspended producer waits in conv1 (tools/run_r2_gpu16.sh)
  FLAGS.append("-DSNNQP_C1_SUSPEND")
if os.environ.get("SNNQP_EXP_WARPS"):       # experiment: number of expander warps of the bit-packed tile kernel
  FLAGS.append("-DSNNQP_EXP_WARPS=" + os.environ["SNNQP_EXP_WARPS"])
if os.environ.get("SNNQP_BISECT"):          # debug-only bisection switches inside the hot loops (tools/)
  FLAGS.append("-DSNNQP_C1_BISECT")


def _stale() -> bool:
  if not os.path.exists(OUT):
    return True
  t = os.path.getmtime(OUT)
  deps = [os.path.join(HERE, s) for s in SOURCES] + [
      h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
  deps.append(os.path.abspath(__file__))
  return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
  if not force and not _stale():
    return OUT
  objs = []
  build_dir = os.path.join(HERE, "build")
  os.makedirs(build_dir, exist_ok=True)
  procs = []
  for s in SOURCES:
    o = os.path.join(build_dir, s.replace(".cu", ".o").replace(".cc", ".o"))
    objs.append(o)
    cmd = [NVCC, *FLAGS, "-I", os.path.join(ROOT, "include"), "-I", HERE, *XLA_INC, "-c",
           os.path.join(HERE, s), "-o", o]
    procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
  logs = []
  for s, pr in procs:
    out, _ = pr.communicate()
    logs.append(f"==== {s}\n{out}")
    if pr.returncode != 0:
      sys.stderr.write("\n".join(logs))
      raise RuntimeError(f"nvcc failed on {s}")
  with open(os.path.join(build_dir, "ptxas.log"), "w") as f:
    f.write("\n".join(logs))
  if verbose:
    print("\n".join(logs))
  cmd = [NVCC, "-shared", "-o", OUT, *objs, "-lcudart"]
  subprocess.run(cmd, check=True)
  return OUT


if __name__ == "__main__":
  print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
