"""Generate golden fixtures by EXECUTING THE UNMODIFIED REFERENCE SOURCES.

    python tests/golden/make_from_reference.py [--full]

Runs in the build container only (it reads /root/reference); the fixtures it
writes (tests/golden/from_reference_*.npz) travel to the GPU box, this script
and the shim do not need to.  `jax`, `flax.linen` and `ml_collections` are the
numpy-backed stand-ins of tests/golden/ref_shim (see its README for what is
reference code and what is restated third-party arithmetic).  Executed
reference code:

  quant.py                      DuQ (:428-469), prune (:472-491), round_ewgs (:88-90),
                                gaussian_init / max_init (:296-309)
  spiking_learning.py           atan (:221-224), multi_step_LIF (:390-416),
                                SpikingBlock + initialize_carry (:441-472)
  flax_qconv.py, flax_qdense.py QuantConv / QuantDense __call__
  examples/tcja/models.py       CextNet.__call__ incl. TCJA, pools, flatten, vote
  examples/train_inpt_spikingjelly.py:147-229
                                mask construction (local + global) and DuQ
                                calibration -- exec'd from the source text,
                                because it is inline in train_and_evaluate

Inputs come from snnquantprune_b200.synthetic with stable=True (integer-hash
generator: identical streams on any numpy), so tests regenerate them and FAIL
on a digest mismatch instead of skipping.
"""
import argparse
import hashlib
import importlib.util
import json
import os
import sys
import textwrap
import time
from functools import partial

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
F32 = np.float32


def load_reference():
  sys.path[:0] = [os.path.join(HERE, "ref_shim"), REF, os.path.join(REF, "examples", "tcja"),
                  os.path.join(REF, "examples")]
  import quant, spiking_learning, flax_qconv, flax_qdense  # noqa: E401
  spec = importlib.util.spec_from_file_location("ref_tcja_models", os.path.join(REF, "examples", "tcja", "models.py"))
  models = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(models)
  for m in (quant, spiking_learning, flax_qconv, flax_qdense, models):
    assert os.path.realpath(m.__file__).startswith(REF + "/"), m.__file__
  return quant, spiking_learning, flax_qconv, flax_qdense, models


def sha(*arrays) -> str:
  h = hashlib.sha256()
  for a in arrays:
    h.update(np.ascontiguousarray(a).tobytes())
  return h.hexdigest()


def variables_digest(v) -> str:
  arrs = []
  for name in sorted(v["params"].keys()):
    lay = v["params"][name]
    if "kernel" in lay:
      arrs += [lay["kernel"], lay["prune_0"]["mask"], lay["DuQ_0"]["a"], lay["DuQ_0"]["c"]]
    else:
      arrs += [lay["scale"], lay["bias"], v["batch_stats"][name]["mean"], v["batch_stats"][name]["var"]]
  return sha(*[np.asarray(a, F32) for a in arrs])


# ------------------------------------------------------------------ mask construction / calibration
def reference_masks_and_calibration(params, bits, p, prune_global):
  """exec of examples/train_inpt_spikingjelly.py:147-229 on a params tree
  {name: {'kernel', 'DuQ_0': {'a','c'}, 'prune_0': {'mask'}}, 'BatchNorm_i': {...}}."""
  import jax
  import jax.numpy as jnp
  import ml_collections
  import quant
  src = open(os.path.join(REF, "examples", "train_inpt_spikingjelly.py")).read().split("\n")
  i0 = next(i for i, l in enumerate(src) if "def update_prune_mask" in l)
  i1 = next(i for i, l in enumerate(src) if "Successfully restored model" in l)
  assert (i0 + 1, i1) == (147, 229), (i0, i1)           # source lines 147-229
  code = textwrap.dedent("\n".join(src[i0:i1]))

  class _Log:
    @staticmethod
    def info(*a):
      pass

  class _State:
    pass

  config = ml_collections.ConfigDict()
  config.prune_percentage = p             # (sic) the local branch reads config.prune_percentage
  config.quant = ml_collections.ConfigDict()
  config.quant.prune_percentage = p
  config.quant.prune_global = prune_global
  config.quant.bits = bits
  config.quant.init_fn = quant.gaussian_init
  config.quant.start_epoch = -1
  state = _State()
  state.params = {"params": params}
  g = {"np": np, "jnp": jnp, "jax": jax, "config": config, "state": state, "logging": _Log}
  exec(compile(code, "train_inpt_spikingjelly.py:147-229", "exec"), g)
  return state.params["params"]


def raw_tree(v):
  """kernels only, DuQ/prune at their flax initial values (a = c = -1, mask = 1)."""
  out = {}
  for n, lay in v["params"].items():
    if "kernel" in lay:
      out[n] = {"kernel": np.array(lay["kernel"], F32), "DuQ_0": {"a": np.full((1,), -1, F32), "c": np.full((1,), -1, F32)},
                "prune_0": {"mask": np.ones(lay["kernel"].shape, F32)}}
    else:
      out[n] = {k: np.array(a, F32) for k, a in lay.items()}
  return out


# ------------------------------------------------------------------ elementwise ops
def ops_fixture(quant, sl, flax_qconv, flax_qdense):
  import ml_collections
  fx = {}
  rng = np.random.default_rng(11)
  w = (rng.standard_normal(257) * 0.3).astype(F32)
  edge = np.array([0.0, -0.0, 1e-9, -1e-9, 0.5, -0.5, 1.0, -1.0, 2.0, -2.0, 1.0000001, 0.99999994], F32)
  halves = np.concatenate([(np.arange(-7, 7) + 0.5) / 7, (np.arange(-127, 127) + 0.5) / 127]).astype(F32)
  w = np.concatenate([w, edge, halves])
  fx["duq_w"] = w
  cases = []
  for bits in (2, 3, 4, 8):
    for a, c in ((1.0, 1.0), (0.37, 0.41), (float(quant.gaussian_init(w, bits, True)),) * 2):
      mod = quant.DuQ(bits=bits, round_fn=quant.round_ewgs)
      y = mod.apply({"params": {"a": np.array([a], F32), "c": np.array([c], F32)}}, w)
      assert y.dtype == F32
      fx[f"duq_b{bits}_case{len(cases)}"] = y
      cases.append({"bits": bits, "a": a, "c": c, "key": f"duq_b{bits}_case{len(cases)}"})
  # pass-through forms (quant.py:453-454, 469)
  fx["duq_passthrough_a"] = quant.DuQ(bits=4).apply({"params": {"a": np.array([-1], F32), "c": np.array([-1], F32)}}, w)
  fx["duq_passthrough_bits"] = quant.DuQ(bits=-1).apply({"params": {}}, w)
  mask = (rng.uniform(size=w.shape) > 0.4).astype(F32)
  fx["prune_mask"] = mask
  fx["prune_out"] = quant.prune().apply({"params": {"mask": mask}}, w)
  # calibrators
  cal_in = {"randn": (rng.standard_normal((3, 3, 8, 16)) * 0.2 + 0.01).astype(F32),
            "zeros": np.zeros((4, 5), F32),
            "nonpos": -np.abs(rng.standard_normal(50)).astype(F32) * (np.arange(50) > 0),   # max(x) == 0, x != 0
            "big": (rng.standard_normal(20000) * 0.05).astype(F32)}
  for k, x in cal_in.items():
    fx[f"cal_in_{k}"] = np.asarray(x, F32)
    for bits in (2, 8):
      fx[f"cal_gauss_{k}_b{bits}"] = np.asarray(quant.gaussian_init(np.asarray(x, F32), bits, True), F32)
      fx[f"cal_max_{k}_b{bits}"] = np.asarray(quant.max_init(np.asarray(x, F32), bits, True), F32)
  # atan forward (Heaviside, >= inclusive)
  xs = np.array([0.0, -0.0, 1e-30, -1e-30, 1.0, -1.0, 5.9604645e-08, -5.9604645e-08], F32)
  fx["atan_in"], fx["atan_out"] = xs, sl.atan(xs)
  # multi_step_LIF over T steps, incl. exact threshold ties
  lif_cases = []
  for ci, (tau, vth, vr) in enumerate(((2.0, 1.0, 0.0), (2.0, 1.0, 0.0), (1.7, 0.8, 0.1))):
    T, n = 8, 1024
    x = (rng.standard_normal((T, n)) * 0.9 + 0.6).astype(F32)
    u0 = (rng.uniform(-1.0, 1.5, n)).astype(F32) if ci else np.zeros(n, F32)
    if ci == 1:
      u0[:8] = [0.5, 0.0, 0.25, 0.75, -1.0, 0.9999999, 1.5, 0.0]
      x[0, :8] = [1.5, 2.0, 1.75, 1.25, 3.0, 1.0000001, 0.5, 1.9999999]      # un == 1 (ties) and neighbours
    mod = sl.multi_step_LIF(tau=tau, spike_fn=sl.atan, v_threshold=vth, v_reset=vr)
    u = u0.copy()
    us, ss = [], []
    for t in range(T):
      u, s = mod.apply({}, u.copy(), x[t])
      assert u.dtype == F32 and s.dtype == F32
      us.append(u); ss.append(s)
    fx[f"lif{ci}_x"], fx[f"lif{ci}_u0"] = x, u0
    fx[f"lif{ci}_u"], fx[f"lif{ci}_s"] = np.stack(us), np.stack(ss).astype(np.uint8)
    lif_cases.append({"tau": tau, "v_threshold": vth, "v_reset": vr})
  # LIF on a grid of exactly representable pre-activations x = count * 2^-6 - 0.25 (count = uint8): a fused GPU
  # block with an identity centre tap reproduces exactly these x, so its LIF can be held to the reference's
  # bit for bit (folded fmaf == unfused multiply-add on this grid).  Layout (T, B=1, H=8, W=16, C=128).
  cnt = rng.integers(0, 256, (8, 1, 8, 16, 128)).astype(np.uint8)
  cnt[:, :, :, :, :8] = np.minimum(cnt[:, :, :, :, :8], 90)          # some channels stay mostly sub-threshold
  xg = (cnt.astype(F32) * F32(2.0 ** -6) - F32(0.25)).astype(F32)
  mod = sl.multi_step_LIF(tau=2.0, spike_fn=sl.atan)
  u = np.zeros(xg.shape[1:], F32)
  sg = []
  for t in range(xg.shape[0]):
    u, s_ = mod.apply({}, u.copy(), xg[t])
    sg.append(s_)
  fx["lifgrid_counts"], fx["lifgrid_uT"] = cnt, u
  fx["lifgrid_bits"] = np.packbits(np.stack(sg).astype(np.uint8).reshape(-1))
  # QuantConv / QuantDense standalone (layer facades): 3x3 pad 1, 1-D k=4 'SAME', dense
  cfg = ml_collections.ConfigDict()
  cfg.bits = 4
  cfg.g_scale = 0.0
  cfg.weight = partial(quant.DuQ, round_fn=quant.round_ewgs)
  cfg.prune_percentage = 0.5
  sys.path.insert(0, ROOT)
  from snnquantprune_b200.synthetic import StableRNG
  def layer_case(tag, mod, x, kshape, seed):
    # kernel / mask are regenerated by the tests from StableRNG(seed) (not stored: 590 KB for the 3x3x128x128 case)
    srng = StableRNG(seed)
    k = (srng.standard_normal(kshape) * 0.3).astype(F32)
    m = (srng.uniform(0, 1, kshape) > 0.5).astype(F32)
    ac = np.asarray(quant.gaussian_init(k, 4, True), F32).reshape(1)
    y = mod.apply({"params": {"kernel": k, "DuQ_0": {"a": ac, "c": ac * F32(1.25)}, "prune_0": {"mask": m}}}, x.astype(F32))
    fx[f"{tag}_x"], fx[f"{tag}_a"], fx[f"{tag}_c"] = x, ac, ac * F32(1.25)
    fx[f"{tag}_kshape"], fx[f"{tag}_seed"], fx[f"{tag}_ksha"] = np.array(kshape), np.array(seed), np.array(sha(k, m))
    fx[f"{tag}_y"] = np.asarray(y, F32)
  layer_case("qconv3x3", flax_qconv.QuantConv(features=128, kernel_size=(3, 3), padding=((1, 1), (1, 1)), use_bias=False,
                                             config=cfg, bits=4, g_scale=0.0),
             rng.integers(0, 2, (1, 8, 16, 128)).astype(np.uint8), (3, 3, 128, 128), 101)
  layer_case("qconv1d", flax_qconv.QuantConv(features=5, kernel_size=[4], padding="SAME", use_bias=False, config=cfg,
                                            bits=4, g_scale=0.0),
             (rng.integers(0, 65, (2, 9, 3)) / 64).astype(F32), (4, 3, 5), 102)
  layer_case("qdense", flax_qdense.QuantDense(110, use_bias=False, config=cfg, bits=4, g_scale=0.0),
             rng.integers(0, 2, (6, 512)).astype(np.uint8), (512, 110), 103)
  # mask construction on a toy tree, local and global, p = 0.3 / 0.75
  toy = {"params": {"QuantConv_0": {"kernel": (rng.standard_normal((3, 3, 2, 8))).astype(F32)},
                    "QuantConv_1": {"kernel": (rng.standard_normal((4, 5, 5)) * 0.5).astype(F32)},
                    "QuantConv_10": {"kernel": (rng.standard_normal((7,)) * 2).astype(F32)},   # sorts before _2
                    "QuantConv_2": {"kernel": (rng.standard_normal((3, 3, 8, 8)) * 0.1).astype(F32)},
                    "QuantDense_0": {"kernel": (rng.standard_normal((32, 10)) * 0.7).astype(F32)},
                    "BatchNorm_0": {"scale": np.ones(8, F32), "bias": np.zeros(8, F32)}}}
  for n, lay in toy["params"].items():
    if "kernel" in lay:
      fx[f"toy_kernel_{n}"] = lay["kernel"]
  for gl in (False, True):
    for p in (0.3, 0.75):
      out = reference_masks_and_calibration(raw_tree(toy), 8, p, gl)
      for n, lay in out.items():
        if "kernel" in lay:
          tag = f"toy_{'global' if gl else 'local'}_p{int(p * 100)}_{n}"
          fx[tag + "_mask"] = np.asarray(lay["prune_0"]["mask"], F32)
          fx[tag + "_a"] = np.asarray(lay["DuQ_0"]["a"], F32).reshape(-1)
          assert np.array_equal(np.asarray(lay["DuQ_0"]["a"]), np.asarray(lay["DuQ_0"]["c"]))
  fx["meta"] = np.array(json.dumps({"duq_cases": cases, "lif_cases": lif_cases,
                                    "toy_names": [n for n in toy["params"] if n.startswith("Quant")]}))
  return fx


# ------------------------------------------------------------------ whole network through the reference's CextNet
def network_fixture(quant, sl, models, bits, p, T, H, B, seed_w, seed_x, num_classes=11, full=False):
  import flax.linen as nn
  import jax.nn
  import ml_collections
  sys.path[:0] = [ROOT, os.path.dirname(HERE)]
  from snnquantprune_b200 import synthetic
  v = synthetic.make_variables(bits=bits, prune_percentage=p, T=T, H=H, seed=seed_w, num_classes=num_classes, stable=True)
  frames = synthetic.make_frames(B, T, H, H, seed=seed_x, stable=True)

  # masks + DuQ calibration by the reference's own code; the product's host code must have produced the same
  ref_tree = reference_masks_and_calibration(raw_tree(v), bits, p, True)
  for n, lay in v["params"].items():
    if "kernel" in lay:
      assert np.array_equal(lay["prune_0"]["mask"], np.asarray(ref_tree[n]["prune_0"]["mask"], F32)), n
      assert np.array_equal(lay["DuQ_0"]["a"], np.asarray(ref_tree[n]["DuQ_0"]["a"], F32).reshape(-1)), n
      assert np.array_equal(lay["DuQ_0"]["c"], np.asarray(ref_tree[n]["DuQ_0"]["c"], F32).reshape(-1)), n

  config = ml_collections.ConfigDict()
  config.channels = 128
  config.dropout = 0.5
  config.neuron_dynamics = partial(sl.multi_step_LIF, spike_fn=sl.atan, tau=2.0)   # prune_quant_joint.py:27
  config.quant = ml_collections.ConfigDict()
  config.quant.bits = bits
  config.quant.g_scale = 5e-3
  config.quant.weight = partial(quant.DuQ, round_fn=quant.round_ewgs)              # prune_quant_joint.py:56
  config.quant.prune_percentage = p
  model = models.CextNet(num_classes=num_classes, dtype=F32, config=config)

  blocks, atts = [], []
  nn.SCAN_HOOKS.append(lambda mod, xs, out: blocks.append((np.asarray(out[0]), np.asarray(out[1]))))
  orig_sigmoid = jax.nn.sigmoid
  def rec_sigmoid(x):
    y = orig_sigmoid(x)
    atts.append(np.asarray(y))
    return y
  jax.nn.sigmoid = rec_sigmoid
  t0 = time.time()
  try:
    ref_vars = {"params": {k: dict(d) for k, d in ref_tree.items()}, "batch_stats": v["batch_stats"]}
    (logits, _), sown = model.apply(ref_vars, frames.astype(F32), None, False, None, mutable=["intermediates"])
  finally:
    nn.SCAN_HOOKS.clear()
    jax.nn.sigmoid = orig_sigmoid
  assert len(blocks) == 7 and len(atts) == 2
  names = ["conv1", "conv2", "conv3", "conv4", "conv5", "dense1", "dense2"]
  fx = {"logits": np.asarray(logits, F32), "att4": atts[0].astype(F32), "att5": atts[1].astype(F32)}
  rates = {}
  for n, (uT, s) in zip(names, blocks):
    s8 = (s != 0).astype(np.uint8)
    assert np.array_equal(s8.astype(F32), s)
    rates[n] = float(s8.mean())
    fx[f"{n}_sha"] = np.array(sha(np.packbits(s8.reshape(-1))))
    fx[f"{n}_shape"] = np.array(s8.shape)
    if s8.ndim == 5:
      fx[f"{n}_counts"] = s8.sum(axis=(2, 3), dtype=np.int32)          # (T,B,C)
      pooled = s8.reshape(s8.shape[0], s8.shape[1], s8.shape[2] // 2, 2, s8.shape[3] // 2, 2, -1).max(axis=(3, 5))
      keep = s8 if n in ("conv4", "conv5") else pooled                  # what the next layer / TCJA consumes
      fx[f"{n}_bits"] = np.packbits(keep.reshape(-1))      # complete: per-layer teacher forcing needs every input spike
      fx[f"{n}_bits_shape"] = np.array(keep.shape)
      if full and n == "conv1":
        # stored as the difference to the oracle's conv1 and the digest (tests/reffix.py load_network rebuilds it):
        # the bits themselves would take the file over 1 MB
        import reffix
        diff = np.flatnonzero(reffix.oracle_conv1_pooled(v, bits, frames).reshape(-1) != keep.reshape(-1))
        fx[f"{n}_bits_sha"] = np.array(sha(fx.pop(f"{n}_bits")))
        fx[f"{n}_bits_diff"] = diff.astype(np.int64)
      st = max(1, uT.shape[1] // 8)                                  # 8 x 8 sub-grid of final membranes
      fx[f"{n}_uT"] = np.ascontiguousarray(uT[:, ::st, ::st, :], F32)
      fx[f"{n}_uT_stride"] = np.array(st)
    else:
      fx[f"{n}_bits"] = np.packbits(s8.reshape(-1))
      fx[f"{n}_uT"] = np.asarray(uT, F32)
  dens = {k: float(np.asarray(val[-1])) for k, val in sown.get("intermediates", {}).items()}
  fx["meta"] = np.array(json.dumps(dict(
      bits=bits, prune=p, T=T, H=H, B=B, seed_w=seed_w, seed_x=seed_x, num_classes=num_classes, stable=True,
      variables_sha=variables_digest(v), frames_sha=sha(frames), rates=rates, sown=dens,
      seconds=round(time.time() - t0, 1))))
  print(f"  b{bits} p{p} T{T} H{H} B{B}: {time.time() - t0:.1f} s, rates {rates}")
  return fx


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--full", action="store_true", help="also the H=128 / T=20 configurations (minutes)")
  ap.add_argument("--only-full", action="store_true")
  args = ap.parse_args()
  quant, sl, qc, qd, models = load_reference()
  if not args.only_full:
    np.savez_compressed(os.path.join(HERE, "from_reference_ops.npz"), **ops_fixture(quant, sl, qc, qd))
    for tag, cfg in (("T4_H32_b8_p50", (8, 0.5, 4, 32, 2, 1, 0)), ("T3_H32_b4_p80", (4, 0.8, 3, 32, 2, 5, 7)),
                     ("T3_H32_b2_p90", (2, 0.9, 3, 32, 2, 6, 8))):
      np.savez_compressed(os.path.join(HERE, f"from_reference_cextnet_{tag}.npz"),
                          **network_fixture(quant, sl, models, *cfg))
    # configs[3] geometry: T = 10, 10 classes (Dense2 -> 100), reduced resolution
    np.savez_compressed(os.path.join(HERE, "from_reference_cextnet_T10_H32_b8_p50_c10.npz"),
                        **network_fixture(quant, sl, models, 8, 0.5, 10, 32, 2, 9, 10, num_classes=10))
  if args.full or args.only_full:
    for tag, cfg in (("T20_H128_b8_p50", (8, 0.5, 20, 128, 1, 1, 0)), ("T20_H128_b4_p80", (4, 0.8, 20, 128, 1, 5, 7)),
                     ("T20_H128_b2_p90", (2, 0.9, 20, 128, 1, 6, 8))):
      np.savez_compressed(os.path.join(HERE, f"from_reference_cextnet_{tag}.npz"),
                          **network_fixture(quant, sl, models, *cfg, full=True))
  print("from-reference fixtures written")


if __name__ == "__main__":
  main()
