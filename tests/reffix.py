"""Helpers for the fixtures made by EXECUTING the unmodified reference
(tests/golden/make_from_reference.py): loading, input regeneration (digest
mismatch = failure, never a skip) and the north-star comparison rules."""
import hashlib
import json
import os

import numpy as np

from snnquantprune_b200 import synthetic

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
F32 = np.float32
BLOCKS = ("conv1", "conv2", "conv3", "conv4", "conv5", "dense1", "dense2")


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


def oracle_conv1_pooled(v, bits, frames):
  """Pooled conv1 spikes (T,B,H/2,W/2,C) uint8 of the integer-path oracle.  conv1 reads nothing but the frames, so
  no reference data goes into them."""
  from oracle import ref_int, ref_net
  c = ref_net.pack_network(v, bits, frames.shape[2])["conv"][0]
  s, _ = ref_int.spiking_conv3x3(np.ascontiguousarray(np.swapaxes(frames, 0, 1)), c["q"], c["scale"], c["bias"],
                                 pool=True, want=True, tau=2.0, v_th=1.0, v_reset=0.0)
  return s


def load_network(tag):
  """-> (fixture, meta, variables, frames).  The synthetic inputs are regenerated from the version-independent
  generator; a digest mismatch is a test FAILURE.

  The full-size fixtures do not store the reference's pooled conv1 spikes (1.3 MB of nearly incompressible bits)
  but the positions where they differ from the oracle's and their digest: they are rebuilt here from the oracle and
  must match the digest bit for bit."""
  fx = np.load(os.path.join(GOLD, f"from_reference_cextnet_{tag}.npz"))
  m = json.loads(str(fx["meta"]))
  v = synthetic.make_variables(bits=m["bits"], prune_percentage=m["prune"], T=m["T"], H=m["H"], seed=m["seed_w"],
                               num_classes=m["num_classes"], stable=True)
  fr = synthetic.make_frames(m["B"], m["T"], m["H"], m["H"], seed=m["seed_x"], stable=True)
  assert variables_digest(v) == m["variables_sha"], "synthetic variables differ from the ones the reference ran on"
  assert sha(fr) == m["frames_sha"], "synthetic frames differ from the ones the reference ran on"
  if "conv1_bits_diff" in fx:
    fx = dict(fx)
    s = oracle_conv1_pooled(v, m["bits"], fr).reshape(-1)
    s[fx["conv1_bits_diff"]] ^= 1
    fx["conv1_bits"] = np.packbits(s)
    assert sha(fx["conv1_bits"]) == str(fx["conv1_bits_sha"]), "rebuilt conv1 spikes differ from the reference's"
  return fx, m, v, fr


def ref_spikes(fx, name):
  """Reference spikes of a block as stored: conv1-3 pooled, conv4/conv5 un-pooled, dense full; (T,B,...) uint8."""
  if f"{name}_bits_shape" in fx:
    shape = tuple(int(x) for x in fx[f"{name}_bits_shape"])
  else:
    shape = tuple(int(x) for x in fx[f"{name}_shape"])
  n = int(np.prod(shape))
  return np.unpackbits(fx[f"{name}_bits"])[:n].reshape(shape)


def compare_block(fx, name, spikes_tb, u_final=None, counts_tbc=None, upstream_flips=0):
  """spikes_tb: (T,B,...) uint8 in the stored form (pooled for conv1-3).  Returns the number of flipped spikes.
  Rules (BASELINE.json north_star): flip rate <= 1e-4; final membranes within 1e-5 (relative to max(1, |u|)) on every
  neuron that is not downstream of a counted flip -- with no flips anywhere so far that is EVERY neuron."""
  ref = ref_spikes(fx, name)
  got = np.asarray(spikes_tb)
  if ref.ndim == 5:
    got = got[:, :, :ref.shape[2]]
  assert got.shape == ref.shape, (name, got.shape, ref.shape)
  flips = int((got != ref).sum())
  assert flips <= 1e-4 * ref.size + (0 if upstream_flips == 0 else 64 * upstream_flips), (name, flips, ref.size)
  if counts_tbc is not None and f"{name}_counts" in fx:
    dc = int(np.abs(np.asarray(counts_tbc, np.int64) - fx[f"{name}_counts"]).sum())
    assert dc <= 1e-4 * int(np.prod(fx[f"{name}_shape"])) + 64 * upstream_flips, (name, "spike counts", dc)
    if upstream_flips == 0 and flips == 0 and dc == 0 and ref.shape == tuple(fx[f"{name}_shape"]):
      pass
  if u_final is not None:
    uref = fx[f"{name}_uT"]
    ug = np.asarray(u_final, F32)
    if uref.ndim == 4:
      st = int(fx[f"{name}_uT_stride"])
      ug = ug[:, ::st, ::st, :]
    assert ug.shape == uref.shape, (name, ug.shape, uref.shape)
    bad = np.abs(ug - uref) > 1e-5 * np.maximum(1.0, np.abs(uref))
    if upstream_flips == 0 and flips == 0:
      assert not bad.any(), (name, "membrane", float(np.abs(ug - uref).max()))
    else:
      # a flipped spike perturbs its 3x3 (x channels) neighbourhood in the next layer and that neuron's later steps
      assert bad.sum() <= 2048 * (upstream_flips + flips), (name, int(bad.sum()), upstream_flips + flips)
  return flips


def logits_tolerance(T, group, flips_total):
  """One flipped output spike moves a logit by 1 / (T * group) (vote, models.py:253-255)."""
  return 1e-6 + (1.0 / (T * group)) * min(flips_total, 16)
