"""Device engine for the TCJA-SNN (``CextNet``) eval forward: one pass of the hot
path = the sequence of fused C-ABI calls below, all on the caller's stream.

Graph (reference examples/tcja/models.py:101-257, eval branch):
  3 x [QuantConv3x3 -> BN -> LIF -> maxpool2]            one fused launch per block
  2 x [QuantConv3x3 -> BN -> LIF -> TCJA -> maxpool2]    fused conv block (pooled spikes + per-(b,t,c)
                                                         spike counts), then the attention kernel
  flatten (folded into dense1 weights) -> [QuantDense -> LIF] x 2 -> vote

Activations stay on the device as uint8 spikes, batch-major [B][T][H][W][C]
(the reference's input layout, examples/train_inpt_spikingjelly.py:300-305), so
a batch shard is one contiguous slab.  The TCJA output ``x_seq * att`` is never
materialised: att > 0 is constant over (h, w), so maxpool(att * s) =
att * maxpool(s) and the consumers take the (pooled spikes, att) pair; the TCJA
mean over (h, w) only needs the spike counts, which the conv epilogue
accumulates.  The first three blocks run per ``chunk`` samples (their
activations then stay L2-resident between launches); the small tail layers run
once over the whole batch so that they fill the machine.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _lib
from ._lib import BlockParams
from .pack import PackedCextNet


class _HeadPipe:
  """Chunk pipeline of the head (conv1 -> conv2 -> conv3).  Un-fused: the three launches per chunk.  Fused
  (``engine.fused_head``): conv1 of the pushed chunk shares one persistent kernel with conv2 of the previous chunk
  (two s1 buffers in flight); ``finish`` drains the last chunk."""

  def __init__(self, eng, ws, collect=None):
    self.eng, self.ws, self.collect = eng, ws, collect
    self.fused = eng.fused_head and collect is None
    self.prev = None
    self.i = 0

  def _s1(self, i):
    return self.ws["s1"] if (i & 1) == 0 else self.ws["s1b"]

  def push(self, frames_chunk, b0, n):
    eng, ws = self.eng, self.ws
    if not self.fused:
      eng._head(frames_chunk, b0, n, ws, self.collect)
      return
    H, C = eng.pk.H, eng.pk.channels
    pb0, pn = self.prev if self.prev else (0, 0)
    eng._head_fused(frames_chunk, n, self._s1(self.i), self._s1(self.i - 1), pn, ws["s2"])
    if pn:
      eng._conv(2, ws["s2"][:pn], ws["s3"][pb0:pb0 + pn], pn, H // 4, C, 1)
    self.prev = (b0, n)
    self.i += 1

  def finish(self):
    if not self.fused or not self.prev:
      return
    eng, ws = self.eng, self.ws
    H, C = eng.pk.H, eng.pk.channels
    pb0, pn = self.prev
    eng._head_fused(None, 0, None, self._s1(self.i - 1), pn, ws["s2"])
    eng._conv(2, ws["s2"][:pn], ws["s3"][pb0:pb0 + pn], pn, H // 4, C, 1)
    self.prev = None


class CextNetEngine:
  def __init__(self, packed: PackedCextNet, impl: int = _lib.IMPL_AUTO,
               tau: float = 2.0, v_threshold: float = 1.0, v_reset: float = 0.0,
               chunk: int = 296, device="cuda", lif_mode: int = _lib.LIF_TENSOR,
               packed_spikes: Optional[bool] = None, fused_head: Optional[bool] = None,
               track_densities: bool = False):
    """``packed_spikes``: conv1 -> conv2 -> conv3 -> conv4 exchange bit-packed spikes (SNNQP_SPIKES_BITS, 8x fewer
    bytes; tcgen05 kernels only, the default unless impl == IMPL_SIMT).  ``lif_mode`` concerns conv1, the block bound by its LIF epilogue
    (every other block always runs the reference's op order): LIF_EXACT = the reference's op order, bit-identical to
    the oracle; LIF_FAST = single-rounding fma on the CUDA cores (membranes within 1 ulp per step, 12 flipped spikes in
    3.1e9); LIF_TENSOR (default) = the leak runs on the tensor core (tcgen05.mma scale-input-d, membranes resident in
    TMEM; csrc/umma_conv1_tc.cu): 44 % less conv1 time, tolerance parity -- 45 flipped spikes in 3.1e9 (1.5e-8; bar
    1e-4), final membranes within 1e-5 (tools/time_conv1.py, tests/test_gpu_parity.py).  Outside the kernel's
    envelope (H = W = 128 multiples, standard LIF constants) LIF_TENSOR means LIF_EXACT."""
    self.pk = packed
    self.impl = impl
    self.lif_mode = lif_mode
    # input densities of conv2 / conv3 / conv4 (the reference sows them, models.py:128-142) straight from the
    # epilogues' ballot words (snnqp_block_params.y_popcount) instead of a separate pass over the tensors
    self.track_densities = bool(track_densities)
    # the tcgen05 envelopes of conv1 .. conv4 (W = 128 / 64 / 32 / 16, 128 channels) = the reference geometry
    in_envelope = impl != _lib.IMPL_SIMT and packed.H == 128 and packed.channels == 128
    if packed_spikes and not in_envelope:
      raise ValueError("packed_spikes needs the tcgen05 kernels: H = 128, 128 channels, impl != IMPL_SIMT")
    self.packed_spikes = in_envelope if packed_spikes is None else bool(packed_spikes)
    # conv1 of chunk k+1 and conv2 of chunk k in one persistent kernel (snnqp_spiking_head_fwd); needs the bit-packed
    # layout and the standard LIF constants.  Off by default: see DESIGN.md section 4.6 for the measured state.
    self.fused_head = False if fused_head is None else bool(fused_head)
    if self.fused_head and not self.packed_spikes:
      raise ValueError("fused_head needs packed_spikes")
    self.tau, self.v_th, self.v_reset = tau, v_threshold, v_reset
    self.chunk = chunk
    self.device = torch.device(device)
    self.max_workspaces = 4
    self._ws: Dict[tuple, Dict[str, torch.Tensor]] = {}
    self._graphs: Dict[tuple, tuple] = {}

  # -- workspace -------------------------------------------------------------
  def _workspace(self, B: int, Bc: int) -> Dict[str, torch.Tensor]:
    key = (B, Bc)
    ws = self._ws.get(key)
    if ws is not None:
      self._ws[key] = self._ws.pop(key)        # most recently used last
      return ws
    while len(self._ws) >= self.max_workspaces:  # bounded: a serving loop over many batch sizes must not pin HBM
      old = next(iter(self._ws))
      self._graphs = {k: g for k, g in self._graphs.items() if k[1] != old[0]}
      del self._ws[old]
    pk = self.pk
    T, H, C = pk.T, pk.H, pk.channels
    u8 = dict(device=self.device, dtype=torch.uint8)
    f32 = dict(device=self.device, dtype=torch.float32)
    Cs = C // 8 if self.packed_spikes else C                     # bytes per position of s1 / s2 / s3
    ws = {
        "s1": torch.empty((Bc, T, H // 2, H // 2, Cs), **u8),    # per chunk
        "s1b": torch.empty((Bc, T, H // 2, H // 2, Cs), **u8) if self.fused_head else None,   # second chunk in flight
        "s2": torch.empty((Bc, T, H // 4, H // 4, Cs), **u8),    # per chunk
        "s3": torch.empty((B, T, H // 8, H // 8, Cs), **u8),     # whole batch from here on
        "p4": torch.empty((B, T, H // 16, H // 16, C), **u8),
        "p5": torch.empty((B, T, H // 32, H // 32, C), **u8),
        "att4": torch.empty((B, T, C), **f32),
        "att5": torch.empty((B, T, C), **f32),
        "cnt4": torch.zeros((B, T, C), device=self.device, dtype=torch.int32),
        "cnt5": torch.zeros((B, T, C), device=self.device, dtype=torch.int32),
        "d1": torch.empty((B, T, pk.dense1.cout), **u8),
        "d2": torch.empty((B, T, pk.dense2.cout), **u8),
        # spikes emitted per (b, t) by conv1 / conv2 / conv3 (track_densities)
        "dens": torch.zeros((3, B, T), device=self.device, dtype=torch.int32),
    }
    self._ws[key] = ws
    return ws

  def _bp(self, B, H, Cin, Cout, x: torch.Tensor, y: Optional[torch.Tensor],
          pool: int, att: Optional[torch.Tensor] = None, att_mod: int = 0) -> BlockParams:
    p = BlockParams()
    # a spike tensor whose channel axis holds C / 8 bytes is bit-packed (SNNQP_SPIKES_BITS)
    p.x_format = _lib.SPIKES_BITS if (Cin % 32 == 0 and x.dim() == 5 and x.shape[-1] * 8 == Cin) else _lib.SPIKES_U8
    p.y_format = _lib.SPIKES_BITS if (y is not None and y.dim() == 5 and y.shape[-1] * 8 == Cout) else _lib.SPIKES_U8
    p.lif_mode = self.lif_mode
    p.T, p.B, p.H, p.W, p.Cin, p.Cout = self.pk.T, B, H, H, Cin, Cout
    p.x_stride_b, p.x_stride_t = x.stride(0) * x.element_size(), x.stride(1) * x.element_size()
    if y is not None:
      p.y_stride_b, p.y_stride_t = y.stride(0) * y.element_size(), y.stride(1) * y.element_size()
    if att is not None:
      p.att_stride_b, p.att_stride_t = att.stride(0), att.stride(1)
    p.att_mod = att_mod
    p.tau, p.v_threshold, p.v_reset = self.tau, self.v_th, self.v_reset
    p.pool = pool
    p.impl = self.impl
    return p

  # -- launches --------------------------------------------------------------
  def _conv(self, i, x, y, B, Hin, Cin, pool, att=None, counts=None, collect=None, key=None, popcount=None,
            collect_acc=True):
    L, P = _lib.lib(), _lib.ptr
    pk, C = self.pk, self.pk.channels
    lay = pk.convs[i]
    p = self._bp(B, Hin, Cin, C, x, y, pool, att, C)
    if popcount is not None:
      p.y_popcount = popcount.data_ptr()
    dump = u = None
    if collect is not None and key is not None:
      dt = torch.float32 if att is not None else torch.int32
      u = torch.empty((B, Hin, Hin, C), device=self.device, dtype=torch.float32)
      collect[key + "_u"] = u
      if collect_acc:       # (membranes alone keep conv1's LIF_TENSOR kernel eligible: it has no accumulator to dump)
        dump = torch.empty((pk.T, B, Hin, Hin, C), device=self.device, dtype=dt)
        collect[key + "_acc"] = dump
    _lib.check(L.snnqp_spiking_conv3x3_counts_fwd(p, P(x), P(att), P(lay.wq), P(lay.scale), P(lay.bias),
                                                  P(y), P(u), P(dump), P(counts), _lib.stream()))

  def _tcja(self, i, B, Hs, spikes, counts, att):
    L, P = _lib.lib(), _lib.ptr
    tj, C = self.pk.tcja[i], self.pk.channels
    p = self._bp(B, Hs, C, C, spikes if spikes is not None else att, None, 0, att, C)
    _lib.check(L.snnqp_tcja_fwd(p, P(spikes), P(tj.wq_t), P(tj.wq_c), P(tj.scale_t), P(tj.scale_c),
                                P(counts), P(att), _lib.stream()))

  def _pool(self, B, x, y, Hin):
    C = self.pk.channels
    p = self._bp(B, Hin, C, C, x, y, 1)
    _lib.check(_lib.lib().snnqp_maxpool2_fwd(p, _lib.ptr(x), _lib.ptr(y), _lib.stream()))

  def _dense(self, lay, B, x, att, y, collect=None, key=None):
    L, P = _lib.lib(), _lib.ptr
    p = self._bp(B, 1, lay.cin, lay.cout, x, y, 0, att, self.pk.channels)
    dump = u = None
    if collect is not None and key is not None:
      dt = torch.float32 if att is not None else torch.int32
      dump = torch.empty((self.pk.T, B, lay.cout), device=self.device, dtype=dt)
      u = torch.empty((B, lay.cout), device=self.device, dtype=torch.float32)
      collect[key + "_acc"], collect[key + "_u"] = dump, u
    _lib.check(L.snnqp_spiking_dense_fwd(p, P(x), P(att), P(lay.wq), P(lay.scale), P(lay.bias),
                                         P(y), P(u), P(dump), _lib.stream()))

  # -- forward ---------------------------------------------------------------
  def _run(self, frames: torch.Tensor, logits: torch.Tensor,
           collect: Optional[Dict[str, torch.Tensor]] = None) -> None:
    pk = self.pk
    B = frames.shape[0]
    H, C, T = pk.H, pk.channels, pk.T
    Bc = min(self.chunk, B)
    ws = self._workspace(B, Bc)

    # head: conv1 -> conv2 -> conv3, chunk by chunk
    if self.track_densities:
      ws["dens"].zero_()
    pipe = _HeadPipe(self, ws, collect)
    for b0 in range(0, B, Bc):
      n = min(Bc, B - b0)
      pipe.push(frames[b0:b0 + n], b0, n)
    pipe.finish()
    self._tail(B, ws, logits, collect)

  def _head(self, frames_chunk, b0, n, ws, collect=None):
    H, C = self.pk.H, self.pk.channels
    if collect is not None and self.packed_spikes:
      # instrumented pass: the generic epilogues (un-pooled spikes, membranes, accumulators) emit SNNQP_SPIKES_U8
      ws = self._u8_workspace(ws)
    s1, s2 = ws["s1"][:n], ws["s2"][:n]
    track = self.track_densities and self.packed_spikes and collect is None
    dens = [ws["dens"][k, b0:b0 + n] if track else None for k in range(3)]
    self._conv(0, frames_chunk, s1, n, H, 2, 1, collect=collect, key="conv1", popcount=dens[0])
    self._conv(1, s1, s2, n, H // 2, C, 1, collect=collect, key="conv2", popcount=dens[1])
    self._conv(2, s2, ws["s3"][b0:b0 + n], n, H // 4, C, 1, collect=collect, key="conv3", popcount=dens[2])

  def _u8_workspace(self, ws):
    if "u8" not in ws:
      C = self.pk.channels
      u8 = dict(ws)
      for k in ("s1", "s2", "s3"):
        u8[k] = torch.empty(tuple(ws[k].shape[:-1]) + (C,), device=self.device, dtype=torch.uint8)
      ws["u8"] = u8
    return ws["u8"]

  @staticmethod
  def unpack_spikes(x: torch.Tensor) -> torch.Tensor:
    """SNNQP_SPIKES_BITS (..., C/8) uint8 -> SNNQP_SPIKES_U8 (..., C) uint8 (bit c & 7 of byte c >> 3)."""
    sh = torch.arange(8, device=x.device, dtype=torch.uint8)
    return ((x.unsqueeze(-1) >> sh) & 1).reshape(tuple(x.shape[:-1]) + (x.shape[-1] * 8,))

  def _head_fused(self, frames_chunk, n1, s1_out, s1_in, n2, s2_out):
    """One launch of snnqp_spiking_head_fwd: conv1 on ``frames_chunk`` (n1 samples, may be 0) and conv2 on ``s1_in``
    (n2 samples, may be 0)."""
    L, P = _lib.lib(), _lib.ptr
    pk, H, C = self.pk, self.pk.H, self.pk.channels
    p1 = p2 = None
    x1 = y1 = x2 = y2 = None
    if n1:
      x1, y1 = frames_chunk, s1_out[:n1]
      p1 = self._bp(n1, H, 2, C, x1, y1, 1)
    if n2:
      x2, y2 = s1_in[:n2], s2_out[:n2]
      p2 = self._bp(n2, H // 2, C, C, x2, y2, 1)
    l1, l2 = pk.convs[0], pk.convs[1]
    _lib.check(L.snnqp_spiking_head_fwd(p1, P(x1), P(l1.wq), P(l1.scale), P(l1.bias), P(y1),
                                        p2, P(x2), P(l2.wq), P(l2.scale), P(l2.bias), P(y2), _lib.stream()))

  def _tail(self, B, ws, logits, collect=None):
    pk = self.pk
    H, C, T = pk.H, pk.channels, pk.T
    if collect is not None and self.packed_spikes:
      ws = self._u8_workspace(ws)
    if collect is None:
      # tail, fused: pooled spikes + spike counts straight from the conv epilogues
      ws["cnt4"].zero_(); ws["cnt5"].zero_()
      self._conv(3, ws["s3"], ws["p4"], B, H // 8, C, 1, counts=ws["cnt4"])
      self._tcja(0, B, H // 8, None, ws["cnt4"], ws["att4"])
      self._conv(4, ws["p4"], ws["p5"], B, H // 16, C, 1, att=ws["att4"], counts=ws["cnt5"])
      self._tcja(1, B, H // 16, None, ws["cnt5"], ws["att5"])
    else:
      # instrumented tail: un-pooled spikes are materialised so every intermediate can be compared
      dev = self.device
      s4 = torch.empty((B, T, H // 8, H // 8, C), device=dev, dtype=torch.uint8)
      s5 = torch.empty((B, T, H // 16, H // 16, C), device=dev, dtype=torch.uint8)
      self._conv(3, ws["s3"], s4, B, H // 8, C, 0, collect=collect, key="conv4")
      self._tcja(0, B, H // 8, s4, ws["cnt4"], ws["att4"])
      self._pool(B, s4, ws["p4"], H // 8)
      self._conv(4, ws["p4"], s5, B, H // 16, C, 0, att=ws["att4"], collect=collect, key="conv5")
      self._tcja(1, B, H // 16, s5, ws["cnt5"], ws["att5"])
      self._pool(B, s5, ws["p5"], H // 16)
      collect["s4"], collect["s5"] = s4, s5

    self._dense(pk.dense1, B, ws["p5"].view(B, T, -1), ws["att5"], ws["d1"], collect, "dense1")
    self._dense(pk.dense2, B, ws["d1"], None, ws["d2"], collect, "dense2")
    d2 = ws["d2"]
    _lib.check(_lib.lib().snnqp_vote_fwd(_lib.ptr(d2), T, B, pk.dense2.cout, 10, d2.stride(1), d2.stride(0),
                                         _lib.ptr(logits), _lib.stream()))
    if collect is not None:
      for k in ("s1", "s2", "s3", "p4", "p5", "att4", "att5", "d1", "d2"):
        collect[k] = ws[k].clone()

  def densities(self, frames: Optional[torch.Tensor] = None) -> Dict[str, Dict[str, float]]:
    """The input densities the reference sows per layer (examples/tcja/models.py:128-142, 'conv_i_inpt_min/mean',
    'dense*_inpt_*': fraction of non-zeros per (t, b) slice, max ('_min' in the reference's naming) and mean),
    measured with ``snnqp_slice_nonzeros`` on the tensors the LAST forward left in the workspace -- the pooled
    spikes that feed the next layer.  ``frames``: also report the input frames.  conv2 / conv3 inputs cover the
    last head chunk only (they are per-chunk buffers).  Host sync (it returns Python floats)."""
    from .input_pipeline import density_stats
    if not self._ws:
      raise RuntimeError("densities() needs a forward first")
    ws = list(self._ws.values())[-1]
    T = self.pk.T
    # the reference's sown names (models.py:128-173): conv_{0,1,2}_inpt for the first three blocks, conv_t_{0,1}_inpt
    # for the two TCJA blocks (their inputs are s3 and the pooled block-4 spikes)
    named = {"conv_1_inpt": ws["s1"], "conv_2_inpt": ws["s2"], "conv_t_0_inpt": ws["s3"], "conv_t_1_inpt": ws["p4"],
             "dense1_inpt": ws["p5"], "dense2_inpt": ws["d1"], "dense2_out": ws["d2"]}
    if frames is not None:
      named = dict(conv_0_inpt=frames, **named)
    out = {}
    tracked = {"conv_1_inpt": 0, "conv_2_inpt": 1, "conv_t_0_inpt": 2} if (self.track_densities and self.packed_spikes) else {}
    for k, x in named.items():
      if k in tracked:
        # counted by the producing epilogue (whole batch, not only the last head chunk)
        frac = ws["dens"][tracked[k]].to(torch.float64) / float(x[0, 0].numel() * 8)
        out[k] = {"min": float(frac.max()), "mean": float(frac.mean())}
        continue
      d = density_stats(x, x.shape[0] * T, bits=self.packed_spikes and k in ("conv_1_inpt", "conv_2_inpt", "conv_t_0_inpt"))
      out[k] = {"min": float(d["min"]), "mean": float(d["mean"])}
    return out

  def _check(self, frames: torch.Tensor) -> None:
    if not frames.is_cuda or frames.dtype != torch.uint8:
      raise ValueError("frames must be a uint8 CUDA tensor (B,T,H,W,2); no CPU fallback")
    pk = self.pk
    if tuple(frames.shape[1:]) != (pk.T, pk.H, pk.H, 2):
      raise ValueError(f"frames shape {tuple(frames.shape)} != (B,{pk.T},{pk.H},{pk.H},2)")

  def forward(self, frames: torch.Tensor, collect: Optional[Dict[str, torch.Tensor]] = None
              ) -> torch.Tensor:
    """frames: uint8 CUDA tensor (B,T,H,W,2) of event counts.  Returns fp32
    logits (B, num_classes) on the device (no host sync)."""
    self._check(frames)
    frames = frames.contiguous()
    B = frames.shape[0]
    if collect is not None and B > self.chunk:
      raise ValueError("collect= needs B <= chunk")
    logits = torch.empty((B, self.pk.num_classes), device=self.device, dtype=torch.float32)
    self._run(frames, logits, collect)
    return logits

  def host_chunks(self, B: int, first: int = 16, growth: float = 1.5):
    """Chunk schedule of the host path: a small first chunk (its copy is the only one nothing overlaps),
    then sizes growing by ``growth`` -- about the compute/copy time ratio of a chunk, so the copy of chunk
    k+1 ends roughly when the head of chunk k does -- up to ``self.chunk`` (few, large launches; measured best
    at 1.5 with a cap of 256: tools/time_e2e.py)."""
    out, b0, n = [], 0, float(min(first, self.chunk))
    while b0 < B:
      m = min(int(n), self.chunk, B - b0)
      out.append((b0, m))
      b0 += m
      n = min(max(n * growth, n + 1), float(self.chunk))
    return out

  def forward_host(self, host_frames: torch.Tensor, out_host: Optional[torch.Tensor] = None) -> torch.Tensor:
    """End-to-end call from HOST memory: ``host_frames`` is a (pinned) uint8 CPU tensor
    (B,T,H,W,2).  Chunks are copied host->device on a side stream into two staging buffers
    while the previous chunk's conv1-3 run, so the PCIe transfer overlaps compute.  Returns
    the logits on the device, or copies them into ``out_host`` (pinned) if given."""
    if host_frames.is_cuda or host_frames.dtype != torch.uint8:
      raise ValueError("forward_host takes a uint8 CPU (pinned) tensor; use forward() for device tensors")
    pk = self.pk
    if tuple(host_frames.shape[1:]) != (pk.T, pk.H, pk.H, 2):
      raise ValueError(f"frames shape {tuple(host_frames.shape)} != (B,{pk.T},{pk.H},{pk.H},2)")
    B = host_frames.shape[0]
    Bc = min(self.chunk, B)
    ws = self._workspace(B, Bc)
    if "stage" not in ws:
      ws["stage"] = torch.empty((2, Bc) + tuple(host_frames.shape[1:]), device=self.device, dtype=torch.uint8)
    if not hasattr(self, "_copy_stream"):
      self._copy_stream = torch.cuda.Stream(device=self.device)
    cur = torch.cuda.current_stream(self.device)
    logits = torch.empty((B, pk.num_classes), device=self.device, dtype=torch.float32)
    self._copy_stream.wait_stream(cur)
    done = []
    pipe = _HeadPipe(self, ws)
    for i, (b0, n) in enumerate(self.host_chunks(B)):
      buf = ws["stage"][i & 1][:n]
      if i >= 2:
        self._copy_stream.wait_event(done[i - 2])       # staging buffer free again
      with torch.cuda.stream(self._copy_stream):
        buf.copy_(host_frames[b0:b0 + n], non_blocking=True)
        ready = torch.cuda.Event()
        ready.record(self._copy_stream)
      cur.wait_event(ready)
      pipe.push(buf, b0, n)
      ev = torch.cuda.Event()
      ev.record(cur)
      done.append(ev)
    pipe.finish()
    self._tail(B, ws, logits)
    if out_host is not None:
      out_host.copy_(logits, non_blocking=True)
      return out_host
    return logits

  def forward_host_zsf(self, zb, out_host: Optional[torch.Tensor] = None) -> torch.Tensor:
    """End-to-end call from HOST memory in the zero-suppressed wire format (``input_pipeline.ZsfBatch``: cell bitmap
    + non-zero counts, ~5x fewer bytes than dense uint8 frames at the synthetic 14 % density; at 8 GPUs the dense
    frames saturate the box's host -> device bandwidth).  Per chunk: three pinned-memory copies on the side stream,
    ``snnqp_expand_frames_zsf`` into the staging frame buffer, then the same head / tail launches as
    :meth:`forward`; copies of chunk k+1 overlap the conv1-3 kernels of chunk k."""
    from .input_pipeline import zsf_expand
    pk = self.pk
    if tuple(zb.shape[1:]) != (pk.T, pk.H, pk.H, 2):
      raise ValueError(f"frames shape {tuple(zb.shape)} != (B,{pk.T},{pk.H},{pk.H},2)")
    if zb.bitmap.is_cuda:
      raise ValueError("forward_host_zsf takes the (pinned) host tensors of a ZsfBatch")
    B = zb.shape[0]
    Bc = min(self.chunk, B)
    ws = self._workspace(B, Bc)
    chunks = self.host_chunks(B)
    k = zb.blocks_per_sample
    vmax = max(zb.chunk(b0, b0 + n)[2].numel() for b0, n in chunks)
    if "stage" not in ws:
      ws["stage"] = torch.empty((2, Bc, pk.T, pk.H, pk.H, 2), device=self.device, dtype=torch.uint8)
    zkey = ("zsf", vmax)
    if ws.get("zsf_key") != zkey:
      ws["zsf_key"] = zkey
      ws["zsf"] = [(torch.empty(Bc * k * 32, device=self.device, dtype=torch.int32),
                    torch.empty(Bc * k + 1, device=self.device, dtype=torch.int32),
                    torch.empty(vmax + 16, device=self.device, dtype=torch.uint8)) for _ in range(2)]
    if not hasattr(self, "_copy_stream"):
      self._copy_stream = torch.cuda.Stream(device=self.device)
    cur = torch.cuda.current_stream(self.device)
    logits = torch.empty((B, pk.num_classes), device=self.device, dtype=torch.float32)
    self._copy_stream.wait_stream(cur)
    done = []
    pipe = _HeadPipe(self, ws)
    for i, (b0, n) in enumerate(chunks):
      bm, bo, vals, vbase, nblk = zb.chunk(b0, b0 + n)
      dbm, dbo, dv = ws["zsf"][i & 1]
      buf = ws["stage"][i & 1][:n]
      if i >= 2:
        self._copy_stream.wait_event(done[i - 2])       # staging buffers free again
      with torch.cuda.stream(self._copy_stream):
        dbm[:bm.numel()].copy_(bm, non_blocking=True)
        dbo[:bo.numel()].copy_(bo, non_blocking=True)
        dv[:vals.numel()].copy_(vals, non_blocking=True)
        ready = torch.cuda.Event()
        ready.record(self._copy_stream)
      cur.wait_event(ready)
      zsf_expand(dbm, dbo, dv, vbase, nblk, zb.value_bits, buf)
      pipe.push(buf, b0, n)
      ev = torch.cuda.Event()
      ev.record(cur)
      done.append(ev)
    pipe.finish()
    self._tail(B, ws, logits)
    if out_host is not None:
      out_host.copy_(logits, non_blocking=True)
      return out_host
    return logits

  def forward_host_events(self, eb, resolution_scale: int = 1, out_host: Optional[torch.Tensor] = None,
                          n_saturated: Optional[torch.Tensor] = None) -> torch.Tensor:
    """End-to-end call from HOST memory on event recordings (``input_pipeline.EventBatch``: one packed word per event,
    what the reference's loader holds before it integrates frames).  Per chunk: two pinned-memory copies (words,
    offsets) on the side stream, ``snnqp_events_to_frames_packed`` into the staging frame buffer, then the same head /
    tail launches as :meth:`forward`; copies of chunk k+1 overlap the conv1-3 kernels of chunk k.  The frames are
    uint8, saturating at 255: ``n_saturated`` (device int64 scalar), if given, accumulates the saturated cells (no
    host sync)."""
    from .input_pipeline import events_to_frames_packed
    pk = self.pk
    if eb.events.is_cuda:
      raise ValueError("forward_host_events takes the (pinned) host tensors of an EventBatch")
    if int(resolution_scale) != resolution_scale or resolution_scale < 1 or eb.sensor_wh // resolution_scale != pk.H:
      raise ValueError(f"sensor {eb.sensor_wh} // resolution_scale {resolution_scale} != H = {pk.H}")
    B = eb.shape[0]
    Bc = min(self.chunk, B)
    ws = self._workspace(B, Bc)
    chunks = self.host_chunks(B)
    o = eb.offsets.numpy()
    emax = max(int(o[b0 + n] - o[b0]) for b0, n in chunks)
    if "stage" not in ws:
      ws["stage"] = torch.empty((2, Bc, pk.T, pk.H, pk.H, 2), device=self.device, dtype=torch.uint8)
    ev = ws.get("ev")
    if ev is None or ev[0][0].dtype != eb.events.dtype or ev[0][0].numel() < emax:
      # sized to the largest chunk; safe to replace: the side stream waits for the current stream before its first copy
      ws["ev"] = ev = [(torch.empty(max(emax, 1), device=self.device, dtype=eb.events.dtype),
                        torch.empty(Bc + 1, device=self.device, dtype=torch.int64)) for _ in range(2)]
    if n_saturated is None:                             # a scratch counter: no fill launch per chunk
      if "ev_sat" not in ws:
        ws["ev_sat"] = torch.zeros((), device=self.device, dtype=torch.int64)
      n_saturated = ws["ev_sat"]
    if not hasattr(self, "_copy_stream"):
      self._copy_stream = torch.cuda.Stream(device=self.device)
    cur = torch.cuda.current_stream(self.device)
    logits = torch.empty((B, pk.num_classes), device=self.device, dtype=torch.float32)
    self._copy_stream.wait_stream(cur)
    done = []
    pipe = _HeadPipe(self, ws)
    for i, (b0, n) in enumerate(chunks):
      words, offs, base = eb.chunk(b0, b0 + n)
      dev, doff = ev[i & 1]
      buf = ws["stage"][i & 1][:n]
      if i >= 2:
        self._copy_stream.wait_event(done[i - 2])       # staging buffers free again
      with torch.cuda.stream(self._copy_stream):
        dev[:words.numel()].copy_(words, non_blocking=True)
        doff[:n + 1].copy_(offs, non_blocking=True)
        ready = torch.cuda.Event()
        ready.record(self._copy_stream)
      cur.wait_event(ready)
      events_to_frames_packed(dev, doff[:n + 1], eb.format, pk.T, eb.sensor_wh, resolution_scale, out=buf,
                              max_events_per_sample=eb.max_events_per_sample, event_base=base,
                              n_saturated=n_saturated)
      pipe.push(buf, b0, n)
      e = torch.cuda.Event()
      e.record(cur)
      done.append(e)
    pipe.finish()
    self._tail(B, ws, logits)
    if out_host is not None:
      out_host.copy_(logits, non_blocking=True)
      return out_host
    return logits

  def forward_graph(self, frames: torch.Tensor) -> torch.Tensor:
    """Same as :meth:`forward`, replayed from a CUDA graph captured on the first
    call for this (buffer, batch) -- removes the per-launch host overhead.  The
    returned logits tensor is static (overwritten by the next replay)."""
    self._check(frames)
    if not frames.is_contiguous():
      raise ValueError("forward_graph needs a contiguous frames buffer")
    key = (frames.data_ptr(), frames.shape[0])
    ent = self._graphs.get(key)
    if ent is None:
      logits = torch.empty((frames.shape[0], self.pk.num_classes), device=self.device, dtype=torch.float32)
      self._run(frames, logits)                 # eager warm-up: function attributes, workspaces
      torch.cuda.synchronize()
      g = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g):
        self._run(frames, logits)
      ent = (g, logits, frames)
      self._graphs[key] = ent
    ent[0].replay()
    return ent[1]
