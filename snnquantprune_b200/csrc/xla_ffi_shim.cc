// XLA FFI custom-call shim over the C-ABI (see INTEGRATION.md section 3).
// jaxlib's FFI headers are not present in this image, so the handlers are
// compiled only where <xla/ffi/api/ffi.h> exists; elsewhere this TU is empty.
#if defined(__has_include)
#if __has_include("xla/ffi/api/ffi.h")
#define SNNQP_HAVE_XLA_FFI 1
#endif
#endif

#ifdef SNNQP_HAVE_XLA_FFI
#include <cuda_runtime.h>

#include <vector>

#include "snnqp.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

static ffi::Error Status(int rc) {
  return rc == SNNQP_OK ? ffi::Error::Success() : ffi::Error(ffi::ErrorCode::kInvalidArgument, snnqp_last_error());
}

// SpikingBlock(QuantConv3x3, BatchNorm, multi_step_LIF) [+ max-pool]; x: (B,T,H,W,Cin) uint8, batch-major
static ffi::Error SpikingConvImpl(cudaStream_t stream, ffi::Buffer<ffi::U8> x, ffi::Buffer<ffi::S8> wq,
                                  ffi::Buffer<ffi::F32> scale, ffi::Buffer<ffi::F32> bias,
                                  ffi::ResultBuffer<ffi::U8> spikes, int32_t pool, float tau, float v_th,
                                  float v_reset) {
  auto d = x.dimensions();
  snnqp_block_params p{};
  p.B = (int32_t)d[0]; p.T = (int32_t)d[1]; p.H = (int32_t)d[2]; p.W = (int32_t)d[3]; p.Cin = (int32_t)d[4];
  p.Cout = (int32_t)scale.dimensions()[0];
  p.x_stride_t = (int64_t)p.H * p.W * p.Cin; p.x_stride_b = p.x_stride_t * p.T;
  const int Ho = pool ? p.H / 2 : p.H, Wo = pool ? p.W / 2 : p.W;
  p.y_stride_t = (int64_t)Ho * Wo * p.Cout; p.y_stride_b = p.y_stride_t * p.T;
  p.tau = tau; p.v_threshold = v_th; p.v_reset = v_reset; p.pool = pool; p.impl = SNNQP_IMPL_AUTO;
  return Status(snnqp_spiking_conv3x3_fwd(&p, x.typed_data(), nullptr, wq.typed_data(), scale.typed_data(),
                                          bias.typed_data(), spikes->typed_data(), nullptr, nullptr, stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpSpikingConv, SpikingConvImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()
                                  .Arg<ffi::Buffer<ffi::S8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<int32_t>("pool")
                                  .Attr<float>("tau")
                                  .Attr<float>("v_threshold")
                                  .Attr<float>("v_reset"));

// SpikingBlock(QuantDense, multi_step_LIF); x: (B,T,K) uint8
static ffi::Error SpikingDenseImpl(cudaStream_t stream, ffi::Buffer<ffi::U8> x, ffi::Buffer<ffi::S8> wq,
                                   ffi::Buffer<ffi::F32> scale, ffi::Buffer<ffi::F32> bias,
                                   ffi::ResultBuffer<ffi::U8> spikes, float tau, float v_th, float v_reset) {
  auto d = x.dimensions();
  snnqp_block_params p{};
  p.B = (int32_t)d[0]; p.T = (int32_t)d[1]; p.H = p.W = 1; p.Cin = (int32_t)d[2];
  p.Cout = (int32_t)scale.dimensions()[0];
  p.x_stride_t = p.Cin; p.x_stride_b = (int64_t)p.T * p.Cin;
  p.y_stride_t = p.Cout; p.y_stride_b = (int64_t)p.T * p.Cout;
  p.tau = tau; p.v_threshold = v_th; p.v_reset = v_reset; p.impl = SNNQP_IMPL_AUTO;
  return Status(snnqp_spiking_dense_fwd(&p, x.typed_data(), nullptr, wq.typed_data(), scale.typed_data(),
                                        bias.typed_data(), spikes->typed_data(), nullptr, nullptr, stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpSpikingDense, SpikingDenseImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()
                                  .Arg<ffi::Buffer<ffi::S8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<float>("tau")
                                  .Attr<float>("v_threshold")
                                  .Attr<float>("v_reset"));

// TCJA (models.py:41-95) from the spike counts a conv block accumulated; att: (B,T,C) fp32
static ffi::Error TcjaImpl(cudaStream_t stream, ffi::Buffer<ffi::S32> counts, ffi::Buffer<ffi::S8> wq_t,
                           ffi::Buffer<ffi::S8> wq_c, ffi::Buffer<ffi::F32> scale_t, ffi::Buffer<ffi::F32> scale_c,
                           ffi::ResultBuffer<ffi::F32> att, int32_t spatial) {
  auto d = counts.dimensions();                 // (B, T, C)
  snnqp_block_params p{};
  p.B = (int32_t)d[0]; p.T = (int32_t)d[1]; p.Cin = p.Cout = (int32_t)d[2]; p.H = p.W = spatial;
  p.att_stride_t = p.Cin; p.att_stride_b = (int64_t)p.T * p.Cin; p.att_mod = p.Cin;
  return Status(snnqp_tcja_fwd(&p, nullptr, wq_t.typed_data(), wq_c.typed_data(), scale_t.typed_data(),
                               scale_c.typed_data(), counts.typed_data(), att->typed_data(), stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpTcja, TcjaImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::S32>>()
                                  .Arg<ffi::Buffer<ffi::S8>>()
                                  .Arg<ffi::Buffer<ffi::S8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>()
                                  .Attr<int32_t>("spatial"));

// vote (models.py:253-255): spikes (B,T,N) uint8 -> logits (B, N / group) fp32
static ffi::Error VoteImpl(cudaStream_t stream, ffi::Buffer<ffi::U8> spikes, ffi::ResultBuffer<ffi::F32> logits,
                           int32_t group) {
  auto d = spikes.dimensions();
  return Status(snnqp_vote_fwd(spikes.typed_data(), (int)d[1], (int)d[0], (int)d[2], group, d[2], d[1] * d[2],
                               logits->typed_data(), stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpVote, VoteImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()
                                  .Ret<ffi::Buffer<ffi::F32>>()
                                  .Attr<int32_t>("group"));

// event -> frame integration (examples/input_pipeline.py:142-219): addrs (N,3) int32, offsets (B+1) int64
static ffi::Error EventsToFramesImpl(cudaStream_t stream, ffi::Buffer<ffi::S32> addrs, ffi::Buffer<ffi::S64> offsets,
                                     ffi::ResultBuffer<ffi::U8> frames, int32_t sensor_wh, int32_t resolution_scale,
                                     int64_t max_events_per_sample) {
  auto f = frames->dimensions();                // (B, T, wh, wh, 2)
  return Status(snnqp_events_to_frames(addrs.typed_data(), offsets.typed_data(), (int)f[0], (int)f[1], sensor_wh,
                                       resolution_scale, max_events_per_sample, frames->typed_data(), 0, nullptr,
                                       stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpEventsToFrames, EventsToFramesImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::S32>>()
                                  .Arg<ffi::Buffer<ffi::S64>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<int32_t>("sensor_wh")
                                  .Attr<int32_t>("resolution_scale")
                                  .Attr<int64_t>("max_events_per_sample"));

// packed event words (SNNQP_EVENTS_U16 / _U32, include/snnqp.h) -> frames: events is the words' raw bytes (N * 2 or
// N * 4 uint8, e.g. lax.bitcast_convert_type of the uint16 / uint32 words), offsets (B+1) int64 relative to event_base
static ffi::Error EventsToFramesPackedImpl(cudaStream_t stream, ffi::Buffer<ffi::U8> events, ffi::Buffer<ffi::S64> offsets,
                                           ffi::ResultBuffer<ffi::U8> frames, int32_t event_format, int32_t sensor_wh,
                                           int32_t resolution_scale, int64_t max_events_per_sample, int64_t event_base) {
  auto f = frames->dimensions();                // (B, T, wh, wh, 2)
  return Status(snnqp_events_to_frames_packed(events.typed_data(), event_format, offsets.typed_data(), event_base,
                                              (int)f[0], (int)f[1], sensor_wh, resolution_scale, max_events_per_sample,
                                              frames->typed_data(), 0, nullptr, stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpEventsToFramesPacked, EventsToFramesPackedImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()
                                  .Arg<ffi::Buffer<ffi::S64>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<int32_t>("event_format")
                                  .Attr<int32_t>("sensor_wh")
                                  .Attr<int32_t>("resolution_scale")
                                  .Attr<int64_t>("max_events_per_sample")
                                  .Attr<int64_t>("event_base"));

// ---- the att-weighted / counting variants that wire conv4 -> TCJA -> conv5 -> dense1 (examples/tcja/models.py:
// 151-246): the binding a maintainer adds inside SpikingBlock.__call__ (spiking_learning.py:454-462) ---------------
static void FillConv(snnqp_block_params &p, const std::vector<int64_t> &d, int32_t cout, int32_t pool, float tau,
                     float v_th, float v_reset, int32_t x_bits, int32_t y_bits, int32_t lif_mode) {
  p.B = (int32_t)d[0]; p.T = (int32_t)d[1]; p.H = (int32_t)d[2]; p.W = (int32_t)d[3];
  p.Cin = x_bits ? (int32_t)d[4] * 8 : (int32_t)d[4];
  p.Cout = cout;
  p.x_stride_t = (int64_t)p.H * p.W * d[4]; p.x_stride_b = p.x_stride_t * p.T;
  const int Ho = pool ? p.H / 2 : p.H, Wo = pool ? p.W / 2 : p.W;
  p.y_stride_t = (int64_t)Ho * Wo * (y_bits ? cout / 8 : cout); p.y_stride_b = p.y_stride_t * p.T;
  p.att_stride_t = p.Cin; p.att_stride_b = (int64_t)p.T * p.Cin; p.att_mod = p.Cin;
  p.tau = tau; p.v_threshold = v_th; p.v_reset = v_reset; p.pool = pool; p.impl = SNNQP_IMPL_AUTO;
  p.x_format = x_bits ? SNNQP_SPIKES_BITS : SNNQP_SPIKES_U8;
  p.y_format = y_bits ? SNNQP_SPIKES_BITS : SNNQP_SPIKES_U8;
  p.lif_mode = lif_mode;
}

// conv block with spike counts (TCJA numerator), optional bit-packed spikes in / out; counts (B,T,C) int32 is an
// input/output operand (zero-initialised by the caller, aliased to the result)
static ffi::Error SpikingConvCountsImpl(cudaStream_t stream, ffi::Buffer<ffi::U8> x, ffi::Buffer<ffi::S8> wq,
                                        ffi::Buffer<ffi::F32> scale, ffi::Buffer<ffi::F32> bias,
                                        ffi::ResultBuffer<ffi::U8> spikes, ffi::ResultBuffer<ffi::S32> counts,
                                        int32_t pool, float tau, float v_th, float v_reset, int32_t x_bits,
                                        int32_t y_bits, int32_t lif_mode) {
  snnqp_block_params p{};
  FillConv(p, x.dimensions(), (int32_t)scale.dimensions()[0], pool, tau, v_th, v_reset, x_bits, y_bits, lif_mode);
  if (cudaMemsetAsync(counts->typed_data(), 0, sizeof(int32_t) * counts->element_count(), stream) != cudaSuccess)
    return ffi::Error(ffi::ErrorCode::kInternal, "cudaMemsetAsync(counts)");
  return Status(snnqp_spiking_conv3x3_counts_fwd(&p, x.typed_data(), nullptr, wq.typed_data(), scale.typed_data(),
                                                 bias.typed_data(), spikes->typed_data(), nullptr, nullptr,
                                                 counts->typed_data(), stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpSpikingConvCounts, SpikingConvCountsImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()
                                  .Arg<ffi::Buffer<ffi::S8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()
                                  .Ret<ffi::Buffer<ffi::S32>>()
                                  .Attr<int32_t>("pool")
                                  .Attr<float>("tau")
                                  .Attr<float>("v_threshold")
                                  .Attr<float>("v_reset")
                                  .Attr<int32_t>("x_bits")
                                  .Attr<int32_t>("y_bits")
                                  .Attr<int32_t>("lif_mode"));

// conv block on the TCJA output y = x_seq * att (models.py:97): x = pooled spikes (B,T,H,W,C) uint8, att (B,T,C) fp32
static ffi::Error SpikingConvAttImpl(cudaStream_t stream, ffi::Buffer<ffi::U8> x, ffi::Buffer<ffi::F32> att,
                                     ffi::Buffer<ffi::S8> wq, ffi::Buffer<ffi::F32> scale, ffi::Buffer<ffi::F32> bias,
                                     ffi::ResultBuffer<ffi::U8> spikes, ffi::ResultBuffer<ffi::S32> counts,
                                     int32_t pool, float tau, float v_th, float v_reset) {
  snnqp_block_params p{};
  FillConv(p, x.dimensions(), (int32_t)scale.dimensions()[0], pool, tau, v_th, v_reset, 0, 0, SNNQP_LIF_EXACT);
  if (cudaMemsetAsync(counts->typed_data(), 0, sizeof(int32_t) * counts->element_count(), stream) != cudaSuccess)
    return ffi::Error(ffi::ErrorCode::kInternal, "cudaMemsetAsync(counts)");
  return Status(snnqp_spiking_conv3x3_counts_fwd(&p, x.typed_data(), att.typed_data(), wq.typed_data(),
                                                 scale.typed_data(), bias.typed_data(), spikes->typed_data(), nullptr,
                                                 nullptr, counts->typed_data(), stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpSpikingConvAtt, SpikingConvAttImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::S8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()
                                  .Ret<ffi::Buffer<ffi::S32>>()
                                  .Attr<int32_t>("pool")
                                  .Attr<float>("tau")
                                  .Attr<float>("v_threshold")
                                  .Attr<float>("v_reset"));

// dense block on att * x (dense1 after the second TCJA): x (B,T,K) uint8, att (B,T,att_mod) fp32, k -> att[k % att_mod]
static ffi::Error SpikingDenseAttImpl(cudaStream_t stream, ffi::Buffer<ffi::U8> x, ffi::Buffer<ffi::F32> att,
                                      ffi::Buffer<ffi::S8> wq, ffi::Buffer<ffi::F32> scale, ffi::Buffer<ffi::F32> bias,
                                      ffi::ResultBuffer<ffi::U8> spikes, float tau, float v_th, float v_reset) {
  auto d = x.dimensions();
  snnqp_block_params p{};
  p.B = (int32_t)d[0]; p.T = (int32_t)d[1]; p.H = p.W = 1; p.Cin = (int32_t)d[2];
  p.Cout = (int32_t)scale.dimensions()[0];
  p.x_stride_t = p.Cin; p.x_stride_b = (int64_t)p.T * p.Cin;
  p.y_stride_t = p.Cout; p.y_stride_b = (int64_t)p.T * p.Cout;
  p.att_mod = (int32_t)att.dimensions()[2];
  p.att_stride_t = p.att_mod; p.att_stride_b = (int64_t)p.T * p.att_mod;
  p.tau = tau; p.v_threshold = v_th; p.v_reset = v_reset; p.impl = SNNQP_IMPL_AUTO;
  return Status(snnqp_spiking_dense_fwd(&p, x.typed_data(), att.typed_data(), wq.typed_data(), scale.typed_data(),
                                        bias.typed_data(), spikes->typed_data(), nullptr, nullptr, stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpSpikingDenseAtt, SpikingDenseAttImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::S8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<float>("tau")
                                  .Attr<float>("v_threshold")
                                  .Attr<float>("v_reset"));

// ---- the one-time pack step, bound after load_model_fn / mask construction (train_inpt_spikingjelly.py:144-230) ----
// kernel (3,3,cin,cout) fp32 HWIO + mask + DuQ a -> blob (snnqp_conv3x3_blob_bytes(cin, cout) int8)
static ffi::Error PackConvImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> kernel, ffi::Buffer<ffi::F32> mask,
                               ffi::Buffer<ffi::F32> a, ffi::ResultBuffer<ffi::S8> blob, int32_t bits) {
  auto d = kernel.dimensions();
  const int cin = (int)d[2], cout = (int)d[3];
  if ((int64_t)blob->element_count() < snnqp_conv3x3_blob_bytes(cin, cout))
    return ffi::Error(ffi::ErrorCode::kInvalidArgument, "blob smaller than snnqp_conv3x3_blob_bytes(cin, cout)");
  if (cin == 2)
    return Status(snnqp_pack_conv1(kernel.typed_data(), mask.typed_data(), a.typed_data(), bits, cout,
                                   blob->typed_data(), stream));
  return Status(snnqp_pack_conv3x3(kernel.typed_data(), mask.typed_data(), a.typed_data(), bits, cin, cout,
                                   blob->typed_data(), stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpPackConv, PackConvImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::S8>>()
                                  .Attr<int32_t>("bits"));

// QuantDense kernel (K,N) + mask + a (+ row permutation, e.g. the folded flatten of models.py:189-190) -> [N][k_pad]
static ffi::Error PackMatrixImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> kernel, ffi::Buffer<ffi::F32> mask,
                                 ffi::Buffer<ffi::F32> a, ffi::Buffer<ffi::S32> row_perm,
                                 ffi::ResultBuffer<ffi::S8> wq, int32_t bits) {
  auto d = kernel.dimensions();
  const int K = (int)d[0], N = (int)d[1], k_pad = (int)wq->dimensions()[1];
  return Status(snnqp_pack_matrix(kernel.typed_data(), mask.typed_data(), a.typed_data(), bits, K, N,
                                  row_perm.element_count() ? row_perm.typed_data() : nullptr, k_pad,
                                  wq->typed_data(), stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpPackMatrix, PackMatrixImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::S32>>()
                                  .Ret<ffi::Buffer<ffi::S8>>()
                                  .Attr<int32_t>("bits"));

// levels in the kernel's own layout (TCJA 1-D convs, QuantDense / QuantConv facades)
static ffi::Error PackLevelsImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> kernel, ffi::Buffer<ffi::F32> mask,
                                 ffi::Buffer<ffi::F32> a, ffi::ResultBuffer<ffi::S8> q, int32_t bits) {
  return Status(snnqp_pack_levels(kernel.typed_data(), mask.typed_data(), a.typed_data(), bits,
                                  (int64_t)kernel.element_count(), q->typed_data(), stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpPackLevels, PackLevelsImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::S8>>()
                                  .Attr<int32_t>("bits"));

// DuQ scale c / L folded with eval BatchNorm (models.py:101-107) into per-channel fp32 (scale, bias)
static ffi::Error FoldAffineImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> c, ffi::Buffer<ffi::F32> gamma,
                                 ffi::Buffer<ffi::F32> beta, ffi::Buffer<ffi::F32> mean, ffi::Buffer<ffi::F32> var,
                                 ffi::ResultBuffer<ffi::F32> scale, ffi::ResultBuffer<ffi::F32> bias, int32_t bits,
                                 float eps, float extra_div) {
  const int n = (int)scale->element_count();
  const bool bn = gamma.element_count() != 0;
  return Status(snnqp_fold_affine(c.typed_data(), bits, (double)extra_div, bn ? gamma.typed_data() : nullptr,
                                  bn ? beta.typed_data() : nullptr, bn ? mean.typed_data() : nullptr,
                                  bn ? var.typed_data() : nullptr, eps, n, scale->typed_data(), bias->typed_data(),
                                  stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpFoldAffine, FoldAffineImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>()
                                  .Attr<int32_t>("bits")
                                  .Attr<float>("eps")
                                  .Attr<float>("extra_div"));

// zero-suppressed frames -> dense uint8 frames (B,T,H,W,2): the end-to-end input format
static ffi::Error ExpandFramesZsfImpl(cudaStream_t stream, ffi::Buffer<ffi::U32> bitmap, ffi::Buffer<ffi::U32> block_off,
                                      ffi::Buffer<ffi::U8> values, ffi::ResultBuffer<ffi::U8> frames,
                                      int32_t value_bits, int64_t value_base) {
  const int64_t n_blocks = (int64_t)frames->element_count() / 1024;
  return Status(snnqp_expand_frames_zsf(bitmap.typed_data(), block_off.typed_data(), values.typed_data(),
                                        (uint32_t)value_base, n_blocks, value_bits, frames->typed_data(), stream));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(SnnqpExpandFramesZsf, ExpandFramesZsfImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U32>>()
                                  .Arg<ffi::Buffer<ffi::U32>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<int32_t>("value_bits")
                                  .Attr<int64_t>("value_base"));
#endif  // SNNQP_HAVE_XLA_FFI
