/* snnqp.h -- C-ABI of the B200-native quantized + pruned spiking-layer forward
 * pass (drop-in for the hot path of Intelligent-Microsystems-Lab/SNNQuantPrune).
 *
 * The reference has no FFI of its own: the path sits behind Flax modules
 * (citations relative to the reference root):
 *   DuQ.__call__            quant.py:439-469      -> snnqp_duq_forward / snnqp_pack_*
 *   prune.__call__          quant.py:475-491      -> (mask argument of the above)
 *   QuantConv.__call__      flax_qconv.py:94-188  -> snnqp_spiking_conv3x3_fwd (fused
 *   nn.BatchNorm (eval)     examples/tcja/models.py:101-107    with BN + LIF + pool),
 *   multi_step_LIF.__call__ spiking_learning.py:404-416        snnqp_qconv3x3_fwd (plain)
 *   SpikingBlock.__call__   spiking_learning.py:441-472
 *   QuantDense.__call__     flax_qdense.py:59-106 -> snnqp_spiking_dense_fwd
 *   TCJA                    examples/tcja/models.py:41-99  -> snnqp_tcja_fwd
 *   max-pool / flatten      examples/tcja/models.py:145-147,189-190 -> fused / pack-time
 *   vote                    examples/tcja/models.py:253-255 -> snnqp_vote_fwd
 *   compute_metrics         examples/train_utils.py:220-225 -> snnqp_eval_metrics
 * These are the entry points an XLA-FFI custom-call shim binds (INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller unless named *_host;
 *    nothing is retained past the call, nothing is allocated on the hot calls
 *    (TMA descriptors are cached per device, keyed by pointer + shape);
 *  - every launch goes on the caller's stream (cudaStream_t passed as void*);
 *    no host synchronisation;
 *  - return 0 on success, a SNNQP_ERR_* code otherwise; the message of the last
 *    failure on this thread is returned by snnqp_last_error();
 *  - spikes and event counts are uint8 (one byte per neuron, channel-minor:
 *    [...][H][W][C]); timestep / sample strides are explicit (in bytes for
 *    uint8 tensors, in elements for float tensors) so both the reference's
 *    time-major (T,B,...) and batch-major (B,T,...) layouts are accepted;
 *  - there is NO CPU fallback: every entry point fails with SNNQP_ERR_CUDA if
 *    no sm_100 device is present.
 */
#ifndef SNNQP_H_
#define SNNQP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNNQP_ABI_VERSION 4

#define SNNQP_OK 0
#define SNNQP_ERR_INVALID 1      /* bad argument / unsupported shape           */
#define SNNQP_ERR_CUDA 2         /* CUDA runtime / driver error                */
#define SNNQP_ERR_UNSUPPORTED 3  /* valid in the reference, outside this path  */

/* kernel implementation selector for the fused blocks */
#define SNNQP_IMPL_AUTO 0
#define SNNQP_IMPL_SIMT 1        /* dp4a CUDA-core kernels (bring-up / cross-check) */
#define SNNQP_IMPL_TCGEN05 2     /* tcgen05.mma.kind::i8 + TMA + TMEM               */

int snnqp_abi_version(void);
const char *snnqp_last_error(void);
/* 1 if the current device is compute capability 10.x, else 0. */
int snnqp_device_ok(void);

/* ---------------------------------------------------------------- pack ---- */

/* DuQ forward followed by prune forward, elementwise, fp32 out
 * (quant.py:439-469, 475-491).  a, c: device pointers to one float each;
 * mask may be NULL.  bits == -1 or *a == -1 passes the input through. */
int snnqp_duq_forward(const float *w, const float *mask, const float *a,
                      const float *c, int bits, int64_t n, float *out,
                      void *stream);

/* Integer DuQ level (quant.py:463-467) with the mask applied, same layout as
 * the input: q[i] = round_half_even(clip(w[i] / *a, -1, 1) * L) * (mask != 0),
 * L = 2^(bits-1) - 1 (4- and 2-bit levels are stored unpacked in int8). */
int snnqp_pack_levels(const float *w, const float *mask, const float *a,
                      int bits, int64_t n, int8_t *q, void *stream);

/* 3x3 HWIO kernel (3,3,cin,cout) -> packed weight blob of
 * snnqp_conv3x3_blob_bytes(cin, cout) bytes: levels in tile layout
 * [9][cout][cin] (tap-major, one 128-byte K row per output channel when
 * cin == 128) followed, when cin % 32 == 0, by the 9*cin/32 flags of
 * snnqp_conv3x3_slab_bitmap (padded to 64 bytes) that drive the block-sparse
 * skip of all-zero weight K-slabs. */
int64_t snnqp_conv3x3_blob_bytes(int cin, int cout);

/* conv1 (cin == 2): blob of snnqp_conv3x3_blob_bytes(2, cout) = 5*cout*32
 * bytes: [cout][32] with k = tap*2 + ci, then the four quad-position matrices
 * [4][cout][32] (j = 2*dy + dx, k = py*8 + px*2 + ci over the 4x4x2 input
 * patch of a 2x2 pool quad) that the tcgen05 conv1 kernel multiplies. */
int snnqp_pack_conv1(const float *kernel_hwio, const float *mask, const float *a,
                     int bits, int cout, int8_t *wq, void *stream);
int snnqp_pack_conv3x3(const float *kernel_hwio, const float *mask,
                       const float *a, int bits, int cin, int cout, int8_t *wq,
                       void *stream);

/* (K,N) kernel [dense (in,out); 1-D conv (k*cin,cout); conv1 (18,cout)] ->
 * levels in layout [N][k_pad], zero padded.  row_perm (nullable, K int32):
 * packed column r reads kernel row row_perm[r] -- used to fold the reference's
 * NCHW flatten (examples/tcja/models.py:189-190) into the dense1 weights. */
int snnqp_pack_matrix(const float *kernel_kn, const float *mask, const float *a,
                      int bits, int K, int N, const int32_t *row_perm,
                      int k_pad, int8_t *wq, void *stream);

/* Per-channel folded affine so that v = acc * scale[n] + bias[n]:
 *   scale[n] = (c / L / extra_div) * gamma[n] / sqrt(var[n] + eps)
 *   bias[n]  = beta[n] - mean[n] * gamma[n] / sqrt(var[n] + eps)
 * (DuQ dequant scale quant.py:442,467; eval BatchNorm models.py:101-107),
 * evaluated in IEEE double and rounded once.  gamma..var NULL => no BN:
 * scale = c / L / extra_div, bias = 0. */
int snnqp_fold_affine(const float *c, int bits, double extra_div,
                      const float *gamma, const float *beta, const float *mean,
                      const float *var, float eps, int n, float *scale,
                      float *bias, void *stream);

/* Bitmap of all-zero weight K-slabs for the block-sparse skip path:
 * nz[tap * (cin/32) + j] = 1 iff wq[tap][:, 32j..32j+31] has a non-zero. */
int snnqp_conv3x3_slab_bitmap(const int8_t *wq, int cin, int cout,
                              uint8_t *nz, void *stream);

/* ------------------------------------------------------- fused blocks ---- */

typedef struct snnqp_block_params {
  int32_t T, B, H, W;      /* timesteps, samples, input height/width (dense: 1,1) */
  int32_t Cin, Cout;       /* input / output features                            */
  int64_t x_stride_t, x_stride_b; /* bytes between timesteps / samples of x       */
  int64_t y_stride_t, y_stride_b; /* bytes between timesteps / samples of spikes  */
  int64_t att_stride_t, att_stride_b; /* elements, for att[(t,b)][Cin or att_mod] */
  int32_t att_mod;         /* dense: input k uses att[k % att_mod]; conv: = Cin   */
  float tau, v_threshold, v_reset; /* multi_step_LIF, spiking_learning.py:390-397 */
  int32_t pool;            /* 1: fuse the 2x2/2 max-pool (models.py:145-147)      */
  int32_t impl;            /* SNNQP_IMPL_*                                        */
  int32_t x_format;        /* SNNQP_SPIKES_*: layout of x (BITS: binary inputs, Cin % 32 == 0) */
  int32_t y_format;        /* SNNQP_SPIKES_*: layout of the emitted spikes        */
  int32_t lif_mode;        /* SNNQP_LIF_*                                          */
  int32_t *y_popcount;     /* NULL, or device int32 [B][T], caller-zeroed: += the number of
                            * emitted (pooled) spikes of each (b, t) -- the numerator of the input
                            * density the reference sows for the NEXT layer (examples/tcja/
                            * models.py:128-142), for free from the ballot words of the
                            * bit-packed epilogues (y_format == SNNQP_SPIKES_BITS only)        */
} snnqp_block_params;

/* Spike tensor layouts (both channel-minor, strides in bytes):
 *   U8   one byte per spike / event count: [..][H][W][C] uint8;
 *   BITS bit-packed {0,1} spikes: [..][H][W][C/8] bytes, channel c = bit (c & 7)
 *        of byte (c >> 3) (= bit c % 32 of little-endian word c / 32), i.e.
 *        numpy.packbits(..., axis=-1, bitorder="little").  The reference's
 *        spikes are fp32 {0,1} (spiking_learning.py:412-416); 8x fewer bytes
 *        than U8, 32x fewer than fp32.  Emitted by the production epilogues
 *        (pool == 1, no instrumentation outputs) with one 32-channel word per
 *        warp ballot; consumed by the tcgen05 3x3 block, whose expander warps
 *        turn the TMA-staged bits into the u8 MMA operand in shared memory. */
#define SNNQP_SPIKES_U8 0
#define SNNQP_SPIKES_BITS 1
/* LIF arithmetic for tau = 2, v_threshold = 1, v_reset = 0 (other constants
 * always use the reference's op order):
 *   EXACT  u + (x - u) / 2 in the reference's op order (spiking_learning.py:409),
 *          bit-identical to the oracle;
 *   FAST   fma(u, 0.5, x / 2) with the halving folded into scale / bias: one
 *          rounding instead of two, |du| <= 1 ulp per step (north-star bar
 *          1e-5), spikes may flip only when un is within an ulp of 1.
 *          Tested against a float64 band: per step h = fma(acc, s/2, b/2)
 *          and un = fma(u, 0.5, h) round once each, e_t = 2^-24 (|h| + |un|),
 *          delta_t = e_t + delta_{t-1} / 2 until the first step with
 *          |un - 1| <= delta_t; every pooled spike the band decides must
 *          equal float64 (tests/test_gpu_conv1_rounding_band.py). */
#define SNNQP_LIF_EXACT 0
#define SNNQP_LIF_FAST 1
/*   TENSOR (conv1, tcgen05 path, production variant only; EXACT elsewhere): the
 *          leak runs on the tensor core -- tcgen05.mma's scale-input-d computes
 *          D = A * B + D / 2, so the TMEM accumulator IS the membrane (scale
 *          folded into two fp16 weight pieces, bias on a constant-one K
 *          column) and the epilogue only compares, resets and packs.  The
 *          accumulation rounding is the tensor core's, not IEEE fma: tolerance
 *          parity (membrane 1e-5, spike flips <= 1e-4), not bit parity.
 *          Tested against a float64 band (same propagation as FAST) whose
 *          per-step bound, in threshold units, is
 *            e_t = (A_t rw + rb) / dom + c_acc 2^-24 (A_t |s| + |b| + |u|) / 2
 *          with A_t = sum |q| x, dom the domain scale below, rw / rb the
 *          exact error of the fp16 weight / bias pieces (at least 2^-25 per
 *          unit of |q| once a piece is an fp16 subnormal) and c_acc = 10: one
 *          truncation of the fp32 result per MMA, 5 MMAs.  Measured on a
 *          B200: the accumulation error per step is <= 2.96 * 2^-24 M, and the
 *          accumulation truncates -- with bias 1 and no input the membrane
 *          stays at 1 - 2^-24 from step 24 on and never fires, where the
 *          reference rounds 1 - 2^-25 up to 1.0 and fires at step 25.
 *          Envelope: all 128 channels share one power-of-two domain scale,
 *          fitted to the largest 63.5 * |scale| or |bias| / 2 (fully pruned
 *          channels included).  A channel ~100x the others (all weights
 *          pruned, running var 0) stays inside both bars; with one channel
 *          2^16 or 2^20 times the others the other channels' lo weight
 *          pieces become fp16 subnormals: membranes then miss 1e-5 by up to
 *          2.3e-4 relative (B200), which the band's 2^-25 floor accounts for
 *          (measured at 0.56 and 0.90 of delta_T), and the flip bar holds.
 *          Use EXACT or FAST for such checkpoints. */
#define SNNQP_LIF_TENSOR 2

/* SpikingBlock(QuantConv 3x3 pad 1, BatchNorm, multi_step_LIF) over T steps
 * with zero initial carry (spiking_learning.py:441-472), optionally followed
 * by the 2x2 max-pool.
 *   x       uint8 [T,B,H,W,Cin] via strides (event counts or {0,1} spikes)
 *   att     NULL, or fp32 per-(t,b,cin) multiplier: input = att * x
 *           (TCJA output y = x_seq * att, models.py:97).  With att, x holds
 *           spikes: any non-zero x byte is a spike (input = att), on every
 *           implementation.  tcgen05 (SNNQP_IMPL_TCGEN05 / AUTO): att in [0, 1]
 *           as 24-bit fixed point, round(att 2^24) half to even clamped to
 *           0xFFFFFF (1.0 reads as 1 - 2^-24), three exact byte-plane
 *           contractions S2, S1, S0 recombined as fma((float)S2, 65536,
 *           fma((float)S1, 256, (float)S0)) * 2^-24: |acc - sum att x q| <=
 *           sum |q| 2^-25 (2^-24 where clamped) + 5 2^-24 M, M = 2^-24 (2^16 |S2|
 *           + 2^8 |S1| + |S0|).  SIMT: one sequential fp32 fma chain per output
 *           (kh, kw, channel ascending; dense: k ascending).  Both are bit-exact
 *           to an emulation (tests/attref.py), which a float64 LIF band checks
 *           (tests/test_gpu_attention_path.py).
 *   wq      blob from snnqp_pack_conv3x3 (Cin==128) or snnqp_pack_conv1 (Cin==2)
 *   scale/bias fp32 [Cout] from snnqp_fold_affine
 *   spikes  uint8 [T,B,H',W',Cout] via strides, H' = H/2 if pool else H
 *   u_final NULL or fp32 [B][H][W][Cout]: membrane after the last step
 *   acc_dump NULL or [T][B][H][W][Cout] contiguous: int32 accumulators
 *           (fp32 accumulators when att != NULL) -- parity instrumentation. */
int snnqp_spiking_conv3x3_fwd(const snnqp_block_params *p, const uint8_t *x,
                              const float *att, const int8_t *wq,
                              const float *scale, const float *bias,
                              uint8_t *spikes, float *u_final, void *acc_dump,
                              void *stream);

/* Same, plus spike_counts (nullable): int32 [B][T][Cout], caller-zeroed;
 * += the number of UN-pooled spikes of each (b, t, channel) -- the numerator of
 * the TCJA mean over (h, w) (models.py:42) -- so that the attention can be
 * computed without materialising the un-pooled spikes (snnqp_tcja_fwd with
 * spikes == NULL).  On the tcgen05 path att must lie in [0, 1] (it is a
 * sigmoid): it is evaluated as 24-bit fixed point (three u8 byte planes). */
int snnqp_spiking_conv3x3_counts_fwd(const snnqp_block_params *p, const uint8_t *x,
                                     const float *att, const int8_t *wq,
                                     const float *scale, const float *bias,
                                     uint8_t *spikes, float *u_final, void *acc_dump,
                                     int32_t *spike_counts, void *stream);

/* Plain quantized contraction behind the QuantDense facade (flax_qdense.py:
 * 59-106, lax.dot_general :87-89) and the 1-D k = 4 'SAME' QuantConv facade
 * (flax_qconv.py:131-168 as TCJA uses it, examples/tcja/models.py:52-59,77-84;
 * rows = im2col of the (1, 2)-padded input):
 *   y[m][n] = (sum_k x[m][k] * q[k][n]) * scale[0]
 * x: fp32 or uint8 [M][K] contiguous; q_kn: int8 levels in the reference's own
 * (in, out) / (k, in, out) layout (snnqp_pack_levels); scale: device scalar
 * c / L (snnqp_fold_affine, n = 1).  Not a hot-path call. */
int snnqp_qlinear_fwd(const void *x, int x_is_u8, const int8_t *q_kn,
                      const float *scale, int64_t M, int K, int N, float *y,
                      void *stream);

/* SpikingBlock(QuantDense, multi_step_LIF), no norm (models.py:200-246).
 *   x uint8 [T,B,Cin] via strides; wq int8 [Cout][k_pad] with k_pad = Cin
 *   rounded up to 16; att as above with index k % att_mod. */
int snnqp_spiking_dense_fwd(const snnqp_block_params *p, const uint8_t *x,
                            const float *att, const int8_t *wq,
                            const float *scale, const float *bias,
                            uint8_t *spikes, float *u_final, void *acc_dump,
                            void *stream);

/* Plain QuantConv 3x3 forward (no norm / neuron): y fp32 [T,B,H,W,Cout]
 * contiguous = acc * scale + bias (flax_qconv.py:158-168 on packed weights). */
int snnqp_qconv3x3_fwd(const snnqp_block_params *p, const uint8_t *x,
                       const int8_t *wq, const float *scale, const float *bias,
                       float *y, void *stream);

/* TCJA attention (models.py:41-95) from the block's un-pooled spikes.
 *   spikes uint8 [T,B,H,W,C] via p->x_stride_*;  p->Cin = C; NULL => counts
 *          already holds the spike counts (snnqp_spiking_conv3x3_counts_fwd)
 *   wq_t int8 levels of the (4,T,T) kernel, wq_c of the (4,C,C) kernel, both in
 *   the reference's own (k,in,out) layout (snnqp_pack_levels)
 *   scale_t / scale_c: device scalars c / L / (H*W) (snnqp_fold_affine, n=1)
 *   counts  workspace int32 [B][T][C]
 *   att     fp32 out, [(t,b)][C] via p->att_stride_* */
int snnqp_tcja_fwd(const snnqp_block_params *p, const uint8_t *spikes,
                   const int8_t *wq_t, const int8_t *wq_c, const float *scale_t,
                   const float *scale_c, int32_t *counts, float *att,
                   void *stream);

/* 2x2 / stride 2 max-pool of uint8 spikes (models.py:145-147,185-187) for the
 * blocks whose un-pooled spikes are also needed (TCJA): x [T,B,H,W,C] via
 * p->x_stride_*, y [T,B,H/2,W/2,C] via p->y_stride_*, C = p->Cin. */
int snnqp_maxpool2_fwd(const snnqp_block_params *p, const uint8_t *x, uint8_t *y,
                       void *stream);

/* vote (models.py:253-255): logits[b][g] = mean_j mean_t spikes[t,b,g*group+j]. */
int snnqp_vote_fwd(const uint8_t *spikes, int T, int B, int N, int group,
                   int64_t stride_t, int64_t stride_b, float *logits,
                   void *stream);

/* compute_metrics with mse_loss (train_utils.py:209-225): out[0] += number of
 * argmax hits, out[1] += sum of squared errors vs one-hot (fp32 atomics). */
int snnqp_eval_metrics(const float *logits, const int32_t *labels, int B,
                       int classes, float *out2, void *stream);

/* Spike-tile skip statistics of the bit-packed tcgen05 3x3 block: an input
 * box (one 16x8 tile x one timestep) whose bits are all zero issues no MMAs (its
 * accumulators are taken as 0; the LIF update still runs).  *skipped / *total =
 * boxes skipped / seen by all launches since the last reset (device-wide
 * counters; the call synchronises with the device). */
int snnqp_tile_skip_stats(int64_t *skipped, int64_t *total, int reset);

/* Number of kernels this library has launched on this thread since the last
 * call with reset != 0 (bench.py's gpu_launches). */
int64_t snnqp_launch_count(int reset);

/* ---- rows next to the hot path (SURVEY.md section 8f) ----------------------
 * Event -> frame integration, "split by number" (examples/input_pipeline.py:
 * 142-219 preprocess_data_number): addrs = int32 [N_total][3] (x, y, p) records
 * of all samples back to back in time order, offsets = int64 [B+1] record
 * offsets.  Sample b's events are cut into T groups of N_b / T events (the
 * last takes the remainder); group t is histogrammed into frame (b, t):
 * cell (floor(y/rs)*wh + floor(x/rs), p != 0), wh = sensor_wh / rs (floor, as
 * the reference's floor-division: a negative coordinate rounds down, so (-1, y)
 * at rs = 2 is the previous row's last pixel).  frames: [B][T][wh][wh][2]
 * uint8 saturating at 255 (out_int32 == 0; *n_saturated += saturated cells, may
 * be NULL) or exact int32 (out_int32 != 0).  Like the reference, the FLAT
 * position is histogrammed (an x beyond the row lands in the next row); only
 * positions outside the frame are dropped (the reference's scatter would fail
 * on them).  max_events_per_sample: an upper bound of offsets[b+1]-offsets[b]
 * known to the caller (it built the offsets), or 0 if unknown; when it proves
 * every frame holds < 65536 events the histogram uses 16-bit counters (three
 * frames in flight per SM instead of one).  Results are identical either way. */
int snnqp_events_to_frames(const int32_t *addrs, const int64_t *offsets, int B,
                           int T, int sensor_wh, int resolution_scale,
                           int64_t max_events_per_sample, void *frames,
                           int out_int32, uint64_t *n_saturated, void *stream);

/* Packed event words: the host -> device wire format of event input.  One word
 * per event, in time order:
 *   SNNQP_EVENTS_U16  uint16 w: x = w & 0x7F, y = (w >> 7) & 0x7F, p = w >> 15;
 *                     bit 14 is zero.  Every x, y < 128 (a 128 x 128 sensor).
 *   SNNQP_EVENTS_U32  uint32 w: x = w & 0x7FFF, y = (w >> 15) & 0x7FFF,
 *                     p = w >> 31; bit 30 is zero.  Every x, y < 32768.
 * p is the polarity bit (p != 0 of the record).  Encoder on the host:
 * snnquantprune_b200/input_pipeline.py (encode_events). */
#define SNNQP_EVENTS_U16 1
#define SNNQP_EVENTS_U32 2

/* snnqp_events_to_frames on packed event words (event_format = SNNQP_EVENTS_*):
 * same split, cells, flat-position rule, saturation and counter choice.  Sample
 * b's events are events[offsets[b] - event_base, offsets[b+1] - event_base):
 * a batch is encoded once, and any sample range [b0, b1) is then the words
 * [offsets[b0], offsets[b1]) plus offsets[b0 .. b1], shipped as they are with
 * event_base = offsets[b0].  events and frames must be 16-byte aligned (the
 * words are read as 16-byte vectors; group bounds may fall at any word). */
int snnqp_events_to_frames_packed(const void *events, int event_format,
                                  const int64_t *offsets, int64_t event_base,
                                  int B, int T, int sensor_wh,
                                  int resolution_scale,
                                  int64_t max_events_per_sample, void *frames,
                                  int out_int32, uint64_t *n_saturated,
                                  void *stream);

/* Activation-density numerators (examples/tcja/models.py:128-142 sows
 * sum(x != 0) over (H,W,C) per (t,b) slice / slice size, then max and mean):
 * counts[i] = number of non-zero bytes of slice i (slice_bytes long, slices
 * stride_slice apart).  counts is zeroed by the call. */
int snnqp_slice_nonzeros(const uint8_t *x, int n_slices, int64_t slice_bytes,
                         int64_t stride_slice, int32_t *counts, void *stream);

/* Zero-suppressed frames: the host -> device wire format of the end-to-end path.
 * The reference hands the model dense (T, H, W, 2) event-count frames
 * (examples/input_pipeline.py:142-219, train_inpt_spikingjelly.py:300-305); they
 * are mostly zeros, and at 8 GPUs the dense uint8 frames saturate the host ->
 * device links.  Cells are the flattened [B][T][H][W][2] frame bytes in blocks
 * of 1024 (n_cells % 1024 == 0):
 *   bitmap    uint32 [n_blocks][32]: bit (i & 31) of word (i >> 5) <=> cell i != 0
 *   block_off uint32 [n_blocks + 1]: index (in values, counted in elements)
 *             of each block's first value, minus value_base -- a batch is encoded
 *             once and any sample range of it can be shipped and expanded
 *   values    the non-zero counts in cell order, value_bits = 4 (low nibble
 *             first; every count <= 15) or 8 bits each
 * Writes frames uint8 [n_blocks * 1024] (16-byte aligned).  Encoder / decoder on
 * the host: snnquantprune_b200/input_pipeline.py (zsf_encode), oracle/ref_events.py. */
int snnqp_expand_frames_zsf(const uint32_t *bitmap, const uint32_t *block_off,
                            const uint8_t *values, uint32_t value_base,
                            int64_t n_blocks, int value_bits, uint8_t *frames,
                            void *stream);

/* Same for a bit-packed spike tensor (SNNQP_SPIKES_BITS): counts[s] = set bits
 * of slice s -- the same numerator, one eighth of the bytes. */
int snnqp_slice_popcount(const uint8_t *x, int n_slices, int64_t slice_bytes,
                         int64_t stride_slice, int32_t *counts, void *stream);

/* Diagnostic (no reference counterpart): dense int8 tensor-pipe ceiling of the
 * current device -- back-to-back tcgen05.mma.kind::i8 128x256x32 from shared
 * memory on every SM, best of `reps` launches of `iters` x 4 MMAs per SM, in
 * TOP/s.  bench.py uses it as the roofline denominator of the tensor-bound
 * kernels (MEASURED_PEAKS.json holds no int8 figure).  Synchronises `stream`. */
int snnqp_diag_imma_peak(int iters, int reps, double *tops_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SNNQP_H_ */
