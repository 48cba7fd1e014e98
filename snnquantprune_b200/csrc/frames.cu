// The rows either side of the hot path (SURVEY.md section 8f, N3 / N4) -- HBM-bound integer kernels.
//
// k_events_to_frames: DVS events -> event-count frames, "split by number"
//   (reference examples/input_pipeline.py:142-219, preprocess_data_number): the N events of a sample are
//   cut into T consecutive groups of di = N / T events (the last group takes the remainder), and each
//   group is histogrammed into a (wh, wh, 2) frame: cell = (floor(y / rs) * wh + floor(x / rs)) * 2 + (p != 0).
//   One CTA per (sample, frame): the whole histogram lives in shared memory (64 KB at wh = 128 with 16-bit
//   counters -- three frames in flight per SM; 128 KB with 32-bit ones), events are read once (coalesced 12-byte
//   int32 records, or 2- / 4-byte packed words in 16-byte vectors: snnqp_events_to_frames_packed), all atomics are shared-memory
//   atomics, and the frame leaves as one pass of 128-bit stores in the hot path's own input layout
//   [B][T][H][W][2] (uint8, saturating, saturated cells counted; or exact int32).
//
// k_slice_nonzeros: number of non-zero bytes of each (t, b) slice of a u8 activation tensor -- the
//   numerator of the densities the reference sows (examples/tcja/models.py:128-142: sum(x != 0) over
//   (H, W, C) per (t, b), then max / mean on the host).
#include <type_traits>

#include "common.cuh"

namespace snnqp {
namespace {

// Event record decoders.  I32x3: int32 (x, y, p) triples.  U16 / U32: one packed word per event (include/snnqp.h,
// SNNQP_EVENTS_U16 / _U32), read as 16-byte vectors over the aligned interior of each group.
struct EvI32x3 {};
struct EvU16 {
  using Word = uint16_t;
  __device__ static void decode(uint32_t w, int &x, int &y, int &p) { x = w & 0x7F; y = (w >> 7) & 0x7F; p = w >> 15; }
};
struct EvU32 {
  using Word = uint32_t;
  __device__ static void decode(uint32_t w, int &x, int &y, int &p) { x = w & 0x7FFF; y = (w >> 15) & 0x7FFF; p = w >> 31; }
};

// PACKED: the two polarity counters of a pixel share one 32-bit word (16 bits each) -- 64 KB per frame at
// wh = 128, three CTAs per SM; exact while a frame holds < 65536 events (the launcher checks the caller's bound).
// !PACKED: one int32 per cell (128 KB, one CTA per SM), exact for any count.
// Sample b's events are events[offsets[b] - event_base, offsets[b + 1] - event_base).
template <typename Dec, typename OutT, bool PACKED>
__global__ void __launch_bounds__(512, PACKED ? 3 : 1)
k_events_to_frames(const void *__restrict__ events, const int64_t *__restrict__ offsets, int64_t event_base, int T,
                   int wh, int rs, OutT *__restrict__ frames, unsigned long long *__restrict__ n_saturated) {
  extern __shared__ int hist[];
  const int b = blockIdx.x / T, t = blockIdx.x % T;
  const int pixels = wh * wh;
  const int words = PACKED ? pixels : 2 * pixels;
  for (int i = threadIdx.x; i < words / 4; i += blockDim.x) reinterpret_cast<int4 *>(hist)[i] = make_int4(0, 0, 0, 0);
  __syncthreads();
  const int64_t e0 = offsets[b] - event_base, n = offsets[b + 1] - offsets[b];
  const int64_t di = n / T;
  const int64_t lo = e0 + (int64_t)t * di, hi = (t < T - 1) ? lo + di : e0 + n;
  // the reference histograms the FLAT position y*wh + x (input_pipeline.py:196-199): an x beyond the row
  // lands in the next row, exactly as there; only positions outside the frame are dropped
  auto count = [&](int x, int y, int p) {
    const int64_t pos = (int64_t)y * wh + x;
    if (pos >= 0 && pos < (int64_t)pixels) {
      if constexpr (PACKED) atomicAdd(hist + pos, p != 0 ? 0x10000 : 1);
      else atomicAdd(hist + (pos << 1) + (p != 0 ? 1 : 0), 1);
    }
  };
  if constexpr (std::is_same<Dec, EvI32x3>::value) {
    // 12-byte records: three coalesced word streams.  Coordinates may be negative here: floor(v / rs), as the
    // reference's float floor-division (input_pipeline.py:183-190), not C's truncation toward zero
    const int32_t *addrs = static_cast<const int32_t *>(events);
    auto floor_div = [rs](int v) { return v >= 0 ? v / rs : -1 - (-1 - v) / rs; };
    for (int64_t e = lo + threadIdx.x; e < hi; e += blockDim.x)
      count(floor_div(__ldg(addrs + 3 * e)), floor_div(__ldg(addrs + 3 * e + 1)), __ldg(addrs + 3 * e + 2));
  } else {
    using W = typename Dec::Word;
    constexpr int V = 16 / sizeof(W);                   // words per 16-byte vector (events is 16-byte aligned)
    const W *ev = static_cast<const W *>(events);
    auto one = [&](uint32_t w) {
      int x, y, p;
      Dec::decode(w, x, y, p);
      count(x / rs, y / rs, p);
    };
    // [v0, v1): the whole vectors inside [lo, hi); the head [lo, V v0) and tail [V v1, hi) go word by word
    const int64_t v0 = (lo + V - 1) / V, v1 = hi / V > v0 ? hi / V : v0;
    const int64_t head_end = V * v0 < hi ? V * v0 : hi;
    for (int64_t e = lo + threadIdx.x; e < head_end; e += blockDim.x) one(__ldg(ev + e));
    for (int64_t e = (V * v1 > head_end ? V * v1 : head_end) + threadIdx.x; e < hi; e += blockDim.x) one(__ldg(ev + e));
    const uint4 *vec = reinterpret_cast<const uint4 *>(ev);
    for (int64_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
      const uint4 q = __ldg(vec + v);
      const uint32_t q4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if constexpr (sizeof(W) == 2) {
          one(q4[k] & 0xFFFFu);
          one(q4[k] >> 16);
        } else {
          one(q4[k]);
        }
      }
    }
  }
  __syncthreads();
  // cell c of the frame = (pixel c >> 1, polarity c & 1)
  auto cell4 = [&](int i) {          // cells 4i .. 4i+3
    if constexpr (PACKED) {
      const int2 w = reinterpret_cast<const int2 *>(hist)[i];
      return make_int4(w.x & 0xFFFF, (int)((uint32_t)w.x >> 16), w.y & 0xFFFF, (int)((uint32_t)w.y >> 16));
    } else {
      return reinterpret_cast<const int4 *>(hist)[i];
    }
  };
  const int cells = 2 * pixels;
  OutT *dst = frames + ((int64_t)b * T + t) * cells;
  if constexpr (sizeof(OutT) == 4) {
    for (int i = threadIdx.x; i < cells / 4; i += blockDim.x) reinterpret_cast<int4 *>(dst)[i] = cell4(i);
  } else {
    unsigned sat = 0;
    for (int i = threadIdx.x; i < cells / 16; i += blockDim.x) {
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int4 v = cell4(4 * i + k);
        sat += (v.x > 255) + (v.y > 255) + (v.z > 255) + (v.w > 255);
        w[k] = (uint32_t)min(v.x, 255) | ((uint32_t)min(v.y, 255) << 8) | ((uint32_t)min(v.z, 255) << 16) |
               ((uint32_t)min(v.w, 255) << 24);
      }
      reinterpret_cast<uint4 *>(dst)[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (n_saturated) {
      for (int off = 16; off > 0; off >>= 1) sat += __shfl_xor_sync(0xffffffffu, sat, off);
      if ((threadIdx.x & 31) == 0 && sat) atomicAdd(n_saturated, (unsigned long long)sat);
    }
  }
}

// grid: (blocks_per_slice, n_slices); 16 bytes per thread per iteration
// BITS: the tensor is bit-packed spikes (SNNQP_SPIKES_BITS): count set bits instead of non-zero bytes
template <bool BITS>
__global__ void __launch_bounds__(256)
k_slice_nonzeros(const uint8_t *__restrict__ x, int64_t slice_bytes, int64_t stride_slice, int vec16,
                 int32_t *__restrict__ counts) {
  const uint8_t *base = x + (int64_t)blockIdx.y * stride_slice;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
  const int64_t n16 = vec16 ? slice_bytes / 16 : 0;           // unaligned slices: byte path only
  int c = 0;
  for (int64_t i = tid; i < n16; i += nthr) {
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(base) + i);
    // non-zero bytes of a word: bit 7 of ((b & 0x7F) + 0x7F) | b, per byte
    auto nzb = [](uint32_t w) { return BITS ? __popc(w) : __popc(((w & 0x7F7F7F7Fu) + 0x7F7F7F7Fu | w) & 0x80808080u); };
    c += nzb(v.x) + nzb(v.y) + nzb(v.z) + nzb(v.w);
  }
  for (int64_t i = n16 * 16 + tid; i < slice_bytes; i += nthr) c += BITS ? __popc((uint32_t)base[i]) : (base[i] != 0);
  for (int off = 16; off > 0; off >>= 1) c += __shfl_xor_sync(0xffffffffu, c, off);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(counts + blockIdx.y, c);
}

}  // namespace
}  // namespace snnqp

namespace snnqp {
template <typename Dec, typename OutT, bool PACKED>
static int launch_events(const void *events, const int64_t *offsets, int64_t event_base, int B, int T, int wh, int rs,
                         OutT *frames, unsigned long long *n_sat, cudaStream_t st) {
  const size_t smem = (size_t)(PACKED ? 1 : 2) * wh * wh * sizeof(int);
  auto k = k_events_to_frames<Dec, OutT, PACKED>;
  SNNQP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<B * T, 512, smem, st>>>(events, offsets, event_base, T, wh, rs, frames, n_sat);
  SNNQP_POST_LAUNCH("k_events_to_frames");
  return SNNQP_OK;
}

// checks shared by both entry points (events, offsets and frames are non-null), then the launch
template <typename Dec>
static int events_to_frames(const char *fn, const void *events, const int64_t *offsets, int64_t event_base, int B,
                            int T, int sensor_wh, int resolution_scale, int64_t max_events_per_sample, void *frames,
                            int out_int32, uint64_t *n_saturated, cudaStream_t st) {
  if (B <= 0 || T <= 0 || sensor_wh <= 0 || resolution_scale <= 0) return invalid("%s: B, T, wh, scale must be > 0", fn);
  const int wh = sensor_wh / resolution_scale;
  if (wh <= 0 || (2 * wh * wh) % 16) return invalid("%s: 2*wh*wh must be a multiple of 16 (wh = %d)", fn, wh);
  if ((size_t)2 * wh * wh * sizeof(int) > 200 * 1024)
    return unsupported("%s: frame of %d x %d x 2 does not fit the shared-memory histogram", fn, wh, wh);
  if (reinterpret_cast<uintptr_t>(frames) & 15) return invalid("%s: frames must be 16-byte aligned", fn);
  // a frame holds at most N/T + (T-1) events: 16-bit counters are exact below 65536
  const bool packed = max_events_per_sample > 0 && max_events_per_sample / T + T < 65536;
  const int rs = resolution_scale;
  unsigned long long *ns = reinterpret_cast<unsigned long long *>(n_saturated);
  if (out_int32) {
    int32_t *f = static_cast<int32_t *>(frames);
    return packed ? launch_events<Dec, int32_t, true>(events, offsets, event_base, B, T, wh, rs, f, nullptr, st)
                  : launch_events<Dec, int32_t, false>(events, offsets, event_base, B, T, wh, rs, f, nullptr, st);
  }
  uint8_t *f = static_cast<uint8_t *>(frames);
  return packed ? launch_events<Dec, uint8_t, true>(events, offsets, event_base, B, T, wh, rs, f, ns, st)
                : launch_events<Dec, uint8_t, false>(events, offsets, event_base, B, T, wh, rs, f, ns, st);
}
}  // namespace snnqp

extern "C" int snnqp_events_to_frames(const int32_t *addrs, const int64_t *offsets, int B, int T, int sensor_wh,
                                      int resolution_scale, int64_t max_events_per_sample, void *frames, int out_int32,
                                      uint64_t *n_saturated, void *stream_) {
  using namespace snnqp;
  if (int r = require_device()) return r;
  if (!addrs || !offsets || !frames) return invalid("snnqp_events_to_frames: null pointer");
  return events_to_frames<EvI32x3>("snnqp_events_to_frames", addrs, offsets, 0, B, T, sensor_wh, resolution_scale,
                                   max_events_per_sample, frames, out_int32, n_saturated,
                                   static_cast<cudaStream_t>(stream_));
}

extern "C" int snnqp_events_to_frames_packed(const void *events, int event_format, const int64_t *offsets,
                                             int64_t event_base, int B, int T, int sensor_wh, int resolution_scale,
                                             int64_t max_events_per_sample, void *frames, int out_int32,
                                             uint64_t *n_saturated, void *stream_) {
  using namespace snnqp;
  static const char fn[] = "snnqp_events_to_frames_packed";
  if (int r = require_device()) return r;
  if (!events || !offsets || !frames) return invalid("%s: null pointer", fn);
  if (reinterpret_cast<uintptr_t>(events) & 15) return invalid("%s: events must be 16-byte aligned", fn);
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (event_format == SNNQP_EVENTS_U16)
    return events_to_frames<EvU16>(fn, events, offsets, event_base, B, T, sensor_wh, resolution_scale,
                                   max_events_per_sample, frames, out_int32, n_saturated, st);
  if (event_format == SNNQP_EVENTS_U32)
    return events_to_frames<EvU32>(fn, events, offsets, event_base, B, T, sensor_wh, resolution_scale,
                                   max_events_per_sample, frames, out_int32, n_saturated, st);
  return invalid("%s: event_format = %d (SNNQP_EVENTS_U16 or SNNQP_EVENTS_U32)", fn, event_format);
}

static int slice_count(const uint8_t *x, int n_slices, int64_t slice_bytes, int64_t stride_slice, int32_t *counts,
                       bool bits, void *stream_) {
  using namespace snnqp;
  if (int r = require_device()) return r;
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (!x || !counts) return invalid("snnqp_slice_nonzeros: null pointer");
  if (n_slices <= 0 || slice_bytes <= 0) return invalid("snnqp_slice_nonzeros: n_slices and slice_bytes must be > 0");
  const int vec16 = !((reinterpret_cast<uintptr_t>(x) & 15) || (stride_slice & 15));
  SNNQP_CUDA(cudaMemsetAsync(counts, 0, sizeof(int32_t) * n_slices, st));
  int bx = (int)((slice_bytes / 16 + 255) / 256);
  const int cap = (8 * sm_count() + n_slices - 1) / n_slices;          // ~8 CTAs per SM over the whole grid
  bx = bx < 1 ? 1 : (bx > cap ? (cap < 1 ? 1 : cap) : bx);
  for (int s0 = 0; s0 < n_slices; s0 += 65535) {                         // gridDim.y limit
    const int ns = n_slices - s0 < 65535 ? n_slices - s0 : 65535;
    if (bits)
      k_slice_nonzeros<true><<<dim3(bx, ns), 256, 0, st>>>(x + (int64_t)s0 * stride_slice, slice_bytes, stride_slice, vec16,
                                                           counts + s0);
    else
      k_slice_nonzeros<false><<<dim3(bx, ns), 256, 0, st>>>(x + (int64_t)s0 * stride_slice, slice_bytes, stride_slice, vec16,
                                                            counts + s0);
    count_launch();
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_slice_nonzeros");
  return SNNQP_OK;
}

extern "C" int snnqp_slice_nonzeros(const uint8_t *x, int n_slices, int64_t slice_bytes, int64_t stride_slice,
                                    int32_t *counts, void *stream_) {
  return slice_count(x, n_slices, slice_bytes, stride_slice, counts, false, stream_);
}

extern "C" int snnqp_slice_popcount(const uint8_t *x, int n_slices, int64_t slice_bytes, int64_t stride_slice,
                                    int32_t *counts, void *stream_) {
  return slice_count(x, n_slices, slice_bytes, stride_slice, counts, true, stream_);
}

// ---------------------------------------------------------------------------------------------------------
// Zero-suppressed frames (the host -> device wire format of the end-to-end path).  DVS event-count frames are
// mostly zeros (the reference's frames, input_pipeline.py:142-219, are dense (T, H, W, 2) arrays; the synthetic
// workload has ~14 % non-zero cells), and at 8 GPUs the dense uint8 frames saturate the box's host -> device
// bandwidth.  Wire format per batch of cells (flattened [B][T][H][W][2], 1024 cells per block):
//   bitmap      uint32 [n_blocks][32]   bit (i & 31) of word i >> 5 set <=> cell i is non-zero
//   block_off   uint32 [n_blocks + 1]   running count of non-zero cells before each block
//   values      the non-zero counts in cell order: 4 bits each (value_bits == 4: low nibble first; every count
//               <= 15) or 8 bits each (value_bits == 8)
// k_expand_zsf: one warp per block; lane l owns word l (32 cells): warp prefix sum of the popcounts locates its
// values; the 32 expanded bytes leave as two 128-bit stores.  Bytes moved: ~(1/8 + density * value_bits / 8) per
// cell in, 1 per cell out.
namespace snnqp {
namespace {
template <int VB>
__global__ void __launch_bounds__(256)
k_expand_zsf(const uint32_t *__restrict__ bitmap, const uint32_t *__restrict__ block_off,
             const uint8_t *__restrict__ values, uint32_t value_base, int64_t n_blocks, uint8_t *__restrict__ frames) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t blk = warp; blk < n_blocks; blk += nwarps) {
    const uint32_t bits = __ldg(bitmap + blk * 32 + lane);
    const int n = __popc(bits);
    int incl = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    uint32_t pos = __ldg(block_off + blk) - value_base + (uint32_t)(incl - n);       // index of this lane's first value
    uint32_t out[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t rem = bits;
    while (rem) {
      const int i = __ffs(rem) - 1;
      rem &= rem - 1;
      uint32_t v;
      if (VB == 4) v = (__ldg(values + (pos >> 1)) >> ((pos & 1) * 4)) & 0xFu;
      else v = __ldg(values + pos);
      ++pos;
      out[i >> 2] |= v << ((i & 3) * 8);
    }
    uint4 *dst = reinterpret_cast<uint4 *>(frames + (blk * 32 + lane) * 32);
    dst[0] = make_uint4(out[0], out[1], out[2], out[3]);
    dst[1] = make_uint4(out[4], out[5], out[6], out[7]);
  }
}
}  // namespace
}  // namespace snnqp

extern "C" int snnqp_expand_frames_zsf(const uint32_t *bitmap, const uint32_t *block_off, const uint8_t *values,
                                       uint32_t value_base, int64_t n_blocks, int value_bits, uint8_t *frames,
                                       void *stream_) {
  using namespace snnqp;
  if (int r = require_device()) return r;
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (!bitmap || !block_off || !values || !frames) return invalid("snnqp_expand_frames_zsf: null pointer");
  if (n_blocks <= 0) return invalid("snnqp_expand_frames_zsf: n_blocks must be > 0");
  if (value_bits != 4 && value_bits != 8) return invalid("snnqp_expand_frames_zsf: value_bits=%d (4 or 8)", value_bits);
  if (reinterpret_cast<uintptr_t>(frames) & 15) return invalid("snnqp_expand_frames_zsf: frames must be 16-byte aligned");
  int64_t g = (n_blocks + 7) / 8;                      // 8 warps per CTA
  const int64_t cap = (int64_t)sm_count() * 16;
  if (g > cap) g = cap;
  if (value_bits == 4) k_expand_zsf<4><<<(int)g, 256, 0, st>>>(bitmap, block_off, values, value_base, n_blocks, frames);
  else k_expand_zsf<8><<<(int)g, 256, 0, st>>>(bitmap, block_off, values, value_base, n_blocks, frames);
  SNNQP_POST_LAUNCH("k_expand_zsf");
  return SNNQP_OK;
}
