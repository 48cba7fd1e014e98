// tcgen05 kernels for the layers whose inputs are real-valued: x = att * s with
// s a {0,1} spike and att in [0,1] the TCJA sigmoid attention (reference
// examples/tcja/models.py:95-97; consumers conv5 models.py:150-173 and dense1
// models.py:200-216), plus the binary dense2 (models.py:231-246).
//
// att is taken as 24-bit fixed point, att ~= (b2*2^16 + b1*2^8 + b0) * 2^-24
// with u8 bytes b_i, so that
//     sum_k att_k s_k q_k = 2^-24 * (2^16 * S2 + 2^8 * S1 + S0),  S_i = sum_k (s_k ? b_i,k : 0) * q_k
// and each S_i is an EXACT u8 x s8 -> s32 tensor-core contraction over the same
// packed weights as the binary layers.  "Expander" warps build the three byte
// planes (spike mask AND attention byte; any non-zero x byte is a spike) straight
// into the swizzled MMA operand layout; the epilogue recombines the three
// accumulators in fp32.  The arithmetic is deterministic and exact but for:
//  * ptx::att_fix24: round(att * 2^24) half to even, clamped to 0xFFFFFF, so
//    |att - fix * 2^-24| <= 2^-25, and 2^-24 for att = 1.0 (read as 1 - 2^-24);
//  * ptx::att_combine: f1 = fma((float)S1, 256, (float)S0), then
//    f = fma((float)S2, 65536, f1), then the exact * 2^-24 -- five roundings,
//    each only once a value passes 2^24, each <= 2^-24 M with
//    M = 2^-24 (2^16 |S2| + 2^8 |S1| + |S0|).
// So |acc - sum att s q| <= sum_k s_k |q_k| 2^-25 (2^-24 where clamped) + 5 * 2^-24 M.
// tests/test_gpu_attention_path.py holds both kernels bit-exact to a numpy
// emulation of exactly these steps (tests/attref.py) and checks a float64 band
// on that emulation (T = 20, sigmoid-shaped att: ~1e-5 of the conv5
// neuron-steps undecided, none in dense1).
//
//  * k_conv_att_umma : 3x3 conv on 8-wide images (conv5), flat-shift implicit
//    GEMM exactly as umma_conv.cu, three accumulators per buffer.
//  * k_dense_umma    : [features] x [K] x [(b,t) rows] GEMM with the LIF
//    recurrence over t running along the accumulator columns of one lane.
#include <mutex>

#include "common.cuh"
#include "ptx.cuh"

namespace snnqp {

namespace {

constexpr int kC = 128;
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode2() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

__device__ __forceinline__ uint32_t nz_mask4(uint32_t w) { return __vcmpne4(w, 0u); }   // 0xFF per non-zero byte

// =====================================================================================
// conv-att: W = 8, strips of 8 rows, P = 10, N = 80
// =====================================================================================
namespace ca {
// The three byte planes are INTERLEAVED at position granularity: operand row 3*pos + plane, accumulator column
// 3*pos + plane.  A flat shift by s positions is then a shift by 3*s rows, and ONE MMA of N = 240 covers the 80 flat
// positions of all three planes: 36 MMAs per step at the full-width rate instead of 108 of N = 80 (N = 80 runs at
// 75 % of the N = 240 rate: profiles/README.md).
constexpr int W = 8, TH = 8, P = 10, N = 80, NI = 3 * N;
constexpr int kPlaneBytes = 13312;                 // 104 rows x 128 B (>= 2P+2+N rows) per plane
constexpr int kStageBytes = 3 * kPlaneBytes;       // 312 interleaved rows, 1024-aligned
constexpr int kWBytes = 9 * kC * kC, kTapBytes = kC * kC;
constexpr int kEpiWarps = 8, kExpWarps = 4;
constexpr int kThreads = (kEpiWarps + 1 + kExpWarps) * 32;   // 416
constexpr int kAccStride = 256;
constexpr int kSmemBytes = kWBytes + 2 * kStageBytes + 3 * kC * 2 /*att planes x2*/ + 256 + 1024;
}  // namespace ca

struct ConvAttArgs {
  int T, B, H;
  int strips, total_items;
  int64_t x_stride_t, x_stride_b, y_stride_t, y_stride_b, att_stride_t, att_stride_b;
  float tau, v_th, v_reset;
  int pool;
  const uint8_t *x;
  const float *att;
  const float *scale, *bias;
  const uint8_t *slab_nz;
  uint8_t *spikes;
  float *u_final;
  float *acc_dump;
  int32_t *counts;             // [B][T][C] += un-pooled spike count (nullable)
};

template <bool TAU2>
__global__ void __launch_bounds__(ca::kThreads, 1)
k_conv_att_umma(const __grid_constant__ CUtensorMap tmap_w, const ConvAttArgs a) {
  using namespace ca;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t *w_smem = smem;
  uint8_t *stage_smem = smem + kWBytes;
  uint8_t *att_smem = stage_smem + 2 * kStageBytes;            // [2][3][128] attention bytes
  uint64_t *bars = reinterpret_cast<uint64_t *>(att_smem + 2 * 3 * kC);
  uint64_t *w_full = bars, *in_full = bars + 1, *in_empty = bars + 3, *acc_full = bars + 5, *acc_empty = bars + 7;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 9);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // zero the operand stages once: the rows past the box are only ever read into garbage columns
  for (int i = threadIdx.x; i < 2 * kStageBytes / 16; i += kThreads)
    reinterpret_cast<int4 *>(stage_smem)[i] = make_int4(0, 0, 0, 0);
  ptx::fence_proxy_async();
  if (warp == kEpiWarps && lane == 0) {
    ptx::prefetch_tmap(&tmap_w);
    ptx::mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(in_full + i, kExpWarps);
      ptx::mbar_init(in_empty + i, 1);
      ptx::mbar_init(acc_full + i, 1);
      ptx::mbar_init(acc_empty + i, kEpiWarps);
    }
    ptx::fence_barrier_init();
  }
  if (warp == kEpiWarps) ptx::tmem_alloc<512>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kEpiWarps) {
    // ===================== weights TMA + MMA issuer =====================
    if (ptx::elect_one()) {
      ptx::mbar_expect_tx(w_full, kWBytes);
      for (int tap = 0; tap < 9; ++tap) ptx::tma_load_2d(w_smem + tap * kTapBytes, &tmap_w, w_full, 0, tap * kC);
      uint64_t nz_mask = ~0ull;
      if (a.slab_nz) {
        nz_mask = 0;
        for (int i = 0; i < 36; ++i) nz_mask |= (uint64_t)(a.slab_nz[i] != 0) << i;
        if (nz_mask == 0) nz_mask = 1;
      }
      const uint32_t idesc = ptx::make_idesc_i8(128, NI, true, false);
      const uint32_t w_addr = ptx::smem_u32(w_smem);
      const uint64_t desc_hi = ptx::make_desc_sw128(0, 0);
      const bool dense_path = (nz_mask & 0xFFFFFFFFFull) == 0xFFFFFFFFFull;
      ptx::mbar_wait(w_full, 0);
      uint32_t step = 0;
      for (int item = blockIdx.x; item < a.total_items; item += gridDim.x) {
        for (int t = 0; t < a.T; ++t, ++step) {
          const uint32_t s = step & 1, ph = (step >> 1) & 1;
          ptx::mbar_wait(acc_empty + s, ph ^ 1);
          ptx::mbar_wait(in_full + s, ph);
          ptx::tc_fence_after();
          const uint32_t x_addr = ptx::smem_u32(stage_smem + s * kStageBytes);
          // descriptors: constant high half + 14-bit start address in 16-byte units (never carries out)
          const uint64_t ad0 = desc_hi + (w_addr >> 4);
          const uint32_t d_tmem = tmem_base + s * kAccStride;
          const uint64_t bd0 = desc_hi + (x_addr >> 4);
          if (dense_path) {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap)
#pragma unroll
              for (int k = 0; k < 4; ++k)
                ptx::mma_i8(d_tmem, ad0 + (tap * kTapBytes + k * 32) / 16,
                            bd0 + (3 * ((tap / 3) * P + (tap % 3)) * 128 + k * 32) / 16, idesc, (tap | k) != 0);
          } else {
            uint32_t accumulate = 0;
#pragma unroll 1
            for (int sl = 0; sl < 36; ++sl) {
              if (!((nz_mask >> sl) & 1)) continue;      // block-sparse skip of an all-zero K-slab
              const int tap = sl >> 2, k = sl & 3;
              ptx::mma_i8(d_tmem, ad0 + (tap * kTapBytes + k * 32) / 16,
                          bd0 + (3 * ((tap / 3) * P + (tap % 3)) * 128 + k * 32) / 16, idesc, accumulate);
              accumulate = 1;
            }
          }
          ptx::mma_commit(in_empty + s);
          ptx::mma_commit(acc_full + s);
        }
      }
    }
  } else if (warp > kEpiWarps) {
    // ===================== expander warps: spikes AND attention bytes -> 3 operand planes =====================
    const int et = threadIdx.x - (kEpiWarps + 1) * 32;   // 0..127
    uint32_t step = 0;
    for (int item = blockIdx.x; item < a.total_items; item += gridDim.x) {
      const int b = item / a.strips, h0 = (item % a.strips) * TH;
      for (int t = 0; t < a.T; ++t, ++step) {
        const uint32_t s = step & 1, ph = (step >> 1) & 1;
        // attention bytes of this (t, b): thread = channel
        uint8_t *ab = att_smem + s * 3 * kC;
        const uint32_t fx = ptx::att_fix24(a.att[(int64_t)t * a.att_stride_t + (int64_t)b * a.att_stride_b + et]);
        // every global load of the step (the attention word above and the thread's 7 spike chunks) is issued BEFORE
        // the wait for the stage: the loads do not depend on it, and their latency then hides behind the MMAs that
        // still read the stage (the ncu source view had the expanders 69 % of their time on these loads)
        const uint8_t *xb = a.x + (int64_t)t * a.x_stride_t + (int64_t)b * a.x_stride_b;
        constexpr int kChunks = (TH + 2) * P * 8, kIt = (kChunks + kExpWarps * 32 - 1) / (kExpWarps * 32);
        int4 sv[kIt];
#pragma unroll
        for (int it = 0; it < kIt; ++it) {
          const int ch = et + it * kExpWarps * 32;
          const int pix = ch >> 3, c16 = ch & 7;
          const int ih = h0 - 1 + pix / P, iw = pix % P - 1;
          sv[it] = make_int4(0, 0, 0, 0);
          if (ch < kChunks && ih >= 0 && ih < a.H && iw >= 0 && iw < W)
            sv[it] = __ldg(reinterpret_cast<const int4 *>(xb + ((int64_t)ih * W + iw) * kC + c16 * 16));
        }
        ptx::mbar_wait(in_empty + s, ph ^ 1);        // stage (and its att bytes) no longer read by the MMAs
        ab[0 * kC + et] = (uint8_t)(fx >> 16);
        ab[1 * kC + et] = (uint8_t)(fx >> 8);
        ab[2 * kC + et] = (uint8_t)fx;
        ptx::named_bar_sync(1, kExpWarps * 32);
        uint8_t *dst = stage_smem + s * kStageBytes;
#pragma unroll
        for (int it = 0; it < kIt; ++it) {
          const int ch = et + it * kExpWarps * 32;
          if (ch >= kChunks) break;
          const int pix = ch >> 3, c16 = ch & 7;
          const uint32_t m0 = nz_mask4(sv[it].x), m1 = nz_mask4(sv[it].y), m2 = nz_mask4(sv[it].z), m3 = nz_mask4(sv[it].w);
#pragma unroll
          for (int pl = 0; pl < 3; ++pl) {
            const int4 av = *reinterpret_cast<const int4 *>(ab + pl * kC + c16 * 16);
            int4 o;
            o.x = (int)(m0 & (uint32_t)av.x); o.y = (int)(m1 & (uint32_t)av.y);
            o.z = (int)(m2 & (uint32_t)av.z); o.w = (int)(m3 & (uint32_t)av.w);
            const int row = 3 * pix + pl;                  // interleaved operand row (swizzle on absolute row bits)
            *reinterpret_cast<int4 *>(dst + row * 128 + ((c16 ^ (row & 7)) << 4)) = o;
          }
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(in_full + s);
      }
    }
  } else {
    // ===================== epilogue =====================
    const int q = warp & 3, g = warp >> 2;
    const int c = q * 32 + lane;
    const float sc = a.scale[c], bi = a.bias[c];
    const int r0 = g * 4;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int Wo = a.pool ? W / 2 : W;
    float u[4][8];
    uint32_t step = 0;
    for (int item = blockIdx.x; item < a.total_items; item += gridDim.x) {
      const int b = item / a.strips, h0 = (item % a.strips) * TH;
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int j = 0; j < 8; ++j) u[r][j] = 0.0f;
      for (int t = 0; t < a.T; ++t, ++step) {
        const uint32_t s = step & 1, ph = (step >> 1) & 1;
        ptx::mbar_wait(acc_full + s, ph);
        ptx::tc_fence_after();
        uint32_t acc[4][24];                               // [row][3 * column + plane]
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const uint32_t taddr = lane_addr + s * kAccStride + 3 * (r0 + r) * P;
          uint32_t lo[16], hi[8];
          SNNQP_TMEM_LD_X16(taddr, lo);
          SNNQP_TMEM_LD_X8(taddr + 16, hi);
#pragma unroll
          for (int i = 0; i < 16; ++i) acc[r][i] = lo[i];
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[r][16 + i] = hi[i];
        }
        ptx::tc_wait_ld();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(acc_empty + s);

        uint32_t m[4];
        int nspk = 0;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          m[r] = 0;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float accf = ptx::att_combine((int32_t)acc[r][3 * j], (int32_t)acc[r][3 * j + 1], (int32_t)acc[r][3 * j + 2]);
            const float v = __fmaf_rn(accf, sc, bi);
            bool sp;
            if constexpr (TAU2) {
              const float un = __fadd_rn(u[r][j], __fmul_rn(__fsub_rn(v, __fsub_rn(u[r][j], a.v_reset)), 0.5f));
              sp = __fsub_rn(un, a.v_th) >= 0.0f;
              u[r][j] = sp ? a.v_reset : un;
            } else {
              u[r][j] = lif_step(u[r][j], v, a.tau, a.v_th, a.v_reset, sp);
            }
            m[r] |= (sp ? 1u : 0u) << j;
            if (a.acc_dump)
              a.acc_dump[((((int64_t)t * a.B + b) * a.H + h0 + r0 + r) * W + j) * kC + c] = accf;
          }
          nspk += __popc(m[r]);
        }
        if (a.counts && nspk) atomicAdd(a.counts + ((int64_t)b * a.T + t) * kC + c, nspk);
        uint8_t *yb = a.spikes + (int64_t)t * a.y_stride_t + (int64_t)b * a.y_stride_b + c;
        if (a.pool) {
#pragma unroll
          for (int pr = 0; pr < 2; ++pr) {
            uint32_t mm = m[2 * pr] | m[2 * pr + 1];
            mm |= mm >> 1;
            const int ho = (h0 + r0 + 2 * pr) >> 1;
#pragma unroll
            for (int pc = 0; pc < 4; ++pc) yb[((int64_t)ho * Wo + pc) * kC] = (mm >> (2 * pc)) & 1u;
          }
        } else {
#pragma unroll
          for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int j = 0; j < 8; ++j) yb[((int64_t)(h0 + r0 + r) * Wo + j) * kC] = (m[r] >> j) & 1u;
        }
      }
      if (a.u_final) {
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int j = 0; j < 8; ++j) a.u_final[(((int64_t)b * a.H + h0 + r0 + r) * W + j) * kC + c] = u[r][j];
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kEpiWarps) {
    __syncwarp();
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

// =====================================================================================
// dense: D[feature, (b,t)] = sum_k Wq[feature][k] * X[(b,t)][k], LIF along t
// =====================================================================================
namespace dn {
constexpr int kEpiWarps = 8, kExpWarps = 4;
constexpr int kThreads = (kEpiWarps + 1 + kExpWarps) * 32;   // 416
constexpr int kMaxN = 160;
constexpr int kABytes = 128 * 128;                 // weights k-block: 128 features x 128 B
constexpr int kBPlane = kMaxN * 128;               // 20480
}  // namespace dn

struct DenseArgs {
  int T, B, K, Nout;
  int planes;                  // 1 (binary input) or 3 (att-weighted input)
  int NB, N;                   // samples / columns per tile
  int m_tiles, col_tiles, total_items;
  int64_t y_stride_t, y_stride_b, att_stride_t, att_stride_b;
  int att_mod;
  float tau, v_th, v_reset;
  const uint8_t *x;            // [B*T][K] contiguous, row = b*T + t
  const float *att;
  const float *scale, *bias;
  uint8_t *spikes;
  float *u_final;
  void *acc_dump;
};

template <int PLANES, bool TAU2>
__global__ void __launch_bounds__(dn::kThreads, 1)
k_dense_umma(const __grid_constant__ CUtensorMap tmap_w, const DenseArgs a) {
  using namespace dn;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t *a_smem = smem;                                   // [2][16 KB]
  uint8_t *b_smem = a_smem + 2 * kABytes;                   // [2][PLANES][20 KB]
  uint8_t *att_smem = b_smem + 2 * PLANES * kBPlane;        // [PLANES][kMaxN][128] attention bytes of the tile rows
  uint64_t *bars = reinterpret_cast<uint64_t *>(att_smem + (PLANES == 3 ? 3 * kBPlane : 0));
  uint64_t *a_full = bars, *b_full = bars + 2, *ab_empty = bars + 4, *acc_full = bars + 6, *acc_empty = bars + 7;
  uint64_t *att_ready = bars + 8;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 10);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == kEpiWarps && lane == 0) {
    ptx::prefetch_tmap(&tmap_w);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(a_full + i, 1);
      ptx::mbar_init(b_full + i, kExpWarps);
      ptx::mbar_init(ab_empty + i, 1);
    }
    ptx::mbar_init(acc_full, 1);
    ptx::mbar_init(acc_empty, kEpiWarps);
    ptx::fence_barrier_init();
  }
  if (warp == kEpiWarps) ptx::tmem_alloc<512>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int kblocks = a.K / 128;
  const int rows_total = a.B * a.T;

  if (warp == kEpiWarps) {
    // ===================== weight TMA + MMA issuer =====================
    if (ptx::elect_one()) {
      const uint32_t idesc = ptx::make_idesc_i8(128, a.N, true, false);
      uint32_t kstep = 0, it = 0;
      const int my_items = (int)blockIdx.x < a.total_items
                               ? (a.total_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
      const uint32_t total_steps = (uint32_t)my_items * (uint32_t)kblocks;
      // weight tile of global step g (item-major, K-block minor); issued one step ahead of the MMAs so that
      // the TMA latency overlaps the previous K-block's MMAs
      auto issue_load = [&](uint32_t g) {
        const uint32_t s = g & 1, ph = (g >> 1) & 1;
        const int item = (int)blockIdx.x + (int)(g / kblocks) * (int)gridDim.x;
        ptx::mbar_wait(ab_empty + s, ph ^ 1);
        ptx::mbar_expect_tx(a_full + s, kABytes);
        ptx::tma_load_2d(a_smem + s * kABytes, &tmap_w, a_full + s, (int)(g % kblocks) * 128, (item % a.m_tiles) * 128);
      };
      if (total_steps) issue_load(0);
      for (int item = blockIdx.x; item < a.total_items; item += gridDim.x, ++it) {
        for (int kb = 0; kb < kblocks; ++kb, ++kstep) {
          const uint32_t s = kstep & 1, ph = (kstep >> 1) & 1;
          if (kstep + 1 < total_steps) issue_load(kstep + 1);
          if (kb == 0) ptx::mbar_wait(acc_empty, (it & 1) ^ 1);
          ptx::mbar_wait(a_full + s, ph);
          ptx::mbar_wait(b_full + s, ph);
          ptx::tc_fence_after();
          const uint32_t aa0 = ptx::smem_u32(a_smem + s * kABytes);
          const uint32_t bb0 = ptx::smem_u32(b_smem + s * PLANES * kBPlane);
#pragma unroll
          for (int pl = 0; pl < PLANES; ++pl)
#pragma unroll
            for (int k = 0; k < 4; ++k)
              ptx::mma_i8(tmem_base + pl * kMaxN, ptx::make_desc_sw128(aa0 + k * 32, 0),
                          ptx::make_desc_sw128(bb0 + pl * kBPlane + k * 32, 0), idesc, (kb | k) != 0);
          ptx::mma_commit(ab_empty + s);
        }
        ptx::mma_commit(acc_full);
      }
    }
  } else if (warp > kEpiWarps) {
    // ===================== expander warps: build the B operand (rows = (b,t)) =====================
    const int et = threadIdx.x - (kEpiWarps + 1) * 32;
    uint32_t kstep = 0;
    for (int item = blockIdx.x; item < a.total_items; item += gridDim.x) {
      const int ct = item / a.m_tiles;
      const int row0 = ct * a.N;
      if (PLANES == 3) {
        // attention bytes of the tile rows, once per item: [pl][row][128]
        ptx::named_bar_sync(1, kExpWarps * 32);          // previous item's expander reads are done
        // four channels per thread and iteration (one 16-byte load, three word stores), eight independent loads in
        // flight: one scalar load per iteration left ~160 exposed global-memory latencies per item and made this
        // loop, not the MMAs, the kernel's critical path
        constexpr int kU = 8;
        for (int i0 = et; i0 < a.N * (kC / 4); i0 += kU * kExpWarps * 32) {
          float4 v[kU];
#pragma unroll
          for (int u = 0; u < kU; ++u) {
            const int i4 = i0 + u * kExpWarps * 32;
            const int row = row0 + (i4 >> 5);
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i4 < a.N * (kC / 4) && row < rows_total) {
              const int b = row / a.T, t = row % a.T;
              v[u] = __ldg(reinterpret_cast<const float4 *>(a.att + (int64_t)t * a.att_stride_t + (int64_t)b * a.att_stride_b) +
                           (i4 & 31));
            }
          }
#pragma unroll
          for (int u = 0; u < kU; ++u) {
            const int i4 = i0 + u * kExpWarps * 32;
            if (i4 >= a.N * (kC / 4)) break;
            const uint32_t f0 = ptx::att_fix24(v[u].x), f1 = ptx::att_fix24(v[u].y), f2 = ptx::att_fix24(v[u].z),
                           f3 = ptx::att_fix24(v[u].w);
            // byte plane pl of channels (4k .. 4k+3): byte (2 - pl) of each fixed-point word
            const uint32_t lo01 = __byte_perm(f0, f1, 0x5140), lo23 = __byte_perm(f2, f3, 0x5140);   // (f0.b0 f1.b0 f0.b1 f1.b1)
            const uint32_t hi01 = __byte_perm(f0, f1, 0x7362), hi23 = __byte_perm(f2, f3, 0x7362);   // (f0.b2 f1.b2 f0.b3 f1.b3)
            uint32_t *dst = reinterpret_cast<uint32_t *>(att_smem) + i4;
            dst[0 * (kBPlane / 4)] = __byte_perm(hi01, hi23, 0x5410);      // b2 of the four channels
            dst[1 * (kBPlane / 4)] = __byte_perm(lo01, lo23, 0x7632);      // b1
            dst[2 * (kBPlane / 4)] = __byte_perm(lo01, lo23, 0x5410);      // b0
          }
        }
        ptx::named_bar_sync(1, kExpWarps * 32);
      }
      for (int kb = 0; kb < kblocks; ++kb, ++kstep) {
        const uint32_t s = kstep & 1, ph = (kstep >> 1) & 1;
        // all of this thread's global loads are issued first (and before the stage barrier), so their
        // latency overlaps the MMAs of the previous K-blocks instead of being paid one chunk at a time
        constexpr int kMaxCh = (kMaxN * 8 + kExpWarps * 32 - 1) / (kExpWarps * 32);
        int4 svs[kMaxCh];
#pragma unroll
        for (int i = 0; i < kMaxCh; ++i) {
          const int ch = et + i * kExpWarps * 32;
          const int row = row0 + (ch >> 3);
          svs[i] = make_int4(0, 0, 0, 0);
          if (ch < a.N * 8 && row < rows_total)
            svs[i] = __ldg(reinterpret_cast<const int4 *>(a.x + (int64_t)row * a.K + kb * 128 + (ch & 7) * 16));
        }
        ptx::mbar_wait(ab_empty + s, ph ^ 1);
        uint8_t *dst = b_smem + s * PLANES * kBPlane;
#pragma unroll
        for (int i = 0; i < kMaxCh; ++i) {
          const int ch = et + i * kExpWarps * 32;
          if (ch >= a.N * 8) break;
          const int r = ch >> 3, c16 = ch & 7;
          const int4 sv = svs[i];
          const uint32_t off = (uint32_t)(r * 128 + ((c16 ^ (r & 7)) << 4));
          if (PLANES == 1) {
            *reinterpret_cast<int4 *>(dst + off) = sv;
          } else {
            const uint32_t m0 = nz_mask4(sv.x), m1 = nz_mask4(sv.y), m2 = nz_mask4(sv.z), m3 = nz_mask4(sv.w);
#pragma unroll
            for (int pl = 0; pl < 3; ++pl) {
              const int4 av = *reinterpret_cast<const int4 *>(att_smem + pl * kBPlane + r * 128 + c16 * 16);
              int4 o;
              o.x = (int)(m0 & (uint32_t)av.x); o.y = (int)(m1 & (uint32_t)av.y);
              o.z = (int)(m2 & (uint32_t)av.z); o.w = (int)(m3 & (uint32_t)av.w);
              *reinterpret_cast<int4 *>(dst + pl * kBPlane + off) = o;
            }
          }
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(b_full + s);
      }
    }
  } else {
    // ===================== epilogue: LIF along the columns (t) of each sample =====================
    const int q = warp & 3, g = warp >> 2;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t it = 0;
    for (int item = blockIdx.x; item < a.total_items; item += gridDim.x, ++it) {
      const int mt = item % a.m_tiles, ct = item / a.m_tiles;
      const int n = mt * 128 + q * 32 + lane;
      const bool act = n < a.Nout;
      const float sc = act ? a.scale[n] : 0.f, bi = act ? a.bias[n] : 0.f;
      const int half = a.N / 2;
      const int col0 = g * half;                      // starts on a sample boundary (NB is even)
      ptx::mbar_wait(acc_full, it & 1);
      ptx::tc_fence_after();
      float u = 0.f;
      int tcur = 0;
      int b = ct * a.NB + g * (a.NB / 2);
      for (int cc = 0; cc < half; cc += 8) {
        uint32_t acc[PLANES][8];
#pragma unroll
        for (int pl = 0; pl < PLANES; ++pl) {
          const uint32_t taddr = lane_addr + pl * kMaxN + col0 + cc;
          SNNQP_TMEM_LD_X8(taddr, acc[pl]);
        }
        ptx::tc_wait_ld();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (tcur == 0) u = 0.f;
          float f;
          if (PLANES == 3) f = ptx::att_combine((int32_t)acc[0][j], (int32_t)acc[PLANES - 1 > 0 ? 1 : 0][j], (int32_t)acc[PLANES - 1][j]);
          else f = (float)(int32_t)acc[0][j];
          const float v = __fmaf_rn(f, sc, bi);
          bool sp;
          if constexpr (TAU2) {
            const float un = __fadd_rn(u, __fmul_rn(__fsub_rn(v, __fsub_rn(u, a.v_reset)), 0.5f));
            sp = __fsub_rn(un, a.v_th) >= 0.0f;
            u = sp ? a.v_reset : un;
          } else {
            u = lif_step(u, v, a.tau, a.v_th, a.v_reset, sp);
          }
          if (act && b < a.B) {
            a.spikes[(int64_t)tcur * a.y_stride_t + (int64_t)b * a.y_stride_b + n] = sp ? 1 : 0;
            if (a.acc_dump) {
              const int64_t full = ((int64_t)tcur * a.B + b) * a.Nout + n;
              if (PLANES == 3) reinterpret_cast<float *>(a.acc_dump)[full] = f;
              else reinterpret_cast<int32_t *>(a.acc_dump)[full] = (int32_t)acc[0][j];
            }
            if (a.u_final && tcur == a.T - 1) a.u_final[(int64_t)b * a.Nout + n] = u;
          }
          if (++tcur == a.T) { tcur = 0; ++b; }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(acc_empty);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kEpiWarps) {
    __syncwarp();
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

int encode_weights_2d(CUtensorMap *tm, const int8_t *wq, uint64_t kbytes, uint64_t rows, const char *what) {
  EncodeTiledFn encode = get_encode2();
  if (!encode) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return SNNQP_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)kbytes, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)kbytes};
  cuuint32_t box[2] = {128, 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<int8_t *>(wq), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(%s) failed with CUresult %d", what, (int)r);
    return SNNQP_ERR_CUDA;
  }
  return SNNQP_OK;
}

int gcd_i(int x, int y) { return y == 0 ? x : gcd_i(y, x % y); }

// columns per tile: NB samples (even), NB*T a multiple of 16 and <= 160
bool dense_tile(int T, int *NB, int *N) {
  int nb0 = 16 / gcd_i(T, 16);
  if (nb0 & 1) nb0 *= 2;
  if (nb0 * T > dn::kMaxN) return false;
  *NB = nb0 * (dn::kMaxN / (nb0 * T));
  *N = *NB * T;
  return true;
}

}  // namespace

// ------------------------------------------------------------------ conv-att host ----
bool umma_conv_att_supported(const snnqp_block_params &p, const float *att) {
  if (!att || p.Cin != kC || p.Cout != kC || p.att_mod != kC) return false;
  if (p.W != ca::W || p.H % ca::TH != 0) return false;
  if (p.x_stride_t % 16 || p.x_stride_b % 16) return false;
  return true;
}

int launch_conv_att_umma(const snnqp_block_params &p, const uint8_t *x, const float *att, const int8_t *wq,
                         const float *scale, const float *bias, uint8_t *spikes, float *u_final, float *acc_dump,
                         int32_t *counts, cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(wq) & 15))
    return invalid("tcgen05 conv-att: x and wq must be 16-byte aligned");
  CUtensorMap tmw;
  if (int rc = encode_weights_2d(&tmw, wq, kC, 9 * kC, "conv-att w")) return rc;
  ConvAttArgs a;
  a.T = p.T; a.B = p.B; a.H = p.H;
  a.strips = p.H / ca::TH;
  a.total_items = p.B * a.strips;
  a.x_stride_t = p.x_stride_t; a.x_stride_b = p.x_stride_b;
  a.y_stride_t = p.y_stride_t; a.y_stride_b = p.y_stride_b;
  a.att_stride_t = p.att_stride_t; a.att_stride_b = p.att_stride_b;
  a.tau = p.tau; a.v_th = p.v_threshold; a.v_reset = p.v_reset;
  a.pool = p.pool;
  a.x = x; a.att = att; a.scale = scale; a.bias = bias;
  a.slab_nz = reinterpret_cast<const uint8_t *>(wq) + ca::kWBytes;
  a.spikes = spikes; a.u_final = u_final; a.acc_dump = acc_dump; a.counts = counts;
  const int grid = a.total_items < sm_count() ? a.total_items : sm_count();
  if (p.tau == 2.0f) {
    SNNQP_CUDA(cudaFuncSetAttribute(k_conv_att_umma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ca::kSmemBytes));
    k_conv_att_umma<true><<<grid, ca::kThreads, ca::kSmemBytes, st>>>(tmw, a);
  } else {
    SNNQP_CUDA(cudaFuncSetAttribute(k_conv_att_umma<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ca::kSmemBytes));
    k_conv_att_umma<false><<<grid, ca::kThreads, ca::kSmemBytes, st>>>(tmw, a);
  }
  SNNQP_POST_LAUNCH("k_conv_att_umma");
  return SNNQP_OK;
}

// ------------------------------------------------------------------ dense host ----
bool umma_dense_supported(const snnqp_block_params &p, const float *att, int k_pad) {
  int NB, N;
  if (p.Cin % 128 != 0 || k_pad != p.Cin) return false;
  if (!dense_tile(p.T, &NB, &N)) return false;
  if (p.x_stride_t != p.Cin || p.x_stride_b != (int64_t)p.T * p.Cin) return false;   // rows (b,t) contiguous
  if (att && p.att_mod != kC) return false;
  // the attention rows are read as float4
  if (att && ((reinterpret_cast<uintptr_t>(att) & 15) || (p.att_stride_t & 3) || (p.att_stride_b & 3))) return false;
  return true;
}

int launch_dense_umma(const snnqp_block_params &p, const uint8_t *x, const float *att, const int8_t *wq,
                      const float *scale, const float *bias, uint8_t *spikes, float *u_final, void *acc_dump,
                      cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(wq) & 15))
    return invalid("tcgen05 dense: x and wq must be 16-byte aligned");
  CUtensorMap tmw;
  if (int rc = encode_weights_2d(&tmw, wq, (uint64_t)p.Cin, (uint64_t)p.Cout, "dense w")) return rc;
  DenseArgs a;
  a.T = p.T; a.B = p.B; a.K = p.Cin; a.Nout = p.Cout;
  a.planes = att ? 3 : 1;
  dense_tile(p.T, &a.NB, &a.N);
  a.m_tiles = (p.Cout + 127) / 128;
  a.col_tiles = (p.B + a.NB - 1) / a.NB;
  a.total_items = a.m_tiles * a.col_tiles;
  a.y_stride_t = p.y_stride_t; a.y_stride_b = p.y_stride_b;
  a.att_stride_t = p.att_stride_t; a.att_stride_b = p.att_stride_b;
  a.att_mod = p.att_mod;
  a.tau = p.tau; a.v_th = p.v_threshold; a.v_reset = p.v_reset;
  a.x = x; a.att = att; a.scale = scale; a.bias = bias;
  a.spikes = spikes; a.u_final = u_final; a.acc_dump = acc_dump;
  const int grid = a.total_items < sm_count() ? a.total_items : sm_count();
  const bool tau2 = p.tau == 2.0f;
#define SNNQP_LAUNCH_DENSE(PL, T2)                                                                          \
  do {                                                                                                      \
    const int smem = 2 * dn::kABytes + 2 * PL * dn::kBPlane + (PL == 3 ? 3 * dn::kBPlane : 0) + 256 + 1024;  \
    SNNQP_CUDA(cudaFuncSetAttribute(k_dense_umma<PL, T2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
    k_dense_umma<PL, T2><<<grid, dn::kThreads, smem, st>>>(tmw, a);                                          \
  } while (0)
  if (att) { if (tau2) SNNQP_LAUNCH_DENSE(3, true); else SNNQP_LAUNCH_DENSE(3, false); }
  else { if (tau2) SNNQP_LAUNCH_DENSE(1, true); else SNNQP_LAUNCH_DENSE(1, false); }
#undef SNNQP_LAUNCH_DENSE
  SNNQP_POST_LAUNCH("k_dense_umma");
  return SNNQP_OK;
}

}  // namespace snnqp
