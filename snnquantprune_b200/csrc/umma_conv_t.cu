// Fused SpikingBlock(QuantConv3x3 -> BN -> LIF [-> 2x2 max-pool]) for binary / count inputs, Cin = Cout = 128, on
// tcgen05 with a PAD-FREE spatial tiling (reference semantics spiking_learning.py:441-472, flax_qconv.py:158-168,
// examples/tcja/models.py:101-147).
//
// A work item is a 16 x 8 SPATIAL tile: N = 128 output positions n = g * 8 + j (g = tile row 0..15, j = tile
// column 0..7).  The TMA box is 18 rows x 10 columns x 128 channels (zero-filled halo), 128-byte rows at pitch 10;
// for tap (kh, kw) tile row g is the 8 consecutive box rows starting at (g + kh) * 10 + kw -- exactly a K-major
// 128B-swizzle operand whose 8-row groups are 10 rows (1280 B) apart: the UMMA descriptor's stride-byte-offset
// carries the box pitch (SBO = 1280 instead of 1024), and because the swizzle is a function of absolute
// shared-memory address bits (measured in round 1) the groups may start at any 128-byte row.  So every issued MMA
// column is a real output: 36 MMAs of 128 x 128 x 32 per step.  Reading a strip of full rows at flat shifts of a
// (W+2)-pitch box instead needs N = 144 for the same 128 outputs (2 pad columns per row, rounded to 16): 11 % more
// tensor time and a 2x halo re-read against 1.4x here (DESIGN.md section 4.1).  One kernel shape serves every
// W % 8 == 0 and every even H: the last tile row of an image may be partial (see the epilogue).
#include <mutex>

#include "common.cuh"
#include "epilogue.cuh"
#include "ptx.cuh"
#include "tmap.cuh"

namespace snnqp {

namespace {

// timing-bisection switches exist only in SNNQP_BISECT builds (tools/): never in the shipped hot loops
#ifdef SNNQP_C1_BISECT
#define UMMA_DBG(bit) (a.debug & (bit))
#else
#define UMMA_DBG(bit) false
#endif

// spike-tile skip statistics of the bit-packed path: [0] all-zero input tiles whose 36 MMAs were skipped, [1] tiles seen
__device__ unsigned long long g_tile_skip_t[2];

constexpr int kC = 128;
constexpr int kWBytes = 9 * kC * kC;            // 147456
constexpr int kTapBytes = kC * kC;              // 16384
constexpr int kTileH = 16, kTileW = 8;          // output tile
constexpr int kBoxH = kTileH + 2, kBoxW = kTileW + 2, kBoxRows = kBoxH * kBoxW;   // 180 box positions
constexpr int kN = kTileH * kTileW;             // 128 = MMA N
constexpr int kStagesBits = 6;                  // operand ring depth of the bit-packed variant (expanders run further ahead)
constexpr int kSBO = kBoxW * 128;               // stride between the 8-row groups of the B operand: the box pitch
constexpr int kStageBytes = 23552;              // >= 180 rows * 128 B, 1024-aligned
// 16 epilogue warps: a thread owns one channel x 4 tile rows x 8 columns (32 membranes).  An epilogue warp is bound by
// its own dependent-instruction latency (~4 cycles per instruction), not by issue slots: with 8 warps x 64 neurons a
// step's epilogue took ~2500 cycles -- as long as its 36 MMAs (2304), which is why skipping MMAs (block-sparse weights,
// all-zero spike tiles) gained nothing (profiles/r2_sparse_paths_8warp_epilogue.jsonl); 16 warps halve that latency.
constexpr int kEpiWarps = 16;
constexpr int kRowsPerThread = kTileH / (kEpiWarps / 4);     // 4
constexpr int kColsPerThread = kRowsPerThread * kTileW;      // 32 accumulator columns per thread
// MMA issuers: a lone issuing thread needs ~72 cycles per tcgen05.mma next to the epilogue / expander warps of its SM
// sub-partition (the MMA itself runs 64), so with two issuers each one owns every other step (= one of the two
// accumulator buffers) and has two step times to issue its 36 MMAs (A/B: tools/run_r2_gpu35.sh).
#ifndef SNNQP_MMA_WARPS
#define SNNQP_MMA_WARPS 2
#endif
constexpr int kMmaWarps = SNNQP_MMA_WARPS;
constexpr int kThreads = (kEpiWarps + 1 + kMmaWarps) * 32;  // + TMA warp + MMA warp(s); the second MMA warp is the CTA's last
// Bit-packed input (SNNQP_SPIKES_BITS): TMA stages the packed tile (16 B per position), two expander warps turn
// bits into the u8 K-major 128B-swizzled MMA operand (3 integer ops per 4 bytes: nibble * 0x00204081 & 0x01010101).
#ifndef SNNQP_EXP_WARPS
#define SNNQP_EXP_WARPS 3
#endif
#ifndef SNNQP_T_TAPS
#define SNNQP_T_TAPS 7          // weight taps resident in TMEM (8 fills all 512 columns: A/B in tools/run_r2_gpu34.sh)
#endif
constexpr int kExpWarps = SNNQP_EXP_WARPS;   // 3 keeps the MMA issuer's SM sub-partition free of an expander warp (A/B: tools/run_r2_gpu17.sh)
constexpr int kThreadsX = kThreads + kExpWarps * 32;
constexpr int kPkStages = 6, kPkStageBytes = 2944;   // >= 180 * 16 B, 128-aligned
constexpr int kTmemCols = 512;
// Weights (A operand) of the first SNNQP_T_TAPS taps live in TENSOR MEMORY for the CTA's lifetime, so an MMA reads
// only its B operand from shared memory: an SS-mode MMA pulls (128 + N) * 32 B per ~64-72 cycles, near the 128 B/cycle
// port (measured 94 % of it for N = 144 in round 1, tensor pipe 57 % active).  TMEM budget: 2 x 128 accumulator columns
// + 7 taps x 4 K-steps x 8 columns = 480 of 512.  The other two taps stay in shared memory (32 KB).  How many taps sit
// in TMEM hardly matters (profiles/r2_conv2_tmem_split.txt).
constexpr int kAccStride = 128;                 // TMEM column offset of accumulator buffer 1
constexpr int kACol0 = 2 * kAccStride;          // first TMEM column of the resident weights
constexpr int smem_bytes_for(int tt, int st, bool xbits = false) {
  return (9 - tt) * kTapBytes + st * kStageBytes + (xbits ? kPkStages * kPkStageBytes : 0) + 1024 /*barriers*/ + 1024 /*align slack*/;
}

struct UmmaArgs {
  int T, B, H, W;
  int tiles_x, tiles_per_img, total_items;
  int64_t y_stride_t, y_stride_b;
  float tau, v_th, v_reset;
  int pool;
  int base_off_mode;
  int tb_swapped;            // tensor-map dims 3/4 are (b, t) instead of (t, b)
  int one;                   // always 1 (runtime operand of the magic-number IMAD, see epilogue.cuh)
  int y_bits;                // 1: emit bit-packed spikes (production variants only)
  int32_t *y_popcount;       // nullable [B][T]: += emitted spikes (y_bits only)
  int debug;                 // SNNQP_UMMA_DEBUG: bit0 skip MMA issue, bit1 skip epilogue math (timing bisection only)
  uint32_t stage_tx_bytes;
  const float *scale, *bias;
  const uint8_t *slab_nz;    // 36 flags (tap*4 + k32) or nullptr
  uint8_t *spikes;
  float *u_final;
  int32_t *acc_dump;
  int32_t *counts;           // [B][T][C] += un-pooled spike count (nullable)
  const int8_t *wq;          // packed weights [9][128][128] (read directly for the TMEM-resident taps)
};

// FAST: standard LIF constants (tau 2, threshold 1, reset 0), pooled output, no
// instrumentation outputs -- the production variant; !FAST handles everything else.
template <bool FAST, bool COUNTS, bool XBITS, bool POPC = false>
__global__ void __launch_bounds__(XBITS ? kThreadsX : kThreads, 1)
k_conv3x3_tile(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
               const UmmaArgs a) {
  constexpr int kTmemTaps = SNNQP_T_TAPS, kStages = XBITS ? kStagesBits : 4;
  constexpr int kWSmemBytes = (9 - kTmemTaps) * kTapBytes;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t *w_smem = smem;
  uint8_t *stage_smem = smem + kWSmemBytes;
  uint8_t *pk_smem = stage_smem + kStages * kStageBytes;          // XBITS: packed-tile ring
  uint64_t *bars = reinterpret_cast<uint64_t *>(pk_smem + (XBITS ? kPkStages * kPkStageBytes : 0));
  uint64_t *w_full = bars + 0;
  uint64_t *a_ready = bars + 1;                 // weights stored to TMEM by the epilogue warps
  uint64_t *in_full = bars + 2;                 // [kStages]
  uint64_t *in_empty = in_full + kStages;       // [kStages]
  uint64_t *acc_full = in_empty + kStages;      // [2]
  uint64_t *acc_empty = acc_full + 2;           // [2]
  uint64_t *pk_full = acc_empty + 2;             // [kPkStages]
  uint64_t *pk_empty = pk_full + kPkStages;      // [kPkStages]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(pk_empty + kPkStages);
  // spike-tile skip (XBITS): zin[stage] = 1 if the whole input box of that stage is zero (written by the expanders,
  // read by the MMA issuer), zacc[buffer] = 1 if the step of that accumulator buffer was skipped (MMA issuer ->
  // epilogue), wz[warp] = per-expander-warp "saw a set bit"
  volatile uint32_t *zin = tmem_slot + 1;
  volatile uint32_t *zacc = zin + kStages * kExpWarps;
  // block-sparse path: compact list of the non-zero K-slabs, built once by the MMA issuer:
  // .x = A operand (TMEM address, or low word of the shared-memory descriptor), .y = B row offset (16-byte units) * 2 + (A in TMEM)
  uint2 *slist = reinterpret_cast<uint2 *>(bars + 64);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == kEpiWarps && lane == 0) {
    ptx::prefetch_tmap(&tmap_x);
    ptx::prefetch_tmap(&tmap_w);
    ptx::mbar_init(w_full, 1);
    ptx::mbar_init(a_ready, kEpiWarps);
    for (int i = 0; i < kStages; ++i) {
      ptx::mbar_init(in_full + i, XBITS ? kExpWarps : 1);
      ptx::mbar_init(in_empty + i, 1);
    }
    for (int i = 0; i < kPkStages; ++i) {
      ptx::mbar_init(pk_full + i, 1);
      ptx::mbar_init(pk_empty + i, kExpWarps);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(acc_full + i, 1);
      ptx::mbar_init(acc_empty + i, kEpiWarps);
    }
    ptx::fence_barrier_init();
  }
  if (warp == kEpiWarps + 1) ptx::tmem_alloc<kTmemCols>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  constexpr int kMma1Warp = kEpiWarps + 2 + (XBITS ? kExpWarps : 0);      // (only with kMmaWarps == 2)
  if (warp == kEpiWarps) {
    // ===================== TMA producer =====================
    if (ptx::elect_one()) {
      if (kWSmemBytes) ptx::mbar_expect_tx(w_full, kWSmemBytes); else ptx::mbar_arrive(w_full);
      for (int tap = kTmemTaps; tap < 9; ++tap)
        ptx::tma_load_2d(w_smem + (tap - kTmemTaps) * kTapBytes, &tmap_w, w_full, 0, tap * kC);
      uint32_t step = 0;
      for (int item = blockIdx.x; item < a.total_items; item += gridDim.x) {
        const int b = item / a.tiles_per_img, tl = item % a.tiles_per_img;
        const int h0 = (tl / a.tiles_x) * kTileH, x0 = (tl % a.tiles_x) * kTileW;
        for (int t = 0; t < a.T; ++t, ++step) {
          if constexpr (XBITS) {
            const uint32_t s = step % kPkStages, ph = (step / kPkStages) & 1;
            ptx::mbar_wait(pk_empty + s, ph ^ 1);
            ptx::mbar_expect_tx(pk_full + s, a.stage_tx_bytes);
            ptx::tma_load_5d(pk_smem + s * kPkStageBytes, &tmap_x, pk_full + s, 0, x0 - 1, h0 - 1,
                             a.tb_swapped ? b : t, a.tb_swapped ? t : b);
          } else {
            const uint32_t s = step % kStages, ph = (step / kStages) & 1;
            ptx::mbar_wait(in_empty + s, ph ^ 1);
            ptx::mbar_expect_tx(in_full + s, a.stage_tx_bytes);
            ptx::tma_load_5d(stage_smem + s * kStageBytes, &tmap_x, in_full + s, 0, x0 - 1, h0 - 1,
                             a.tb_swapped ? b : t, a.tb_swapped ? t : b);
          }
        }
      }
    }
  } else if (warp == kEpiWarps + 1 || (kMmaWarps == 2 && warp == kMma1Warp)) {
    // ===================== MMA issuer(s) =====================
    const uint32_t mma_id = warp == kEpiWarps + 1 ? 0u : 1u;
    // The leader is chosen with elect.sync: inside a plain `lane == 0` branch ptxas treats the region as divergent
    // and wraps every UTCIMMA in an ELECT / BRA.U.ANY serialisation loop (~18 instructions per MMA, measured
    // 112 cycles per 128x144x32 MMA instead of 72).
    if (ptx::elect_one()) {
      uint64_t nz_mask = ~0ull;
      if (a.slab_nz) {
        nz_mask = 0;
        for (int i = 0; i < 36; ++i) nz_mask |= (uint64_t)(a.slab_nz[i] != 0) << i;
        if (nz_mask == 0) nz_mask = 1;   // keep one (all-zero) slab so the accumulator is still cleared
      }
      const uint32_t idesc = ptx::make_idesc_i8(128, kN, /*A = weights s8*/ true, /*B = inputs u8*/ false);
      const uint32_t w_addr = ptx::smem_u32(w_smem);
      const uint64_t desc_hi = ptx::make_desc_sw128(0, 0);                 // A (weights): 8-row groups 1024 B apart
      const uint64_t ad0 = desc_hi + (w_addr >> 4);
      // B (activations): same layout, but the 8-row groups (tile rows) are one box pitch apart
      const uint64_t bdesc_hi = (desc_hi & ~((uint64_t)0x3FFF << 32)) | ((uint64_t)(kSBO >> 4) << 32);
      uint32_t tap_off16[9];                       // (kh * P + kw) rows of 128 B, in 16-byte units
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) tap_off16[tap] = (uint32_t)(((tap / 3) * kBoxW + (tap % 3)) * 8);
      // The list-driven skip loop costs ~150 issue cycles per MMA against 72 in the unrolled dense sequence (a lone
      // issuing thread is bound by its dependent-instruction latency), so it only pays when at most a third of the 36
      // slabs is left (measured, profiles/r2_sparse_paths.jsonl); otherwise the zero slabs are simply multiplied.
      const bool dense_path = (__popcll(nz_mask & 0xFFFFFFFFFull) > 12) && !UMMA_DBG(1);
      int n_slabs = 0;
      if (!dense_path) {
        for (int sl = 0; sl < 36; ++sl) {
          if (!((nz_mask >> sl) & 1) || UMMA_DBG(1)) continue;
          const int tap = sl >> 2, k = sl & 3;
          const uint32_t boff = (uint32_t)(((tap / 3) * kBoxW + (tap % 3)) * 8 + 2 * k);
          if (tap < kTmemTaps) slist[n_slabs] = make_uint2(tmem_base + kACol0 + sl * 8, (boff << 1) | 1u);
          else slist[n_slabs] = make_uint2((w_addr + (tap - kTmemTaps) * kTapBytes + k * 32) >> 4, boff << 1);
          ++n_slabs;
        }
        slist[n_slabs] = make_uint2(0u, 0u);
      }
      ptx::mbar_wait(w_full, 0);
      ptx::mbar_wait(a_ready, 0);
      ptx::tc_fence_after();
      uint32_t step = 0;
      unsigned long long n_tiles = 0, n_skipped = 0;
      for (int item = blockIdx.x; item < a.total_items; item += gridDim.x) {
        for (int t = 0; t < a.T; ++t, ++step) {
          const uint32_t s = step & 1, ph = (step >> 1) & 1;
          const uint32_t si = step % kStages, phi = (step / kStages) & 1;
          if (kMmaWarps == 2 && s != mma_id) continue;          // the other issuer's step (and accumulator buffer)
          ptx::mbar_wait(acc_empty + s, ph ^ 1);
          ptx::mbar_wait(in_full + si, phi);
          if constexpr (XBITS) {
            // Spike-tile skip: an all-zero input box contributes nothing -- no MMAs; the epilogue takes acc = 0.
            // Plain (release) arrivals replace the two commits: nothing asynchronous was issued for this step.
            bool zero_tile = true;
#pragma unroll
            for (int i = 0; i < kExpWarps; ++i) zero_tile = zero_tile && zin[si * kExpWarps + i] != 0;
            zacc[s] = zero_tile ? 1u : 0u;
            ++n_tiles;
            if (zero_tile) {
              ++n_skipped;
              ptx::mbar_arrive(in_empty + si);
              ptx::mbar_arrive(acc_full + s);
              continue;
            }
          }
          ptx::tc_fence_after();
          const uint32_t x_addr = ptx::smem_u32(stage_smem + si * kStageBytes);
          const uint32_t d_tmem = tmem_base + s * kAccStride;
          // descriptors: constant high half; the 14-bit start-address field (16-byte units) is the only
          // part that changes, and shared-memory addresses never carry out of it
          const uint64_t bd0 = bdesc_hi + (x_addr >> 4);
          if (dense_path) {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const uint64_t bd_tap = bd0 + tap_off16[tap];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                if (tap < kTmemTaps)
                  ptx::mma_i8_ts(d_tmem, tmem_base + kACol0 + (tap * 4 + k) * 8, bd_tap + 2 * k, idesc, (tap | k) != 0);
                else
                  ptx::mma_i8(d_tmem, ad0 + ((tap - kTmemTaps) * kTapBytes + k * 32) / 16, bd_tap + 2 * k, idesc, (tap | k) != 0);
              }
            }
          } else {
            // block-sparse path: only the non-zero K-slabs, from the compact list (one 8-byte shared-memory load, one
            // add and the MMA per slab, the next entry prefetched: ~50 issue cycles per MMA < the 72 it runs).  r2
            // history (profiles/r2_sparse_paths.jsonl): a rolled loop doing the tap / k / descriptor arithmetic per slab
            // and a fully unrolled predicated sequence both cost ~3500 cycles per step whatever the number of slabs --
            // SLOWER than the 36 dense MMAs: a lone issuing thread is bound by its own dependent-instruction latency.
            uint2 e = slist[0];
#pragma unroll 1
            for (int i = 0; i < n_slabs; ++i) {
              const uint2 nx = slist[i + 1];          // slist has a sentinel entry
              const uint64_t bd = bd0 + (e.y >> 1);
              if (e.y & 1u) ptx::mma_i8_ts(d_tmem, e.x, bd, idesc, i != 0);
              else ptx::mma_i8(d_tmem, desc_hi + e.x, bd, idesc, i != 0);
              e = nx;
            }
          }
          ptx::mma_commit(in_empty + si);  // input stage reusable once these MMAs have read it
          ptx::mma_commit(acc_full + s);   // accumulator ready for the epilogue
        }
      }
      if (XBITS && n_tiles) {
        atomicAdd(&g_tile_skip_t[0], n_skipped);
        atomicAdd(&g_tile_skip_t[1], n_tiles);
      }
    }
  } else if (warp >= kEpiWarps + 2 && warp < kEpiWarps + 2 + kExpWarps) {
    // ===================== expanders (XBITS): packed bits -> u8 operand rows =====================
    if constexpr (XBITS) {
      const int et = threadIdx.x - (kEpiWarps + 2) * 32;          // 0 .. 32 * kExpWarps - 1
      constexpr int ntask = 2 * kBoxRows;                         // (position, 64-channel half)
      uint32_t step = 0;
      for (int item = blockIdx.x; item < a.total_items; item += gridDim.x) {
        for (int t = 0; t < a.T; ++t, ++step) {
          const uint32_t ps = step % kPkStages, pph = (step / kPkStages) & 1;
          const uint32_t si = step % kStages, phi = (step / kStages) & 1;
          ptx::mbar_wait(pk_full + ps, pph);
          ptx::mbar_wait(in_empty + si, phi ^ 1);
          const uint32_t src = ptx::smem_u32(pk_smem + ps * kPkStageBytes);
          const uint32_t dst = ptx::smem_u32(stage_smem + si * kStageBytes);
          // pass 1: this thread's packed words (<= kMaxTasks of them, kept in registers) and whether any bit is set
          constexpr int kMaxTasks = (ntask + 32 * kExpWarps - 1) / (32 * kExpWarps);
          uint2 pkd[kMaxTasks];
          uint32_t any = 0;
#pragma unroll
          for (int i = 0; i < kMaxTasks; ++i) {
            const int task = et + i * 32 * kExpWarps;
            pkd[i] = task < ntask ? ptx::lds64(src + (task >> 1) * 16 + (task & 1) * 8) : make_uint2(0u, 0u);
            any |= pkd[i].x | pkd[i].y;
          }
          // per-warp verdict (no cross-warp barrier): the MMA issuer skips the step only if ALL expander warps saw
          // zeros; a warp whose share is zero cannot know that, so it still writes its rows (as zeros, no arithmetic)
          any = __reduce_or_sync(0xffffffffu, any);
          if (lane == 0) zin[si * kExpWarps + (warp - (kEpiWarps + 2))] = any ? 0u : 1u;
          {
#pragma unroll
            for (int i = 0; i < kMaxTasks; ++i) {
              const int task = et + i * 32 * kExpWarps;
              if (task < ntask) {
                const int r = task >> 1, hf = task & 1;
                const uint32_t row = dst + r * 128;
#pragma unroll
                for (int k = 0; k < 4; ++k) {                           // 16 channels = one 16-byte chunk
                  const uint32_t h16 = ((k & 2) ? pkd[i].y : pkd[i].x) >> ((k & 1) * 16);
                  uint4 o;
                  o.x = ((h16 & 0xFu) * 0x00204081u) & 0x01010101u;
                  o.y = (((h16 >> 4) & 0xFu) * 0x00204081u) & 0x01010101u;
                  o.z = (((h16 >> 8) & 0xFu) * 0x00204081u) & 0x01010101u;
                  o.w = (((h16 >> 12) & 0xFu) * 0x00204081u) & 0x01010101u;
                  ptx::sts128(row + ((((hf << 2) | k) ^ (r & 7)) << 4), o);
                }
              }
            }
          }
          ptx::fence_proxy_async();          // generic-proxy writes -> visible to the tensor core (async proxy)
          __syncwarp();
          if (lane == 0) {
            ptx::mbar_arrive(in_full + si);
            ptx::mbar_arrive(pk_empty + ps);
          }
        }
      }
    }
  } else {
    // ===================== epilogue: dequant+BN affine, LIF, pool, store =====================
    const int q = warp & 3, g = warp >> 2;          // TMEM lane quarter, column group
    const int c = q * 32 + lane;                    // output channel
    const float sc = a.scale[c], bi = a.bias[c];
    // this thread's 32 outputs: tile rows 4g .. 4g+3 (accumulator columns 32g .. 32g+31), all 8 tile columns
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int Wo = a.pool ? a.W / 2 : a.W;
    {
      // one-time: this thread's weight row (output channel c) of the TMEM-resident taps -> tensor memory.
      // A-operand layout: lane = row, 32-bit column j of a K-step holds K bytes 4j .. 4j+3.
      for (int tap = g; tap < kTmemTaps; tap += kEpiWarps / 4) {        // the column groups share the taps
        const int4 *wrow = reinterpret_cast<const int4 *>(a.wq + ((int64_t)tap * kC + c) * kC);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int4 lo = __ldg(wrow + 2 * k), hi = __ldg(wrow + 2 * k + 1);
          const uint32_t wv[8] = {(uint32_t)lo.x, (uint32_t)lo.y, (uint32_t)lo.z, (uint32_t)lo.w,
                                  (uint32_t)hi.x, (uint32_t)hi.y, (uint32_t)hi.z, (uint32_t)hi.w};
          const uint32_t taddr = lane_addr + kACol0 + (tap * 4 + k) * 8;
          SNNQP_TMEM_ST_X8(taddr, wv);
        }
      }
      ptx::tc_wait_st();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(a_ready);
    }
    constexpr int RT = kRowsPerThread;
    float u[RT][8];                 // membranes [tile row - RT*g][tile column]: in registers for all T steps of a tile
    uint32_t step = 0;
    for (int item = blockIdx.x; item < a.total_items; item += gridDim.x) {
      const int b = item / a.tiles_per_img, tl = item % a.tiles_per_img;
      const int h0 = (tl / a.tiles_x) * kTileH + RT * g, x0 = (tl % a.tiles_x) * kTileW;   // first output row / column of this thread
      // Partial tile (the last tile row of an image with H % 16 != 0): its rows h0 + r >= H read TMA's zero fill and
      // run the LIF like the others, but nothing of them may leave the kernel.  H is even and h0 a multiple of 4, so
      // the two rows of a pooled pair are both inside or both outside.  FAST: such rows start at a NaN membrane, which
      // never reaches the threshold (epilogue.cuh), so they add nothing to ballots, counts or popcounts; only the
      // ballot-word store, which is addressed by row, tests the bound.  FAST with u8 output never gets a partial tile
      // (the host runs those on the generic epilogue), so its stores need no test.  Generic: their spike words are
      // cleared and their stores skipped.
      const bool partial = (tl / a.tiles_x) * kTileH + kTileH > a.H;
#pragma unroll
      for (int r = 0; r < RT; ++r)
#pragma unroll
        for (int j = 0; j < 8; ++j) u[r][j] = FAST && h0 + r >= a.H ? __int_as_float(0x7fc00000) : 0.0f;   // zero carry (spiking_learning.py:464-472)
      for (int t = 0; t < a.T; ++t, ++step) {
        const uint32_t s = step & 1, ph = (step >> 1) & 1;
        ptx::mbar_wait(acc_full + s, ph);
        ptx::tc_fence_after();
        const bool zstep = XBITS && zacc[s] != 0;
        const uint32_t tcol = lane_addr + s * kAccStride + kColsPerThread * g;
        if constexpr (FAST) {
          // Production epilogue: accumulators in chunks of 16 columns = 2 tile rows x 8 columns = 4 pooled outputs;
          // the TMEM buffer is released once the last chunk is in registers.  I2FP: exact for every int32.
          const LifParams<true> lifs{2.0f, 1.0f, 0.0f};
          int nspk = 0;
          uint32_t mine = 0;          // y_bits: the 32-channel word of pooled position `lane` (16 per thread-step)
#pragma unroll
          for (int ch = 0; ch < RT / 2; ++ch) {
            uint32_t av[16];
            if (!zstep) {
              SNNQP_TMEM_LD_X16(tcol + 16 * ch, av);
              ptx::tc_wait_ld();
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) av[j] = 0u;      // skipped all-zero tile: accumulators are 0
            }
            if (ch == RT / 2 - 1) {
              ptx::tc_fence_before();
              __syncwarp();
              if (lane == 0) ptx::mbar_arrive(acc_empty + s);        // TMEM buffer free for step + 2
            }
            uint8_t *yrow = a.spikes + (int64_t)t * a.y_stride_t + (int64_t)b * a.y_stride_b + c +
                            ((int64_t)((h0 >> 1) + ch) * Wo + (x0 >> 1)) * kC;
#pragma unroll
            for (int pc = 0; pc < 4; ++pc) {
              bool any = false;
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int r = 2 * ch + (e >> 1), j = 2 * pc + (e & 1);
                const bool sp = lifs.step(u[r][j], __fmaf_rn((float)(int32_t)av[8 * (e >> 1) + j], sc, bi));
                any |= sp;
                if constexpr (COUNTS) nspk += sp ? 1 : 0;
              }
              if (a.y_bits) {
                const uint32_t bal = __ballot_sync(0xffffffffu, any);
                if (lane == 4 * ch + pc) mine = bal;
              } else {
                yrow[pc * kC] = any ? 1 : 0;
              }
            }
          }
          if (a.y_bits && lane < (partial ? 2 * min(a.H - h0, RT) : 2 * RT)) {
            uint8_t *yw = a.spikes + (int64_t)t * a.y_stride_t + (int64_t)b * a.y_stride_b +
                          ((int64_t)((h0 >> 1) + (lane >> 2)) * Wo + (x0 >> 1) + (lane & 3)) * (kC / 8) + q * 4;
            *reinterpret_cast<uint32_t *>(yw) = mine;
          }
          if constexpr (POPC) {               // density numerator of the next layer's input, from the ballot words
            const int n = __reduce_add_sync(0xffffffffu, lane < 2 * RT ? __popc(mine) : 0);
            if (lane == 0 && n) atomicAdd(a.y_popcount + (int64_t)b * a.T + t, n);
          }
          if constexpr (COUNTS) {
            if (nspk) atomicAdd(a.counts + ((int64_t)b * a.T + t) * kC + c, nspk);
          }
          continue;
        }
        // generic / instrumented variant: any LIF constants, optional un-pooled output, membranes, accumulators
        uint32_t acc[RT][8];
#pragma unroll
        for (int r2 = 0; r2 < RT / 2; ++r2) {
          uint32_t av[16];
          if (zstep) {
#pragma unroll
            for (int j = 0; j < 16; ++j) av[j] = 0u;
          } else {
            SNNQP_TMEM_LD_X16(tcol + 16 * r2, av);
            ptx::tc_wait_ld();
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[2 * r2 + (j >> 3)][j & 7] = av[j];
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(acc_empty + s);        // TMEM buffer free for step + 2
        if (UMMA_DBG(2)) continue;
        const LifParams<false> lif{a.tau, a.v_th, a.v_reset};
        uint32_t m[RT];
        int nspk = 0;
#pragma unroll
        for (int r = 0; r < RT; ++r) {
          m[r] = 0;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const bool sp = lif.step(u[r][j], __fmaf_rn((float)(int32_t)acc[r][j], sc, bi));
            m[r] |= (sp ? 1u : 0u) << j;
          }
          if (h0 + r >= a.H) m[r] = 0;
          nspk += __popc(m[r]);
        }
        if (a.counts && nspk) atomicAdd(a.counts + ((int64_t)b * a.T + t) * kC + c, nspk);
        uint8_t *yb = a.spikes + (int64_t)t * a.y_stride_t + (int64_t)b * a.y_stride_b + c;
        if (a.pool) {
#pragma unroll
          for (int pr = 0; pr < RT / 2; ++pr) {
            if (h0 + 2 * pr >= a.H) break;
            uint32_t mm = m[2 * pr] | m[2 * pr + 1];
            mm |= mm >> 1;
#pragma unroll
            for (int pc = 0; pc < 4; ++pc)
              yb[((int64_t)((h0 >> 1) + pr) * Wo + (x0 >> 1) + pc) * kC] = (mm >> (2 * pc)) & 1u;
          }
        } else {
#pragma unroll
          for (int r = 0; r < RT; ++r) {
            if (h0 + r >= a.H) break;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              yb[((int64_t)(h0 + r) * Wo + x0 + j) * kC] = (m[r] >> j) & 1u;
          }
        }
        if (a.acc_dump) {
#pragma unroll
          for (int r = 0; r < RT; ++r) {
            if (h0 + r >= a.H) break;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              a.acc_dump[((((int64_t)t * a.B + b) * a.H + h0 + r) * a.W + x0 + j) * kC + c] = (int32_t)acc[r][j];
          }
        }
      }
      if (!FAST && a.u_final) {          // (the host runs FAST only without u_final)
#pragma unroll
        for (int r = 0; r < RT; ++r) {
          if (h0 + r >= a.H) break;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            a.u_final[(((int64_t)b * a.H + h0 + r) * a.W + x0 + j) * kC + c] = u[r][j];
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kEpiWarps + 1) {
    __syncwarp();
    ptx::tc_fence_after();
    ptx::tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// ---------------------------------------------------------------- host side ----
}  // namespace

bool umma_conv3x3_tile_supported(const snnqp_block_params &p, const float *att) {
  if (att) return false;
  if (p.Cin != kC || p.Cout != kC) return false;
  if (p.W % kTileW != 0) return false;       // any (even) H: the last tile row may be partial
  if (p.x_stride_t % 16 || p.x_stride_b % 16) return false;
  return true;
}

int launch_conv3x3_tile(const snnqp_block_params &p, const uint8_t *x, const int8_t *wq, const float *scale,
                        const float *bias, uint8_t *spikes, float *u_final, int32_t *acc_dump, int32_t *counts,
                        cudaStream_t st) {
  EncodeTiledFn encode = tmap_encoder();
  if (!encode) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return SNNQP_ERR_CUDA;
  }
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(wq) & 15))
    return invalid("tcgen05 conv: x and wq must be 16-byte aligned");

  const bool xbits = p.x_format == SNNQP_SPIKES_BITS;
  const int cbytes = xbits ? kC / 8 : kC;       // bytes per position of x
  // a size-1 dimension may carry any stride: give it a sane one
  const uint64_t img = (uint64_t)p.H * p.W * cbytes;
  const uint64_t st_t = p.T == 1 ? img : (uint64_t)p.x_stride_t;
  const uint64_t st_b = p.B == 1 ? img * p.T : (uint64_t)p.x_stride_b;
  const bool tb_swapped = st_t > st_b;          // keep the outer strides non-decreasing
  // tensor maps are cached per (pointer, geometry): encoding costs microseconds of host time per launch
  const TmapKey kx{x, {p.T, p.B, p.H, p.W, xbits ? 1 : 0, 21}, {(int64_t)st_t, (int64_t)st_b}};
  const CUtensorMap *tmx_p = tmap_cache_get(kx, [&](CUtensorMap *tm) {
    cuuint64_t dims[5] = {(cuuint64_t)cbytes, (cuuint64_t)p.W, (cuuint64_t)p.H,
                          (cuuint64_t)(tb_swapped ? p.B : p.T), (cuuint64_t)(tb_swapped ? p.T : p.B)};
    cuuint64_t strides[4] = {(cuuint64_t)cbytes, (cuuint64_t)p.W * cbytes, tb_swapped ? st_b : st_t, tb_swapped ? st_t : st_b};
    cuuint32_t box[5] = {(cuuint32_t)cbytes, (cuuint32_t)kBoxW, (cuuint32_t)kBoxH, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    return encode(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 5, const_cast<uint8_t *>(x), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, xbits ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  });
  if (!tmx_p) {
    set_error("cuTensorMapEncodeTiled(x) failed (T=%d B=%d H=%d W=%d strides %lld/%lld bits=%d)", p.T, p.B, p.H, p.W,
              (long long)p.x_stride_t, (long long)p.x_stride_b, (int)xbits);
    return SNNQP_ERR_CUDA;
  }
  const TmapKey kw{wq, {9, kC, kC, 0, 0, 1}, {0, 0}};
  const CUtensorMap *tmw_p = tmap_cache_get(kw, [&](CUtensorMap *tm) {
    cuuint64_t dims[2] = {(cuuint64_t)kC, (cuuint64_t)9 * kC};
    cuuint64_t strides[1] = {(cuuint64_t)kC};
    cuuint32_t box[2] = {(cuuint32_t)kC, (cuuint32_t)kC};
    cuuint32_t estr[2] = {1, 1};
    return encode(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<int8_t *>(wq), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  });
  if (!tmw_p) {
    set_error("cuTensorMapEncodeTiled(w) failed");
    return SNNQP_ERR_CUDA;
  }
  const CUtensorMap &tmx = *tmx_p, &tmw = *tmw_p;

  UmmaArgs a;
  a.T = p.T; a.B = p.B; a.H = p.H; a.W = p.W;
  a.tiles_x = p.W / kTileW;
  a.tiles_per_img = a.tiles_x * ((p.H + kTileH - 1) / kTileH);
  a.total_items = p.B * a.tiles_per_img;
  a.y_stride_t = p.y_stride_t; a.y_stride_b = p.y_stride_b;
  a.tau = p.tau; a.v_th = p.v_threshold; a.v_reset = p.v_reset;
  a.pool = p.pool;
  a.tb_swapped = tb_swapped ? 1 : 0;
  a.one = 1;
  a.y_bits = p.y_format == SNNQP_SPIKES_BITS ? 1 : 0;
  a.y_popcount = p.y_popcount;
  a.base_off_mode = 0;   // the hardware applies the 128B swizzle on absolute smem address bits (measured)
#ifdef SNNQP_C1_BISECT
  static const int dbg_env = getenv("SNNQP_UMMA_DEBUG") ? atoi(getenv("SNNQP_UMMA_DEBUG")) : 0;   // bisection switches (tools/)
  a.debug = dbg_env;
#else
  a.debug = 0;
#endif
  a.stage_tx_bytes = (uint32_t)(kBoxRows * cbytes);
  a.scale = scale; a.bias = bias;
  a.slab_nz = reinterpret_cast<const uint8_t *>(wq) + kWBytes;   // blob tail written by snnqp_pack_conv3x3
  a.spikes = spikes; a.u_final = u_final; a.acc_dump = acc_dump; a.counts = counts; a.wq = wq;

  const int grid = a.total_items < sm_count() ? a.total_items : sm_count();
  // FAST with u8 output stores unconditionally: a partial last tile row takes the generic epilogue there (same bits)
  const bool fast = p.tau == 2.0f && p.v_threshold == 1.0f && p.v_reset == 0.0f && p.pool && !u_final && !acc_dump &&
                    (a.y_bits || p.H % kTileH == 0);
  if (a.y_bits && !fast)
    return unsupported("tcgen05 conv: bit-packed output needs the production variant (standard LIF constants, pool = 1, "
                       "no u_final / acc_dump)");
#define SNNQP_LAUNCH_TILE(FA, CO, XB)                                                                          \
  do {                                                                                                         \
    constexpr int kSm = smem_bytes_for(SNNQP_T_TAPS, XB ? kStagesBits : 4, XB);                                                              \
    if (int rc = ensure_smem_attr<k_conv3x3_tile<FA, CO, XB>>(kSm)) return rc;                                 \
    k_conv3x3_tile<FA, CO, XB><<<grid, XB ? kThreadsX : kThreads, kSm, st>>>(tmx, tmw, a);                     \
  } while (0)
  if (a.y_popcount) {
    if (!(xbits && fast && a.y_bits && !counts))
      return unsupported("tcgen05 conv: y_popcount needs bit-packed input and output, the production variant, no spike_counts");
    constexpr int kSm = smem_bytes_for(SNNQP_T_TAPS, kStagesBits, true);
    if (int rc = ensure_smem_attr<k_conv3x3_tile<true, false, true, true>>(kSm)) return rc;
    k_conv3x3_tile<true, false, true, true><<<grid, kThreadsX, kSm, st>>>(tmx, tmw, a);
  } else if (xbits) {
    if (!fast) SNNQP_LAUNCH_TILE(false, false, true);
    else if (counts) SNNQP_LAUNCH_TILE(true, true, true);
    else SNNQP_LAUNCH_TILE(true, false, true);
  } else {
    if (!fast) SNNQP_LAUNCH_TILE(false, false, false);
    else if (counts) SNNQP_LAUNCH_TILE(true, true, false);
    else SNNQP_LAUNCH_TILE(true, false, false);
  }
#undef SNNQP_LAUNCH_TILE
  SNNQP_POST_LAUNCH("k_conv3x3_tile");
  return SNNQP_OK;
}

}  // namespace snnqp

extern "C" int snnqp_tile_skip_stats(int64_t *skipped, int64_t *total, int reset) {
  using namespace snnqp;
  if (int rc = require_device()) return rc;
  unsigned long long h[2] = {0, 0};
  SNNQP_CUDA(cudaMemcpyFromSymbol(h, g_tile_skip_t, sizeof(h)));
  if (skipped) *skipped = (int64_t)h[0];
  if (total) *total = (int64_t)h[1];
  if (reset) {
    const unsigned long long z[2] = {0, 0};
    SNNQP_CUDA(cudaMemcpyToSymbol(g_tile_skip_t, z, sizeof(z)));
  }
  return SNNQP_OK;
}
