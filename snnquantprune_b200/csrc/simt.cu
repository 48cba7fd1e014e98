// CUDA-core (dp4a) implementations of the fused spiking blocks, the TCJA
// attention, the vote and the eval metrics.  These are the bring-up /
// cross-check kernels (SNNQP_IMPL_SIMT) and the production path for the small
// layers (conv1's K=18 contraction, conv5/dense1 whose inputs are real-valued,
// dense2, TCJA); the heavy binary-input convolutions run on tcgen05
// (umma_conv.cu).  Each kernel keeps the T loop inside, so membrane potentials
// live in registers and never touch HBM between timesteps
// (reference SpikingBlock scan: spiking_learning.py:441-472).
#include <stdlib.h>

#include "common.cuh"

namespace snnqp {

// ---------------------------------------------------------------------------
// 3x3 conv, Cin % 4 == 0 (binary / count inputs through dp4a, or att-weighted
// real inputs through fp32 FMAs).  One thread owns the 2x2 quad of output
// neurons that one pooled output pixel covers, for one output channel.
// Weights live in shared memory as [tap][cin/4][cout] 32-bit words.
// MODE 0: LIF (+pool)   MODE 1: plain conv, fp32 out
// ---------------------------------------------------------------------------
template <bool ATT, int MODE>
__global__ void __launch_bounds__(512, 1)
k_conv3x3_simt(const snnqp_block_params p, const uint8_t *__restrict__ x,
               const float *__restrict__ att, const int8_t *__restrict__ wq,
               const float *__restrict__ scale, const float *__restrict__ bias,
               uint8_t *__restrict__ spikes, float *__restrict__ u_final,
               void *__restrict__ acc_dump, float *__restrict__ y_plain, int32_t *__restrict__ counts) {
  extern __shared__ uint32_t sw[];   // [9][C4][Cout]
  const int Cin = p.Cin, Cout = p.Cout, C4 = Cin / 4;
  const uint32_t *wq32 = reinterpret_cast<const uint32_t *>(wq);
  for (int d = threadIdx.x; d < 9 * Cout * C4; d += blockDim.x) {
    const int c4 = d % C4, o = (d / C4) % Cout, tap = d / (C4 * Cout);
    sw[(tap * C4 + c4) * Cout + o] = wq32[d];
  }
  __syncthreads();

  const int o = threadIdx.x % Cout;
  const int lane_q = threadIdx.x / Cout, nlane = blockDim.x / Cout;
  const int H = p.H, W = p.W, QH = H / 2, QW = W / 2;
  const int64_t total = (int64_t)p.B * QH * QW;
  const float sc = scale[o], bi = bias[o];
  const int Ho = p.pool ? QH : H, Wo = p.pool ? QW : W;

  // threads beyond nlane * Cout (Cout does not divide the block, e.g. 96) would redo the next block's quad 0
  // and double-count its spikes: they only helped staging the weights
  for (int64_t quad = lane_q < nlane ? (int64_t)blockIdx.x * nlane + lane_q : total; quad < total;
       quad += (int64_t)gridDim.x * nlane) {
    const int qw = (int)(quad % QW), qh = (int)((quad / QW) % QH), b = (int)(quad / ((int64_t)QW * QH));
    float u[4] = {0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < p.T; ++t) {
      const uint8_t *xb = x + (int64_t)t * p.x_stride_t + (int64_t)b * p.x_stride_b;
      const float *ab = ATT ? att + (int64_t)t * p.att_stride_t + (int64_t)b * p.att_stride_b : nullptr;
      int acc[4] = {0, 0, 0, 0};
      float accf[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int py = 0; py < 4; ++py) {
        const int ih = 2 * qh - 1 + py;
        if (ih < 0 || ih >= H) continue;
#pragma unroll
        for (int px = 0; px < 4; ++px) {
          const int iw = 2 * qw - 1 + px;
          if (iw < 0 || iw >= W) continue;
          const uint32_t *xp = reinterpret_cast<const uint32_t *>(xb + ((int64_t)ih * W + iw) * Cin);
          for (int c4 = 0; c4 < C4; ++c4) {
            const uint32_t xw = __ldg(xp + c4);
            if (!ATT && xw == 0u) continue;   // warp-uniform: same pixel for the whole warp
            float xs[4];
            if (ATT) {
              // with att a non-zero x byte is a spike (input = att), as in the tcgen05 byte-plane expanders
#pragma unroll
              for (int j = 0; j < 4; ++j) xs[j] = ((xw >> (8 * j)) & 0xffu) ? __ldg(ab + c4 * 4 + j) : 0.0f;
            }
#pragma unroll
            for (int dy = 0; dy < 2; ++dy) {
              const int kh = py - dy;
              if (kh < 0 || kh > 2) continue;
#pragma unroll
              for (int dx = 0; dx < 2; ++dx) {
                const int kw = px - dx;
                if (kw < 0 || kw > 2) continue;
                const uint32_t ww = sw[((kh * 3 + kw) * C4 + c4) * Cout + o];
                if (ATT) {
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float qf = (float)(int8_t)((ww >> (8 * j)) & 0xffu);
                    accf[dy * 2 + dx] = __fmaf_rn(xs[j], qf, accf[dy * 2 + dx]);
                  }
                } else {
                  acc[dy * 2 + dx] = dp4a_us(xw, (int)ww, acc[dy * 2 + dx]);
                }
              }
            }
          }
        }
      }
      // epilogue: folded dequant+BN affine, then LIF / plain store
      bool any = false;
      int nspk = 0;
#pragma unroll
      for (int pos = 0; pos < 4; ++pos) {
        const int oh = 2 * qh + (pos >> 1), ow = 2 * qw + (pos & 1);
        const float f = ATT ? accf[pos] : (float)acc[pos];
        const float v = __fmaf_rn(f, sc, bi);
        const int64_t full = ((((int64_t)t * p.B + b) * H + oh) * W + ow) * Cout + o;
        if (MODE == 1) {
          y_plain[full] = v;
          continue;
        }
        if (acc_dump) {
          if (ATT) reinterpret_cast<float *>(acc_dump)[full] = accf[pos];
          else reinterpret_cast<int32_t *>(acc_dump)[full] = acc[pos];
        }
        bool s;
        u[pos] = lif_step(u[pos], v, p.tau, p.v_threshold, p.v_reset, s);
        any |= s;
        nspk += s ? 1 : 0;
        if (!p.pool)
          spikes[(int64_t)t * p.y_stride_t + (int64_t)b * p.y_stride_b + ((int64_t)oh * Wo + ow) * Cout + o] = s ? 1 : 0;
      }
      if (MODE == 0 && p.pool)
        spikes[(int64_t)t * p.y_stride_t + (int64_t)b * p.y_stride_b + ((int64_t)qh * Wo + qw) * Cout + o] = any ? 1 : 0;
      if (MODE == 0 && counts && nspk) atomicAdd(counts + ((int64_t)b * p.T + t) * Cout + o, nspk);
    }
    if (MODE == 0 && u_final) {
#pragma unroll
      for (int pos = 0; pos < 4; ++pos) {
        const int oh = 2 * qh + (pos >> 1), ow = 2 * qw + (pos & 1);
        u_final[(((int64_t)b * H + oh) * W + ow) * Cout + o] = u[pos];
      }
    }
  }
}

// ---------------------------------------------------------------------------
// conv1: 3x3 conv with Cin == 2 (event counts), K = 18 padded to 32:
// wq [Cout][32], k = tap * 2 + ci.  Weights in registers, input through L1.
// ---------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256)
k_conv3x3_c2_simt(const snnqp_block_params p, const uint8_t *__restrict__ x,
                  const int8_t *__restrict__ wq, const float *__restrict__ scale,
                  const float *__restrict__ bias, uint8_t *__restrict__ spikes,
                  float *__restrict__ u_final, int32_t *__restrict__ acc_dump,
                  float *__restrict__ y_plain) {
  const int Cout = p.Cout;
  const int o = threadIdx.x % Cout;
  const int lane_q = threadIdx.x / Cout, nlane = blockDim.x / Cout;
  int wreg[18];
  {
    const int8_t *wr = wq + (int64_t)o * 32;
#pragma unroll
    for (int k = 0; k < 18; ++k) wreg[k] = wr[k];
  }
  const int H = p.H, W = p.W, QH = H / 2, QW = W / 2;
  const int64_t total = (int64_t)p.B * QH * QW;
  const float sc = scale[o], bi = bias[o];
  const int Ho = p.pool ? QH : H, Wo = p.pool ? QW : W;
  (void)Ho;
  // threads beyond nlane * Cout (Cout does not divide the block, e.g. 96) would redo the next block's quad 0
  // and double-count its spikes: they only helped staging the weights
  for (int64_t quad = lane_q < nlane ? (int64_t)blockIdx.x * nlane + lane_q : total; quad < total;
       quad += (int64_t)gridDim.x * nlane) {
    const int qw = (int)(quad % QW), qh = (int)((quad / QW) % QH), b = (int)(quad / ((int64_t)QW * QH));
    float u[4] = {0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < p.T; ++t) {
      const uint8_t *xb = x + (int64_t)t * p.x_stride_t + (int64_t)b * p.x_stride_b;
      int acc[4] = {0, 0, 0, 0};
#pragma unroll
      for (int py = 0; py < 4; ++py) {
        const int ih = 2 * qh - 1 + py;
        if (ih < 0 || ih >= H) continue;
#pragma unroll
        for (int px = 0; px < 4; ++px) {
          const int iw = 2 * qw - 1 + px;
          if (iw < 0 || iw >= W) continue;
          const uint16_t xv = __ldg(reinterpret_cast<const uint16_t *>(xb + ((int64_t)ih * W + iw) * 2));
          const int x0 = xv & 0xff, x1 = xv >> 8;
#pragma unroll
          for (int dy = 0; dy < 2; ++dy) {
            const int kh = py - dy;
            if (kh < 0 || kh > 2) continue;
#pragma unroll
            for (int dx = 0; dx < 2; ++dx) {
              const int kw = px - dx;
              if (kw < 0 || kw > 2) continue;
              const int tap = kh * 3 + kw;
              acc[dy * 2 + dx] += x0 * wreg[tap * 2] + x1 * wreg[tap * 2 + 1];
            }
          }
        }
      }
      bool any = false;
#pragma unroll
      for (int pos = 0; pos < 4; ++pos) {
        const int oh = 2 * qh + (pos >> 1), ow = 2 * qw + (pos & 1);
        const float v = __fmaf_rn((float)acc[pos], sc, bi);
        const int64_t full = ((((int64_t)t * p.B + b) * H + oh) * W + ow) * Cout + o;
        if (MODE == 1) {
          y_plain[full] = v;
          continue;
        }
        if (acc_dump) acc_dump[full] = acc[pos];
        bool s;
        u[pos] = lif_step(u[pos], v, p.tau, p.v_threshold, p.v_reset, s);
        any |= s;
        if (!p.pool)
          spikes[(int64_t)t * p.y_stride_t + (int64_t)b * p.y_stride_b + ((int64_t)oh * Wo + ow) * Cout + o] = s ? 1 : 0;
      }
      if (MODE == 0 && p.pool)
        spikes[(int64_t)t * p.y_stride_t + (int64_t)b * p.y_stride_b + ((int64_t)qh * Wo + qw) * Cout + o] = any ? 1 : 0;
    }
    if (MODE == 0 && u_final) {
#pragma unroll
      for (int pos = 0; pos < 4; ++pos) {
        const int oh = 2 * qh + (pos >> 1), ow = 2 * qw + (pos & 1);
        u_final[(((int64_t)b * H + oh) * W + ow) * Cout + o] = u[pos];
      }
    }
  }
}

// ---------------------------------------------------------------------------
// dense: x u8 [T,B,K], wq [N][k_pad]; one thread per output n, DB samples per
// block sharing the weight stream; x rows staged in shared memory.
// ---------------------------------------------------------------------------
constexpr int DENSE_DB = 4;

template <bool ATT>
__global__ void __launch_bounds__(128)
k_dense_simt(const snnqp_block_params p, int k_pad, const uint8_t *__restrict__ x,
             const float *__restrict__ att, const int8_t *__restrict__ wq,
             const float *__restrict__ scale, const float *__restrict__ bias,
             uint8_t *__restrict__ spikes, float *__restrict__ u_final,
             void *__restrict__ acc_dump) {
  extern __shared__ __align__(16) uint8_t sx[];   // [DB][k_pad] u8 (+ [DB][k_pad] fp32 when ATT)
  float *sxf = reinterpret_cast<float *>(sx + DENSE_DB * k_pad);
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int b0 = blockIdx.y * DENSE_DB;
  const int K = p.Cin, N = p.Cout;
  const bool act = n < N;
  const float sc = act ? scale[n] : 0.f, bi = act ? bias[n] : 0.f;
  const int8_t *wr = wq + (int64_t)(act ? n : 0) * k_pad;
  float u[DENSE_DB];
#pragma unroll
  for (int j = 0; j < DENSE_DB; ++j) u[j] = 0.f;

  for (int t = 0; t < p.T; ++t) {
    __syncthreads();
    for (int d = threadIdx.x; d < DENSE_DB * k_pad; d += blockDim.x) {
      const int j = d / k_pad, k = d % k_pad;
      const int b = b0 + j;
      uint8_t v = 0;
      if (b < p.B && k < K) v = x[(int64_t)t * p.x_stride_t + (int64_t)b * p.x_stride_b + k];
      sx[d] = v;
      if (ATT) {
        float a = 0.f;
        if (b < p.B && k < K)
          a = att[(int64_t)t * p.att_stride_t + (int64_t)b * p.att_stride_b + (k % p.att_mod)];
        sxf[d] = v ? a : 0.0f;            // with att a non-zero x byte is a spike (input = att)
      }
    }
    __syncthreads();
    if (!act) continue;
    int acc[DENSE_DB];
    float accf[DENSE_DB];
#pragma unroll
    for (int j = 0; j < DENSE_DB; ++j) { acc[j] = 0; accf[j] = 0.f; }
    for (int k16 = 0; k16 < k_pad / 16; ++k16) {
      const int4 wv = __ldg(reinterpret_cast<const int4 *>(wr) + k16);
      const int wws[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) {
        const int k4 = k16 * 4 + q4;
        if (ATT) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float qf = (float)(int8_t)((wws[q4] >> (8 * e)) & 0xff);
#pragma unroll
            for (int j = 0; j < DENSE_DB; ++j)
              accf[j] = __fmaf_rn(sxf[j * k_pad + k4 * 4 + e], qf, accf[j]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < DENSE_DB; ++j) {
            const uint32_t xw = reinterpret_cast<const uint32_t *>(sx + j * k_pad)[k4];
            acc[j] = dp4a_us(xw, wws[q4], acc[j]);
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < DENSE_DB; ++j) {
      const int b = b0 + j;
      if (b >= p.B) continue;
      const float f = ATT ? accf[j] : (float)acc[j];
      const float v = __fmaf_rn(f, sc, bi);
      const int64_t full = ((int64_t)t * p.B + b) * N + n;
      if (acc_dump) {
        if (ATT) reinterpret_cast<float *>(acc_dump)[full] = accf[j];
        else reinterpret_cast<int32_t *>(acc_dump)[full] = acc[j];
      }
      bool s;
      u[j] = lif_step(u[j], v, p.tau, p.v_threshold, p.v_reset, s);
      spikes[(int64_t)t * p.y_stride_t + (int64_t)b * p.y_stride_b + n] = s ? 1 : 0;
    }
  }
  if (u_final && act) {
#pragma unroll
    for (int j = 0; j < DENSE_DB; ++j) {
      const int b = b0 + j;
      if (b < p.B) u_final[(int64_t)b * N + n] = u[j];
    }
  }
}

// ---------------------------------------------------------------------------
// TCJA (reference examples/tcja/models.py:41-95)
// ---------------------------------------------------------------------------
// counts[b][t][c] = sum_{h,w} spikes[t,b,h,w,c]   (mean = counts / HW, exact)
__global__ void __launch_bounds__(256)
k_tcja_counts(const snnqp_block_params p, const uint8_t *__restrict__ s,
              int32_t *__restrict__ counts) {
  const int tb = blockIdx.x;
  const int t = tb % p.T, b = tb / p.T;
  const int C = p.Cin, HW = p.H * p.W;
  const int c4 = threadIdx.x % (C / 4), part = threadIdx.x / (C / 4), nparts = blockDim.x / (C / 4);
  const uint32_t *sp = reinterpret_cast<const uint32_t *>(s + (int64_t)t * p.x_stride_t + (int64_t)b * p.x_stride_b);
  uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  for (int px = part; px < HW; px += nparts) {
    const uint32_t w = __ldg(sp + (int64_t)px * (C / 4) + c4);
    a0 += w & 0xff; a1 += (w >> 8) & 0xff; a2 += (w >> 16) & 0xff; a3 += w >> 24;
  }
  __shared__ int32_t red[128 * 4];
  for (int i = threadIdx.x; i < C; i += blockDim.x) red[i] = 0;
  __syncthreads();
  atomicAdd(&red[c4 * 4 + 0], (int)a0); atomicAdd(&red[c4 * 4 + 1], (int)a1);
  atomicAdd(&red[c4 * 4 + 2], (int)a2); atomicAdd(&red[c4 * 4 + 3], (int)a3);
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x)
    counts[((int64_t)b * p.T + t) * C + i] = red[i];
}

// att[t,b,c] = sigmoid(c_out[t,b,c] * t_out[t,b,c])
//   t_out[t',b,c] = scale_t * sum_{j<4, t} cnt[t][c+j-1] * q_t[j][t][t']   (conv over the channel axis, features = T)
//   c_out[t,b,c'] = scale_c * sum_{j<4, c} cnt[t+j-1][c] * q_c[j][c][c']   (conv over the time axis, features = C)
// 'SAME' pads for k=4: low 1, high 2 (reference flax_qconv.py:131-142).
// One block per sample: the 4*C*C conv_c weights (64 KB) and the sample's counts are staged
// in shared memory once and reused for all T timesteps; thread = (channel, timestep parity).
__global__ void __launch_bounds__(256)
k_tcja_att(const snnqp_block_params p, const int32_t *__restrict__ counts,
           const int8_t *__restrict__ wq_t, const int8_t *__restrict__ wq_c,
           const float *__restrict__ scale_t, const float *__restrict__ scale_c,
           float *__restrict__ att) {
  extern __shared__ __align__(16) uint8_t tcja_smem[];
  const int b = blockIdx.x, T = p.T, C = p.Cin;
  int8_t *qc = reinterpret_cast<int8_t *>(tcja_smem);                       // [4][C][C]
  int32_t *cnt = reinterpret_cast<int32_t *>(tcja_smem + 4 * C * C);        // [T][C]
  int8_t *qt = reinterpret_cast<int8_t *>(cnt + T * C);                     // [4][T][T]
  for (int d = threadIdx.x; d < 4 * C * C / 16; d += blockDim.x)
    reinterpret_cast<int4 *>(qc)[d] = __ldg(reinterpret_cast<const int4 *>(wq_c) + d);
  for (int d = threadIdx.x; d < T * C; d += blockDim.x) cnt[d] = counts[(int64_t)b * T * C + d];
  for (int d = threadIdx.x; d < 4 * T * T; d += blockDim.x) qt[d] = wq_t[d];
  __syncthreads();
  const float st = *scale_t, scc = *scale_c;
  const int c = threadIdx.x % C, part = threadIdx.x / C, nparts = blockDim.x / C;
  for (int t = part; t < T; t += nparts) {
    int acc_c = 0, acc_t = 0;
    for (int j = 0; j < 4; ++j) {
      const int tt = t + j - 1;
      if (tt >= 0 && tt < T) {
        const int32_t *row = cnt + tt * C;
        const int8_t *wc = qc + j * C * C + c;
#pragma unroll 8
        for (int ci = 0; ci < C; ++ci) acc_c += row[ci] * (int)wc[ci * C];
      }
      const int cc = c + j - 1;
      if (cc >= 0 && cc < C)
        for (int ti = 0; ti < T; ++ti) acc_t += cnt[ti * C + cc] * (int)qt[(j * T + ti) * T + t];
    }
    const float to = __fmul_rn((float)acc_t, st);
    const float co = __fmul_rn((float)acc_c, scc);
    const float pr = __fmul_rn(co, to);
    const float a = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-pr)));
    att[(int64_t)t * p.att_stride_t + (int64_t)b * p.att_stride_b + c] = a;
  }
}

// Same result (integer accumulators are exact in any order), dp4a form for C == 128, T <= 32: the conv_c weights
// are re-laid in shared memory as [j][c/4][c'] words (4 input channels per word), the counts as two byte planes
// (low byte, high byte: counts <= H*W <= 65535), so that 4 multiply-adds cost one dp4a per plane instead of
// two shared-memory loads and an IMAD each, and a weight word is loaded once for all of a thread's timesteps.
// HIGH == false when H*W <= 255 (the high plane is all zero).
template <bool HIGH>
__global__ void __launch_bounds__(256)
k_tcja_att_dp4a(const snnqp_block_params p, const int32_t *__restrict__ counts,
                const int8_t *__restrict__ wq_t, const int8_t *__restrict__ wq_c,
                const float *__restrict__ scale_t, const float *__restrict__ scale_c,
                float *__restrict__ att) {
  constexpr int C = 128, C4 = C / 4, NT = 16;                               // NT: timesteps per thread (T <= 32)
  extern __shared__ __align__(16) uint8_t tcja_smem[];
  const int b = blockIdx.x, T = p.T;
  uint32_t *qc4 = reinterpret_cast<uint32_t *>(tcja_smem);                  // [4][C4][C] words
  int32_t *cnt = reinterpret_cast<int32_t *>(qc4 + 4 * C4 * C);             // [T][C]
  uint32_t *lo4 = reinterpret_cast<uint32_t *>(cnt + T * C);                // [T + 3][C4], rows -1 and T, T+1 zero
  uint32_t *hi4 = lo4 + (T + 3) * C4;
  int8_t *qt = reinterpret_cast<int8_t *>(hi4 + (T + 3) * C4);              // [4][T][T]
  // weights: global [j][ci][c'] bytes -> words {ci, ci+1, ci+2, ci+3} at [j][ci/4][c']: four 16-byte row pieces
  // (rows ci .. ci+3, 16 consecutive c') are transposed in registers into 16 words
  for (int d = threadIdx.x; d < 4 * C4 * (C / 16); d += blockDim.x) {
    const int c16 = d % (C / 16), ci4 = (d / (C / 16)) % C4, j = d / ((C / 16) * C4);
    const int4 *src = reinterpret_cast<const int4 *>(wq_c + ((size_t)j * C + 4 * ci4) * C + 16 * c16);
    const int4 r0 = __ldg(src), r1 = __ldg(src + C / 16), r2 = __ldg(src + 2 * (C / 16)), r3 = __ldg(src + 3 * (C / 16));
    uint4 *dst = reinterpret_cast<uint4 *>(qc4 + (j * C4 + ci4) * C + 16 * c16);
    auto tr = [](uint32_t a, uint32_t b, uint32_t c, uint32_t e) {           // 4 x 4 byte transpose
      const uint32_t t0 = __byte_perm(a, b, 0x5140), t1 = __byte_perm(c, e, 0x5140);   // (a0 b0 a1 b1), (c0 e0 c1 e1)
      const uint32_t t2 = __byte_perm(a, b, 0x7362), t3 = __byte_perm(c, e, 0x7362);   // (a2 b2 a3 b3), (c2 e2 c3 e3)
      return make_uint4(__byte_perm(t0, t1, 0x5410), __byte_perm(t0, t1, 0x7632), __byte_perm(t2, t3, 0x5410),
                        __byte_perm(t2, t3, 0x7632));
    };
    dst[0] = tr((uint32_t)r0.x, (uint32_t)r1.x, (uint32_t)r2.x, (uint32_t)r3.x);
    dst[1] = tr((uint32_t)r0.y, (uint32_t)r1.y, (uint32_t)r2.y, (uint32_t)r3.y);
    dst[2] = tr((uint32_t)r0.z, (uint32_t)r1.z, (uint32_t)r2.z, (uint32_t)r3.z);
    dst[3] = tr((uint32_t)r0.w, (uint32_t)r1.w, (uint32_t)r2.w, (uint32_t)r3.w);
  }
  for (int d = threadIdx.x; d < T * C; d += blockDim.x) cnt[d] = counts[(int64_t)b * T * C + d];
  for (int d = threadIdx.x; d < (T + 3) * C4; d += blockDim.x) {
    const int tt = d / C4 - 1, c4 = d % C4;                                  // padded row index -> timestep
    uint32_t l = 0, h = 0;
    if (tt >= 0 && tt < T) {
      const int4 v = *reinterpret_cast<const int4 *>(counts + ((int64_t)b * T + tt) * C + 4 * c4);
      l = (v.x & 255) | ((v.y & 255) << 8) | ((v.z & 255) << 16) | ((uint32_t)(v.w & 255) << 24);
      h = ((v.x >> 8) & 255) | (((v.y >> 8) & 255) << 8) | (((v.z >> 8) & 255) << 16) | ((uint32_t)((v.w >> 8) & 255) << 24);
    }
    lo4[d] = l;
    hi4[d] = h;
  }
  for (int d = threadIdx.x; d < 4 * T * T; d += blockDim.x) qt[d] = wq_t[d];
  __syncthreads();
  const float st = *scale_t, scc = *scale_c;
  const int c = threadIdx.x % C, part = threadIdx.x / C;                     // blockDim.x == 2 * C
  int accl[NT], acch[NT];
#pragma unroll
  for (int i = 0; i < NT; ++i) { accl[i] = 0; acch[i] = 0; }
  for (int ci16 = 0; ci16 < C4 / 4; ++ci16) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) w[k] = (int)qc4[(j * C4 + 4 * ci16 + k) * C + c];
#pragma unroll
      for (int i = 0; i < NT; ++i) {
        const int t = part + 2 * i;
        if (t < T) {
          // padded row (t + j - 1) + 1 = t + j; 'SAME' pads (low 1, high 2) read the zero rows
          const uint4 l = *reinterpret_cast<const uint4 *>(lo4 + (t + j) * C4 + 4 * ci16);
          accl[i] = dp4a_us(l.x, w[0], accl[i]); accl[i] = dp4a_us(l.y, w[1], accl[i]);
          accl[i] = dp4a_us(l.z, w[2], accl[i]); accl[i] = dp4a_us(l.w, w[3], accl[i]);
          if constexpr (HIGH) {
            const uint4 h = *reinterpret_cast<const uint4 *>(hi4 + (t + j) * C4 + 4 * ci16);
            acch[i] = dp4a_us(h.x, w[0], acch[i]); acch[i] = dp4a_us(h.y, w[1], acch[i]);
            acch[i] = dp4a_us(h.z, w[2], acch[i]); acch[i] = dp4a_us(h.w, w[3], acch[i]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NT; ++i) {
    const int t = part + 2 * i;
    if (t >= T) continue;
    const int acc_c = accl[i] + (HIGH ? acch[i] * 256 : 0);
    int acc_t = 0;
    for (int j = 0; j < 4; ++j) {
      const int cc = c + j - 1;
      if (cc >= 0 && cc < C)
        for (int ti = 0; ti < T; ++ti) acc_t += cnt[ti * C + cc] * (int)qt[(j * T + ti) * T + t];
    }
    const float to = __fmul_rn((float)acc_t, st);
    const float co = __fmul_rn((float)acc_c, scc);
    const float pr = __fmul_rn(co, to);
    const float a = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-pr)));
    att[(int64_t)t * p.att_stride_t + (int64_t)b * p.att_stride_b + c] = a;
  }
}

// Tensor-core form of the same arithmetic for C == 128, T <= 32 (legacy mma.sync m16n8k32 u8 x s8 -> s32; the
// GEMM is tiny -- [T x 512] x [512 x 128] per sample -- and latency-bound, not worth a tcgen05 pipeline):
//   c_out accumulators D[t][c'] = sum_{j, ci} cnt[t + j - 1][ci] * q_c[j][ci][c'] with the counts as u8 byte planes
//   (low, high; the high plane is skipped when the sample has no count >= 256), one block per sample,
//   warp w owns output channels 16w .. 16w+15 and both 16-row time tiles.
//   t_out (80 multiply-adds per output) stays scalar and goes through shared memory.
// Integer accumulators: bit-identical to k_tcja_att / k_tcja_att_dp4a.  Shared-memory row strides are padded
// (36 / 136 words) so that the fragment loads of a warp hit 32 different banks.
__global__ void __launch_bounds__(256)
k_tcja_att_mma(const snnqp_block_params p, const int32_t *__restrict__ counts,
               const int8_t *__restrict__ wq_t, const int8_t *__restrict__ wq_c,
               const float *__restrict__ scale_t, const float *__restrict__ scale_c,
               float *__restrict__ att) {
  constexpr int C = 128, C4 = C / 4, SA = C4 + 4, SB = C + 8, ROWS = 36;    // ROWS: padded time rows (-1 .. 34)
  extern __shared__ __align__(16) uint8_t tcja_smem[];
  const int b = blockIdx.x, T = p.T;
  uint32_t *qc4 = reinterpret_cast<uint32_t *>(tcja_smem);                  // [4][C4][SB] words
  uint32_t *lo4 = qc4 + 4 * C4 * SB;                                        // [ROWS][SA]
  uint32_t *hi4 = lo4 + ROWS * SA;                                          // [ROWS][SA]
  int32_t *cnt = reinterpret_cast<int32_t *>(hi4 + ROWS * SA);              // [T][C]
  int32_t *tout = cnt + T * C;                                              // [T][C] t_out accumulators
  int8_t *qt = reinterpret_cast<int8_t *>(tout + T * C);                    // [4][T][T]
  for (int d = threadIdx.x; d < 4 * C4 * (C / 16); d += blockDim.x) {
    const int c16 = d % (C / 16), ci4 = (d / (C / 16)) % C4, j = d / ((C / 16) * C4);
    const int4 *src = reinterpret_cast<const int4 *>(wq_c + ((size_t)j * C + 4 * ci4) * C + 16 * c16);
    const int4 r0 = __ldg(src), r1 = __ldg(src + C / 16), r2 = __ldg(src + 2 * (C / 16)), r3 = __ldg(src + 3 * (C / 16));
    uint4 *dst = reinterpret_cast<uint4 *>(qc4 + (j * C4 + ci4) * SB + 16 * c16);
    auto tr = [](uint32_t a, uint32_t b2, uint32_t c, uint32_t e) {          // 4 x 4 byte transpose
      const uint32_t t0 = __byte_perm(a, b2, 0x5140), t1 = __byte_perm(c, e, 0x5140);
      const uint32_t t2 = __byte_perm(a, b2, 0x7362), t3 = __byte_perm(c, e, 0x7362);
      return make_uint4(__byte_perm(t0, t1, 0x5410), __byte_perm(t0, t1, 0x7632), __byte_perm(t2, t3, 0x5410),
                        __byte_perm(t2, t3, 0x7632));
    };
    dst[0] = tr((uint32_t)r0.x, (uint32_t)r1.x, (uint32_t)r2.x, (uint32_t)r3.x);
    dst[1] = tr((uint32_t)r0.y, (uint32_t)r1.y, (uint32_t)r2.y, (uint32_t)r3.y);
    dst[2] = tr((uint32_t)r0.z, (uint32_t)r1.z, (uint32_t)r2.z, (uint32_t)r3.z);
    dst[3] = tr((uint32_t)r0.w, (uint32_t)r1.w, (uint32_t)r2.w, (uint32_t)r3.w);
  }
  for (int d = threadIdx.x; d < T * C; d += blockDim.x) cnt[d] = counts[(int64_t)b * T * C + d];
  int any_hi = 0;
  for (int d = threadIdx.x; d < ROWS * C4; d += blockDim.x) {
    const int tt = d / C4 - 1, c4 = d % C4;                                  // padded row index -> timestep
    uint32_t l = 0, h = 0;
    if (tt >= 0 && tt < T) {
      const int4 v = *reinterpret_cast<const int4 *>(counts + ((int64_t)b * T + tt) * C + 4 * c4);
      l = (v.x & 255) | ((v.y & 255) << 8) | ((v.z & 255) << 16) | ((uint32_t)(v.w & 255) << 24);
      h = ((v.x >> 8) & 255) | (((v.y >> 8) & 255) << 8) | (((v.z >> 8) & 255) << 16) | ((uint32_t)((v.w >> 8) & 255) << 24);
    }
    lo4[(tt + 1) * SA + c4] = l;
    hi4[(tt + 1) * SA + c4] = h;
    any_hi |= (h != 0);
  }
  for (int d = threadIdx.x; d < 4 * T * T; d += blockDim.x) qt[d] = wq_t[d];
  any_hi = __syncthreads_or(any_hi);
  // ---- t_out[t'][c] = sum_{j, t} cnt[t][c + j - 1] * q_t[j][t][t'] (scalar, 4T multiply-adds each)
  for (int o = threadIdx.x; o < T * C; o += blockDim.x) {
    const int c = o % C, t = o / C;
    int acc_t = 0;
    for (int j = 0; j < 4; ++j) {
      const int cc = c + j - 1;
      if (cc >= 0 && cc < C)
        for (int ti = 0; ti < T; ++ti) acc_t += cnt[ti * C + cc] * (int)qt[(j * T + ti) * T + t];
    }
    tout[o] = acc_t;
  }
  // ---- c_out on the tensor cores
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  int acc[2][2][4], acch[2][2][4];                                           // [m tile][n tile][fragment]
#pragma unroll
  for (int m = 0; m < 2; ++m)
#pragma unroll
    for (int n = 0; n < 2; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) { acc[m][n][e] = 0; acch[m][n][e] = 0; }
  auto mma = [](int (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  };
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t bf[2][2];
#pragma unroll
      for (int n = 0; n < 2; ++n) {
        const int col = 16 * warp + 8 * n + g;
        bf[n][0] = qc4[(j * C4 + ks * 8 + q) * SB + col];
        bf[n][1] = qc4[(j * C4 + ks * 8 + q + 4) * SB + col];
      }
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        // padded row of timestep t + j - 1 is t + j; rows beyond T + 1 are zero (ROWS = 36 >= 31 + 3 + 1)
        const uint32_t *r0 = lo4 + (16 * m + g + j) * SA + ks * 8 + q, *r1 = r0 + 8 * SA;
        const uint32_t a[4] = {r0[0], r1[0], r0[4], r1[4]};
#pragma unroll
        for (int n = 0; n < 2; ++n) mma(acc[m][n], a, bf[n][0], bf[n][1]);
        if (any_hi) {
          const uint32_t *h0 = hi4 + (16 * m + g + j) * SA + ks * 8 + q, *h1 = h0 + 8 * SA;
          const uint32_t ah[4] = {h0[0], h1[0], h0[4], h1[4]};
#pragma unroll
          for (int n = 0; n < 2; ++n) mma(acch[m][n], ah, bf[n][0], bf[n][1]);
        }
      }
    }
  }
  __syncthreads();                                                           // tout complete
  const float st = *scale_t, scc = *scale_c;
#pragma unroll
  for (int m = 0; m < 2; ++m)
#pragma unroll
    for (int n = 0; n < 2; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int t = 16 * m + g + 8 * (e >> 1), c = 16 * warp + 8 * n + 2 * q + (e & 1);
        if (t >= T) continue;
        const int acc_c = acc[m][n][e] + acch[m][n][e] * 256;
        const float to = __fmul_rn((float)tout[t * C + c], st);
        const float co = __fmul_rn((float)acc_c, scc);
        const float pr = __fmul_rn(co, to);
        const float a = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-pr)));
        att[(int64_t)t * p.att_stride_t + (int64_t)b * p.att_stride_b + c] = a;
      }
}

// 2x2 max-pool on uint8, 4 channels per thread (HBM-bound)
__global__ void k_maxpool2(const snnqp_block_params p, const uint8_t *__restrict__ x,
                           uint8_t *__restrict__ y) {
  const int C4 = p.Cin / 4, Ho = p.H / 2, Wo = p.W / 2;
  const int64_t n = (int64_t)p.T * p.B * Ho * Wo * C4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % C4);
    int64_t r = i / C4;
    const int wo = (int)(r % Wo); r /= Wo;
    const int ho = (int)(r % Ho); r /= Ho;
    const int b = (int)(r % p.B);
    const int t = (int)(r / p.B);
    const uint32_t *xp = reinterpret_cast<const uint32_t *>(x + (int64_t)t * p.x_stride_t + (int64_t)b * p.x_stride_b);
    const int64_t base = ((int64_t)(2 * ho) * p.W + 2 * wo) * C4 + c4;
    const uint32_t a = __ldg(xp + base), b2 = __ldg(xp + base + C4);
    const uint32_t c = __ldg(xp + base + (int64_t)p.W * C4), d = __ldg(xp + base + (int64_t)p.W * C4 + C4);
    const uint32_t m = __vmaxu4(__vmaxu4(a, b2), __vmaxu4(c, d));
    reinterpret_cast<uint32_t *>(y + (int64_t)t * p.y_stride_t + (int64_t)b * p.y_stride_b)[((int64_t)ho * Wo + wo) * C4 + c4] = m;
  }
}

// vote: logits[b][g] = (sum_j (cnt[b][g*group+j] / T)) / group, sequential fp32
__global__ void k_vote(const uint8_t *__restrict__ s, int T, int B, int N, int group,
                       int64_t stride_t, int64_t stride_b, float *__restrict__ logits) {
  const int G = N / group;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * G) return;
  const int b = idx / G, g = idx % G;
  float acc = 0.f;
  for (int j = 0; j < group; ++j) {
    int cnt = 0;
    for (int t = 0; t < T; ++t) cnt += s[(int64_t)t * stride_t + (int64_t)b * stride_b + g * group + j];
    acc = __fadd_rn(acc, __fdiv_rn((float)cnt, (float)T));
  }
  logits[idx] = __fdiv_rn(acc, (float)group);
}

__global__ void k_eval_metrics(const float *__restrict__ logits, const int32_t *__restrict__ labels,
                               int B, int classes, float *__restrict__ out2) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  float hit = 0.f, se = 0.f;
  if (b < B) {
    int best = 0;
    float bv = logits[(int64_t)b * classes];
    for (int k = 0; k < classes; ++k) {
      const float v = logits[(int64_t)b * classes + k];
      if (v > bv) { bv = v; best = k; }           // first maximum, like argmax
      const float d = v - (k == labels[b] ? 1.0f : 0.0f);
      se += d * d;
    }
    hit = (best == labels[b]) ? 1.f : 0.f;
  }
  for (int off = 16; off > 0; off >>= 1) {
    hit += __shfl_xor_sync(0xffffffffu, hit, off);
    se += __shfl_xor_sync(0xffffffffu, se, off);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(out2, hit);
    atomicAdd(out2 + 1, se);
  }
}

// ---------------------------------------------------------------------------
// host-side launchers (called from api.cu)
// ---------------------------------------------------------------------------
int launch_conv3x3_simt(const snnqp_block_params &p, const uint8_t *x, const float *att,
                        const int8_t *wq, const float *scale, const float *bias,
                        uint8_t *spikes, float *u_final, void *acc_dump, float *y_plain,
                        int32_t *counts, cudaStream_t st) {
  const int64_t quads = (int64_t)p.B * (p.H / 2) * (p.W / 2);
  if (p.Cin == 2) {
    const int block = 256;
    const int nlane = block / p.Cout;
    int64_t g = (quads + nlane - 1) / nlane;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (g > cap) g = cap;
    if (y_plain)
      k_conv3x3_c2_simt<1><<<(int)g, block, 0, st>>>(p, x, wq, scale, bias, spikes, u_final, (int32_t *)acc_dump, y_plain);
    else
      k_conv3x3_c2_simt<0><<<(int)g, block, 0, st>>>(p, x, wq, scale, bias, spikes, u_final, (int32_t *)acc_dump, y_plain);
    SNNQP_POST_LAUNCH("k_conv3x3_c2_simt");
    return SNNQP_OK;
  }
  const int block = 512;
  const int nlane = block / p.Cout;
  const size_t smem = (size_t)9 * p.Cin * p.Cout;
  int64_t g = (quads + nlane - 1) / nlane;
  if (g > sm_count()) g = sm_count();
#define SNNQP_LAUNCH_CONV(ATTV, MODEV)                                                        \
  do {                                                                                        \
    SNNQP_CUDA(cudaFuncSetAttribute(k_conv3x3_simt<ATTV, MODEV>,                              \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    k_conv3x3_simt<ATTV, MODEV><<<(int)g, block, smem, st>>>(p, x, att, wq, scale, bias,      \
                                                            spikes, u_final, acc_dump, y_plain, counts); \
  } while (0)
  if (y_plain) {
    if (att) SNNQP_LAUNCH_CONV(true, 1); else SNNQP_LAUNCH_CONV(false, 1);
  } else {
    if (att) SNNQP_LAUNCH_CONV(true, 0); else SNNQP_LAUNCH_CONV(false, 0);
  }
#undef SNNQP_LAUNCH_CONV
  SNNQP_POST_LAUNCH("k_conv3x3_simt");
  return SNNQP_OK;
}

int launch_dense_simt(const snnqp_block_params &p, int k_pad, const uint8_t *x, const float *att,
                      const int8_t *wq, const float *scale, const float *bias, uint8_t *spikes,
                      float *u_final, void *acc_dump, cudaStream_t st) {
  dim3 grid((p.Cout + 127) / 128, (p.B + DENSE_DB - 1) / DENSE_DB);
  if (att) {
    const size_t smem = (size_t)DENSE_DB * k_pad * 5;
    SNNQP_CUDA(cudaFuncSetAttribute(k_dense_simt<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_dense_simt<true><<<grid, 128, smem, st>>>(p, k_pad, x, att, wq, scale, bias, spikes, u_final, acc_dump);
  } else {
    const size_t smem = (size_t)DENSE_DB * k_pad;
    k_dense_simt<false><<<grid, 128, smem, st>>>(p, k_pad, x, att, wq, scale, bias, spikes, u_final, acc_dump);
  }
  SNNQP_POST_LAUNCH("k_dense_simt");
  return SNNQP_OK;
}

int launch_tcja(const snnqp_block_params &p, const uint8_t *spikes, const int8_t *wq_t,
                const int8_t *wq_c, const float *scale_t, const float *scale_c, int32_t *counts,
                float *att, cudaStream_t st) {
  if (spikes) {   // else: counts were accumulated by the producing conv block (spike_counts output)
    k_tcja_counts<<<p.T * p.B, 256, 0, st>>>(p, spikes, counts);
    SNNQP_POST_LAUNCH("k_tcja_counts");
  }
  static const int tcja_impl = getenv("SNNQP_TCJA_IMPL") ? atoi(getenv("SNNQP_TCJA_IMPL")) : 2;   // 0 scalar, 1 dp4a, 2 mma.sync
  const bool fast_ok = p.Cin == 128 && p.T <= 32 && (int64_t)p.H * p.W <= 65535 && !(reinterpret_cast<uintptr_t>(counts) & 15) &&
                       !(reinterpret_cast<uintptr_t>(wq_c) & 15);
  if (fast_ok && tcja_impl == 2) {
    const size_t smem_m = (size_t)4 * 32 * 136 * 4 + (size_t)2 * 36 * 36 * 4 + (size_t)2 * p.T * 128 * sizeof(int32_t) +
                          (size_t)4 * p.T * p.T + 16;
    SNNQP_CUDA(cudaFuncSetAttribute(k_tcja_att_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m));
    k_tcja_att_mma<<<p.B, 256, smem_m, st>>>(p, counts, wq_t, wq_c, scale_t, scale_c, att);
    SNNQP_POST_LAUNCH("k_tcja_att_mma");
    return SNNQP_OK;
  }
  if (fast_ok && tcja_impl == 1) {
    const size_t smem4 = (size_t)4 * 128 * 128 + (size_t)p.T * 128 * sizeof(int32_t) + (size_t)2 * (p.T + 3) * 32 * 4 +
                         (size_t)4 * p.T * p.T + 16;
    if ((int64_t)p.H * p.W <= 255) {
      SNNQP_CUDA(cudaFuncSetAttribute(k_tcja_att_dp4a<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
      k_tcja_att_dp4a<false><<<p.B, 256, smem4, st>>>(p, counts, wq_t, wq_c, scale_t, scale_c, att);
    } else {
      SNNQP_CUDA(cudaFuncSetAttribute(k_tcja_att_dp4a<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
      k_tcja_att_dp4a<true><<<p.B, 256, smem4, st>>>(p, counts, wq_t, wq_c, scale_t, scale_c, att);
    }
    SNNQP_POST_LAUNCH("k_tcja_att_dp4a");
    return SNNQP_OK;
  }
  const size_t smem = (size_t)4 * p.Cin * p.Cin + (size_t)p.T * p.Cin * sizeof(int32_t) + (size_t)4 * p.T * p.T + 16;
  SNNQP_CUDA(cudaFuncSetAttribute(k_tcja_att, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_tcja_att<<<p.B, 256, smem, st>>>(p, counts, wq_t, wq_c, scale_t, scale_c, att);
  SNNQP_POST_LAUNCH("k_tcja_att");
  return SNNQP_OK;
}

int launch_maxpool2(const snnqp_block_params &p, const uint8_t *x, uint8_t *y, cudaStream_t st) {
  const int64_t n = (int64_t)p.T * p.B * (p.H / 2) * (p.W / 2) * (p.Cin / 4);
  int64_t g = (n + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (g > cap) g = cap;
  k_maxpool2<<<(int)g, 256, 0, st>>>(p, x, y);
  SNNQP_POST_LAUNCH("k_maxpool2");
  return SNNQP_OK;
}

int launch_vote(const uint8_t *s, int T, int B, int N, int group, int64_t stride_t,
                int64_t stride_b, float *logits, cudaStream_t st) {
  const int n = B * (N / group);
  k_vote<<<(n + 127) / 128, 128, 0, st>>>(s, T, B, N, group, stride_t, stride_b, logits);
  SNNQP_POST_LAUNCH("k_vote");
  return SNNQP_OK;
}

int launch_eval_metrics(const float *logits, const int32_t *labels, int B, int classes,
                        float *out2, cudaStream_t st) {
  k_eval_metrics<<<(B + 127) / 128, 128, 0, st>>>(logits, labels, B, classes, out2);
  SNNQP_POST_LAUNCH("k_eval_metrics");
  return SNNQP_OK;
}

}  // namespace snnqp
