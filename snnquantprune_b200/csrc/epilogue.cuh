// Shared epilogue arithmetic of the fused spiking kernels: folded dequant + BN
// affine, then the multi_step_LIF update (reference spiking_learning.py:404-416).
#pragma once

#include "common.cuh"

namespace snnqp {

// STD == true: tau = 2, v_threshold = 1, v_reset = 0 (every TCJA config,
// examples/tcja/configs/prune_quant_joint.py:27).  Then
//   u + ((x - (u - 0)) / 2)  ==  fma(x - u, 0.5, u)
// bit for bit: (x - u) is rounded once, halving is exact (no subnormals within
// T steps), and the final add is rounded once in both forms;
//   (u - 1 >= 0)  ==  (u >= 1)   since an fp32 difference is zero only for equal operands.
// Both forms must keep two properties of their ordered IEEE compare and NaN-propagating arithmetic: a NaN membrane
// never spikes and stays NaN.  k_conv3x3_tile's production epilogue relies on it to silence the rows of a partial tile
// below the image (tests/test_gpu_persistent_schedules.py fires such rows on the bias alone).
template <bool STD>
struct LifParams {
  float tau, v_th, v_reset;
  __device__ __forceinline__ bool step(float &u, float v) const {
    if constexpr (STD) {
      const float un = __fmaf_rn(__fsub_rn(v, u), 0.5f, u);
      const bool sp = un >= 1.0f;
      u = sp ? 0.0f : un;
      return sp;
    } else {
      bool sp;
      u = lif_step(u, v, tau, v_th, v_reset, sp);
      return sp;
    }
  }
};

__device__ __forceinline__ bool lif_is_std(float tau, float v_th, float v_reset) {
  return tau == 2.0f && v_th == 1.0f && v_reset == 0.0f;
}

// ---------------------------------------------------------------------------
// Packed (2 x fp32) fast path.  ncu on the scalar epilogue showed the half-rate
// ALU pipe (I2FP / FSETP / FSEL / predicate logic) ~80 % busy with the FMA pipe
// at ~30 %, so this version keeps almost everything on the FMA pipe and uses
// Blackwell's FADD2 / FFMA2 (PTX add/sub/fma .f32x2):
//   int32 -> fp32 : as_float(acc * one + 0x4B400000) - 1.5*2^23  (IMAD + FADD2; exact for |acc| < 2^22)
//   v  = fma(f, scale, bias)                                      (FFMA2)
//   un = fma(v - u, 0.5, u)                                       (FADD2 + FFMA2)
//   s  = un >= 1 ? 1.0f : 0.0f                                    (FSET.BF, the one ALU op per neuron)
//   u  = fma(-s, un, un)     (= 0 when s = 1, un when s = 0)      (FFMA2)
// Every result is bit-identical to the scalar form above.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint64_t pack2(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float &a, float &b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// 1.0f if x >= 1 else 0.0f: one FSET.BF (the only ALU-pipe instruction of a neuron update)
__device__ __forceinline__ float fset_ge1(float x) {
  float d;
  asm("set.ge.f32.f32 %0, %1, 0f3F800000;" : "=f"(d) : "f"(x));
  return d;
}

struct Lif2Consts {
  uint64_t sc2, bi2, half2, nmagic2;
  int one;      // runtime 1: keeps the magic-number add an IMAD (FMA pipe) instead of an ALU-pipe IADD3
  __device__ __forceinline__ Lif2Consts(float sc, float bi, int one_)
      : sc2(pack2(sc, sc)), bi2(pack2(bi, bi)), half2(pack2(0.5f, 0.5f)),
        nmagic2(pack2(-12582912.0f, -12582912.0f)), one(one_) {}
};

// One standard-LIF step for two neurons.  u2: packed membranes (in/out);
// acc0/acc1: raw int32 accumulators.  Returns the packed spikes as 1.0f / 0.0f.
__device__ __forceinline__ uint64_t lif2_std(uint64_t &u2, uint32_t acc0, uint32_t acc1, const Lif2Consts &k) {
  uint32_t m0, m1;
  asm("mad.lo.s32 %0, %1, %2, 0x4B400000;" : "=r"(m0) : "r"(acc0), "r"(k.one));
  asm("mad.lo.s32 %0, %1, %2, 0x4B400000;" : "=r"(m1) : "r"(acc1), "r"(k.one));
  const uint64_t f = add2(pack2(__uint_as_float(m0), __uint_as_float(m1)), k.nmagic2);
  const uint64_t v = fma2(f, k.sc2, k.bi2);
  const uint64_t un = fma2(sub2(v, u2), k.half2, u2);
  float a, b;
  unpack2(un, a, b);
  const float s0 = a >= 1.0f ? 1.0f : 0.0f, s1 = b >= 1.0f ? 1.0f : 0.0f;
  u2 = fma2(pack2(-s0, -s1), un, un);
  return pack2(s0, s1);
}

// 1 if any of the four pooled spikes (two packed pairs) fired
__device__ __forceinline__ uint8_t pool2x2(uint64_t s_top, uint64_t s_bot) {
  float a, b;
  unpack2(add2(s_top, s_bot), a, b);
  return (a + b) != 0.0f ? 1 : 0;
}

}  // namespace snnqp
