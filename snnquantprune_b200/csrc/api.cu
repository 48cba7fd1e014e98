// C-ABI entry points of the fused spiking blocks: argument validation and
// dispatch between the tcgen05 kernels (umma_conv1.cu / umma_conv1_tc.cu for
// conv1, umma_conv_t.cu for the 3x3 blocks, umma_att.cu for the attention-
// weighted blocks and dense layers) and the dp4a kernels (simt.cu).  See
// include/snnqp.h for the contract.
#include "common.cuh"

namespace snnqp {
int launch_conv3x3_simt(const snnqp_block_params &p, const uint8_t *x, const float *att,
                        const int8_t *wq, const float *scale, const float *bias,
                        uint8_t *spikes, float *u_final, void *acc_dump, float *y_plain,
                        int32_t *counts, cudaStream_t st);
int launch_dense_simt(const snnqp_block_params &p, int k_pad, const uint8_t *x, const float *att,
                      const int8_t *wq, const float *scale, const float *bias, uint8_t *spikes,
                      float *u_final, void *acc_dump, cudaStream_t st);
int launch_tcja(const snnqp_block_params &p, const uint8_t *spikes, const int8_t *wq_t,
                const int8_t *wq_c, const float *scale_t, const float *scale_c, int32_t *counts,
                float *att, cudaStream_t st);
int launch_maxpool2(const snnqp_block_params &p, const uint8_t *x, uint8_t *y, cudaStream_t st);
int launch_vote(const uint8_t *s, int T, int B, int N, int group, int64_t stride_t,
                int64_t stride_b, float *logits, cudaStream_t st);
int launch_eval_metrics(const float *logits, const int32_t *labels, int B, int classes,
                        float *out2, cudaStream_t st);
// umma_conv_t.cu
bool umma_conv3x3_tile_supported(const snnqp_block_params &p, const float *att);
int launch_conv3x3_tile(const snnqp_block_params &p, const uint8_t *x, const int8_t *wq,
                        const float *scale, const float *bias, uint8_t *spikes, float *u_final,
                        int32_t *acc_dump, int32_t *counts, cudaStream_t st);
// umma_att.cu
bool umma_conv_att_supported(const snnqp_block_params &p, const float *att);
int launch_conv_att_umma(const snnqp_block_params &p, const uint8_t *x, const float *att, const int8_t *wq,
                         const float *scale, const float *bias, uint8_t *spikes, float *u_final, float *acc_dump,
                         int32_t *counts, cudaStream_t st);
bool umma_dense_supported(const snnqp_block_params &p, const float *att, int k_pad);
int launch_dense_umma(const snnqp_block_params &p, const uint8_t *x, const float *att, const int8_t *wq,
                      const float *scale, const float *bias, uint8_t *spikes, float *u_final, void *acc_dump,
                      cudaStream_t st);

// umma_conv1.cu
bool umma_conv1_supported(const snnqp_block_params &p, const float *att);
int launch_conv1_umma(const snnqp_block_params &p, const uint8_t *x, const int8_t *wq4, const float *scale,
                      const float *bias, uint8_t *spikes, float *u_final, int32_t *acc_dump, cudaStream_t st);

static int check_conv(const snnqp_block_params *p, const void *x, const void *wq,
                      const void *scale, const void *bias, const char *fn) {
  if (!p || !x || !wq || !scale || !bias) return invalid("%s: null pointer", fn);
  if (p->T <= 0 || p->B <= 0 || p->H <= 0 || p->W <= 0)
    return invalid("%s: bad shape T=%d B=%d H=%d W=%d", fn, p->T, p->B, p->H, p->W);
  if ((p->H & 1) || (p->W & 1)) return unsupported("%s: H=%d W=%d must be even", fn, p->H, p->W);
  if (!(p->Cin == 2 || (p->Cin % 4 == 0 && p->Cin <= 128)))
    return unsupported("%s: Cin=%d (supported: 2, or a multiple of 4 up to 128)", fn, p->Cin);
  if (p->Cout % 32 != 0 || p->Cout > 128 || p->Cout <= 0)
    return unsupported("%s: Cout=%d (supported: multiples of 32 up to 128)", fn, p->Cout);
  if (!(p->tau > 0.f)) return invalid("%s: tau=%f must be > 0", fn, (double)p->tau);
  if ((unsigned)p->x_format > SNNQP_SPIKES_BITS || (unsigned)p->y_format > SNNQP_SPIKES_BITS)
    return invalid("%s: x_format=%d y_format=%d (SNNQP_SPIKES_U8 / SNNQP_SPIKES_BITS)", fn, p->x_format, p->y_format);
  // 101..103: developer selection of one single-rounding variant (tests / tools); SNNQP_LIF_FAST = the library's pick
  if ((unsigned)p->lif_mode > SNNQP_LIF_TENSOR && !(p->lif_mode >= 101 && p->lif_mode <= 103))
    return invalid("%s: lif_mode=%d", fn, p->lif_mode);
  return SNNQP_OK;
}
static int check_popcount(const snnqp_block_params *p) {
  if (p->y_popcount && p->y_format != SNNQP_SPIKES_BITS)
    return unsupported("y_popcount needs y_format == SNNQP_SPIKES_BITS (it is the popcount of the ballot words)");
  return SNNQP_OK;
}
// SNNQP_IMPL_AUTO falling back to the dp4a SIMT kernels is a 10x+ performance cliff: say so once per process through
// snnqp_last_error() (the call itself still succeeds) instead of degrading silently.
static void note_simt_fallback(const char *what, const snnqp_block_params *p) {
  static bool noted = false;
  if (noted) return;
  noted = true;
  set_error("note: SNNQP_IMPL_AUTO ran %s on the SIMT (dp4a) kernels: shape T=%d B=%d H=%d W=%d Cin=%d Cout=%d is outside "
            "the tcgen05 envelopes (reported once)", what, p->T, p->B, p->H, p->W, p->Cin, p->Cout);
}
static bool any_bits(const snnqp_block_params *p) {
  return p->x_format == SNNQP_SPIKES_BITS || p->y_format == SNNQP_SPIKES_BITS;
}
static int bits_need_tcgen05(const char *what) {
  return unsupported("snnqp_spiking_conv3x3_fwd: bit-packed spikes are implemented by the tcgen05 kernels only (%s)", what);
}
}  // namespace snnqp

using namespace snnqp;

extern "C" {

int snnqp_spiking_conv3x3_fwd(const snnqp_block_params *p, const uint8_t *x, const float *att,
                              const int8_t *wq, const float *scale, const float *bias,
                              uint8_t *spikes, float *u_final, void *acc_dump, void *stream) {
  return snnqp_spiking_conv3x3_counts_fwd(p, x, att, wq, scale, bias, spikes, u_final, acc_dump, nullptr, stream);
}

int snnqp_spiking_conv3x3_counts_fwd(const snnqp_block_params *p, const uint8_t *x, const float *att,
                                     const int8_t *wq, const float *scale, const float *bias,
                                     uint8_t *spikes, float *u_final, void *acc_dump,
                                     int32_t *spike_counts, void *stream) {
  if (int rc = require_device()) return rc;
  if (int rc = check_conv(p, x, wq, scale, bias, "snnqp_spiking_conv3x3_fwd")) return rc;
  if (!spikes) return invalid("snnqp_spiking_conv3x3_fwd: null spikes");
  if (int rc = check_popcount(p)) return rc;
  if (att && p->Cin == 2) return unsupported("snnqp_spiking_conv3x3_fwd: att with Cin=2");
  cudaStream_t st = (cudaStream_t)stream;
  int impl = p->impl;
  if (p->Cin == 2) {
    // conv1 blob = [Cout][32] tap-major (dp4a-era layout) followed by the 4 quad matrices [4][Cout][32]
    if (impl == SNNQP_IMPL_AUTO) {
      impl = umma_conv1_supported(*p, att) ? SNNQP_IMPL_TCGEN05 : SNNQP_IMPL_SIMT;
      if (impl == SNNQP_IMPL_SIMT) note_simt_fallback("the Cin = 2 conv block", p);
    }
    if (spike_counts) return unsupported("snnqp_spiking_conv3x3_fwd: spike_counts with Cin=2");
    if (impl == SNNQP_IMPL_TCGEN05) {
      if (!umma_conv1_supported(*p, att))
        return unsupported("snnqp_spiking_conv3x3_fwd: tcgen05 conv1 path needs Cout=128, W %% 64 == 0 (got Cout=%d W=%d)",
                           p->Cout, p->W);
      return launch_conv1_umma(*p, x, wq + (int64_t)p->Cout * 32, scale, bias, spikes, u_final, (int32_t *)acc_dump, st);
    }
    if (impl != SNNQP_IMPL_SIMT) return invalid("snnqp_spiking_conv3x3_fwd: impl=%d", p->impl);
    if (any_bits(p)) return bits_need_tcgen05("conv1 outside the tcgen05 envelope or SNNQP_IMPL_SIMT");
    return launch_conv3x3_simt(*p, x, att, wq, scale, bias, spikes, u_final, acc_dump, nullptr, nullptr, st);
  }
  if (att) {
    if (any_bits(p)) return unsupported("snnqp_spiking_conv3x3_fwd: att-weighted block takes and emits SNNQP_SPIKES_U8");
    // real-valued input att * x: three byte-plane int8 contractions on tcgen05, or fp32 FMAs (SIMT)
    if (impl == SNNQP_IMPL_AUTO) {
      impl = umma_conv_att_supported(*p, att) ? SNNQP_IMPL_TCGEN05 : SNNQP_IMPL_SIMT;
      if (impl == SNNQP_IMPL_SIMT) note_simt_fallback("the attention-weighted conv block", p);
    }
    if (impl == SNNQP_IMPL_TCGEN05) {
      if (!umma_conv_att_supported(*p, att))
        return unsupported("snnqp_spiking_conv3x3_fwd: tcgen05 att path needs Cin=Cout=att_mod=128, W=8, H %% 8 == 0 "
                           "(got Cin=%d Cout=%d W=%d H=%d)", p->Cin, p->Cout, p->W, p->H);
      return launch_conv_att_umma(*p, x, att, wq, scale, bias, spikes, u_final, (float *)acc_dump, spike_counts, st);
    }
    if (impl != SNNQP_IMPL_SIMT) return invalid("snnqp_spiking_conv3x3_fwd: impl=%d", p->impl);
    return launch_conv3x3_simt(*p, x, att, wq, scale, bias, spikes, u_final, acc_dump, nullptr, spike_counts, st);
  }
  if (impl == SNNQP_IMPL_AUTO) {
    impl = umma_conv3x3_tile_supported(*p, att) ? SNNQP_IMPL_TCGEN05 : SNNQP_IMPL_SIMT;
    if (impl == SNNQP_IMPL_SIMT) note_simt_fallback("the 3x3 conv block", p);
  }
  if (impl == SNNQP_IMPL_TCGEN05) {
    if (!umma_conv3x3_tile_supported(*p, att))
      return unsupported("snnqp_spiking_conv3x3_fwd: tcgen05 path needs Cin=Cout=128, W %% 8 == 0, x strides "
                         "multiples of 16 bytes (got Cin=%d Cout=%d W=%d x_stride_t=%lld x_stride_b=%lld)",
                         p->Cin, p->Cout, p->W, (long long)p->x_stride_t, (long long)p->x_stride_b);
    return launch_conv3x3_tile(*p, x, wq, scale, bias, spikes, u_final, (int32_t *)acc_dump, spike_counts, st);
  }
  if (impl != SNNQP_IMPL_SIMT) return invalid("snnqp_spiking_conv3x3_fwd: impl=%d", p->impl);
  if (any_bits(p)) return bits_need_tcgen05("shape outside the tcgen05 envelope or SNNQP_IMPL_SIMT");
  return launch_conv3x3_simt(*p, x, att, wq, scale, bias, spikes, u_final, acc_dump, nullptr, spike_counts, st);
}

int snnqp_qconv3x3_fwd(const snnqp_block_params *p, const uint8_t *x, const int8_t *wq,
                       const float *scale, const float *bias, float *y, void *stream) {
  if (int rc = require_device()) return rc;
  if (int rc = check_conv(p, x, wq, scale, bias, "snnqp_qconv3x3_fwd")) return rc;
  if (!y) return invalid("snnqp_qconv3x3_fwd: null output");
  if (any_bits(p)) return unsupported("snnqp_qconv3x3_fwd: SNNQP_SPIKES_U8 input only");
  return launch_conv3x3_simt(*p, x, nullptr, wq, scale, bias, nullptr, nullptr, nullptr, y, nullptr,
                             (cudaStream_t)stream);
}

int snnqp_spiking_dense_fwd(const snnqp_block_params *p, const uint8_t *x, const float *att,
                            const int8_t *wq, const float *scale, const float *bias,
                            uint8_t *spikes, float *u_final, void *acc_dump, void *stream) {
  if (int rc = require_device()) return rc;
  if (!p || !x || !wq || !scale || !bias || !spikes) return invalid("snnqp_spiking_dense_fwd: null pointer");
  if (p->T <= 0 || p->B <= 0 || p->Cin <= 0 || p->Cout <= 0)
    return invalid("snnqp_spiking_dense_fwd: bad shape T=%d B=%d K=%d N=%d", p->T, p->B, p->Cin, p->Cout);
  if (!(p->tau > 0.f)) return invalid("snnqp_spiking_dense_fwd: tau must be > 0");
  if (p->x_format != SNNQP_SPIKES_U8 || p->y_format != SNNQP_SPIKES_U8 || p->y_popcount)
    return unsupported("snnqp_spiking_dense_fwd: SNNQP_SPIKES_U8 only, no y_popcount");
  const int k_pad = (p->Cin + 15) / 16 * 16;
  if (k_pad > 8192) return unsupported("snnqp_spiking_dense_fwd: K=%d too large (max 8192)", p->Cin);
  if (att && p->att_mod <= 0) return invalid("snnqp_spiking_dense_fwd: att_mod=%d", p->att_mod);
  int impl = p->impl;
  if (impl == SNNQP_IMPL_AUTO) {
    impl = umma_dense_supported(*p, att, k_pad) ? SNNQP_IMPL_TCGEN05 : SNNQP_IMPL_SIMT;
    if (impl == SNNQP_IMPL_SIMT) note_simt_fallback("the dense block", p);
  }
  if (impl == SNNQP_IMPL_TCGEN05) {
    if (!umma_dense_supported(*p, att, k_pad))
      return unsupported("snnqp_spiking_dense_fwd: tcgen05 path needs K %% 128 == 0, rows (b,t) contiguous, "
                         "att_mod=128 (got K=%d T=%d x_stride_t=%lld x_stride_b=%lld)", p->Cin, p->T,
                         (long long)p->x_stride_t, (long long)p->x_stride_b);
    return launch_dense_umma(*p, x, att, wq, scale, bias, spikes, u_final, acc_dump, (cudaStream_t)stream);
  }
  if (impl != SNNQP_IMPL_SIMT) return invalid("snnqp_spiking_dense_fwd: impl=%d", p->impl);
  return launch_dense_simt(*p, k_pad, x, att, wq, scale, bias, spikes, u_final, acc_dump,
                           (cudaStream_t)stream);
}

int snnqp_tcja_fwd(const snnqp_block_params *p, const uint8_t *spikes, const int8_t *wq_t,
                   const int8_t *wq_c, const float *scale_t, const float *scale_c,
                   int32_t *counts, float *att, void *stream) {
  if (int rc = require_device()) return rc;
  if (!p || !wq_t || !wq_c || !scale_t || !scale_c || !counts || !att)
    return invalid("snnqp_tcja_fwd: null pointer");
  if (p->Cin != 128) return unsupported("snnqp_tcja_fwd: C=%d (supported: 128)", p->Cin);
  if (p->T <= 0 || p->T > 32 || p->B <= 0 || p->H <= 0 || p->W <= 0)
    return invalid("snnqp_tcja_fwd: bad shape T=%d B=%d H=%d W=%d", p->T, p->B, p->H, p->W);
  if (p->H * p->W > (1 << 16)) return unsupported("snnqp_tcja_fwd: H*W too large");
  return launch_tcja(*p, spikes, wq_t, wq_c, scale_t, scale_c, counts, att, (cudaStream_t)stream);
}

int snnqp_maxpool2_fwd(const snnqp_block_params *p, const uint8_t *x, uint8_t *y, void *stream) {
  if (int rc = require_device()) return rc;
  if (!p || !x || !y) return invalid("snnqp_maxpool2_fwd: null pointer");
  if (p->T <= 0 || p->B <= 0 || p->H <= 0 || p->W <= 0 || (p->H & 1) || (p->W & 1) || p->Cin % 4 != 0)
    return invalid("snnqp_maxpool2_fwd: bad shape T=%d B=%d H=%d W=%d C=%d", p->T, p->B, p->H, p->W, p->Cin);
  return launch_maxpool2(*p, x, y, (cudaStream_t)stream);
}

int snnqp_vote_fwd(const uint8_t *spikes, int T, int B, int N, int group, int64_t stride_t,
                   int64_t stride_b, float *logits, void *stream) {
  if (int rc = require_device()) return rc;
  if (!spikes || !logits) return invalid("snnqp_vote_fwd: null pointer");
  if (T <= 0 || B <= 0 || N <= 0 || group <= 0 || N % group != 0)
    return invalid("snnqp_vote_fwd: T=%d B=%d N=%d group=%d", T, B, N, group);
  return launch_vote(spikes, T, B, N, group, stride_t, stride_b, logits, (cudaStream_t)stream);
}

int snnqp_eval_metrics(const float *logits, const int32_t *labels, int B, int classes,
                       float *out2, void *stream) {
  if (int rc = require_device()) return rc;
  if (!logits || !labels || !out2 || B <= 0 || classes <= 0)
    return invalid("snnqp_eval_metrics: bad arguments");
  return launch_eval_metrics(logits, labels, B, classes, out2, (cudaStream_t)stream);
}

}  // extern "C"
