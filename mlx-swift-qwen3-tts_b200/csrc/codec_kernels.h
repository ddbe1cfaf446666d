// Launchers of the codec-decoder kernels.
#pragma once
#include "codec.h"

namespace q3 {

void init_codec_kernels();
// Y[m,n] = epi(bias[n] + sum_tap X[m - shift(tap)] . W[tap][n]),  m = b*T + t, rows with t - shift < 0 read zeros.
// CE_RES_SCALE: y = res + scale[n] * (.)  (scale == null -> 1); y may alias res.
void launch_conv_gemm(const LaunchCtx& c, const float* x, const ConvW& w, float* y, const float* res, const float* scale, int M,
                      int T, int epi);
// SnakeW here carries the precomputed exp(alpha) and 1/(exp(beta)+1e-9)
void launch_snake(const LaunchCtx& c, const float* x, const SnakeW& s, size_t rows, float* y);
void launch_dwconv7(const LaunchCtx& c, const float* x, const float* w, const float* b, int C, int T, size_t rows, float* y);
void launch_layernorm(const LaunchCtx& c, const float* x, int rows, int C, const float* w, const float* b, float eps, float* y);
void launch_layernorm_f16(const LaunchCtx& c, const float* x, int rows, int C, const float* w, const float* b, float eps, __half* y);
void launch_silu_mul(const LaunchCtx& c, const float* gu, size_t rows, int I, float* y);
void launch_codec_rope(const LaunchCtx& c, float* qkv, int ld, int M, int T, int n_rot_heads, const float* inv_freq);
void launch_codec_attention(const LaunchCtx& c, const float* qkv, int ld, int B, int T, int nh, int nkv, float* out, int ldo);
// mma: the mma.sync kernel (when ld % 4 == 0 and ldo % 2 == 0) or the SIMT kernel
void launch_codec_attention_f16(const LaunchCtx& c, const float* qkv, int ld, int B, int T, int nh, int nkv, __half* out, int ldo, bool mma = true);
// ICL audio encoder (audio_encoder.cu)
void launch_codec_attention_bidir(const LaunchCtx& c, const float* qkv, int ld, int B, int T, int nh, int nkv, float* out, int ldo);
void launch_elu(const LaunchCtx& c, const float* x, size_t total, float* y);
void launch_rvq_encode(const LaunchCtx& c, const float* lat_sem, const float* lat_ac, const float* const* books, const float* const* books_sq, int n_sem,
                       int n_out, int D, int size, int T, int* codes);
void launch_rvq_embed(const LaunchCtx& c, const int* codes, const float* const* codebooks, int Q, int n_sem, int D, int size, int M,
                      float* emb);
void launch_out_conv(const LaunchCtx& c, const float* x, const float* w, const float* bias, int C, int B, int T, float* y);
void launch_out_conv_f16(const LaunchCtx& c, const __half* x, const float* w, const float* bias, int C, int B, int T, float* y);
// streaming form (one pass over the activations, weights in registers); C in {32, 64, 96, 128}
bool out_conv_stream_supported(int C);
// strip_rows: outputs per warp, rounded down to a multiple of 32; below 32 = the default (256)
void launch_out_conv_stream_f16(const LaunchCtx& c, const __half* x, const float* w, const float* bias, int C, int B, int T, float* y,
                                int strip_rows = 0);
// emb fp32 [M][2D] (bit-exact gather-sums) and/or its fp16 copy
void launch_rvq_embed_f16(const LaunchCtx& c, const int* codes, const float* const* codebooks, int Q, int n_sem, int D, int size, int M,
                          __half* emb16);

}  // namespace q3
