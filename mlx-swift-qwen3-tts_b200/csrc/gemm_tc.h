// tcgen05 / TMEM / TMA implicit-GEMM for sm_100a: the dense contractions of the codec decoder (causal convs, polyphase
// transposed convs, linears) and of batched talker decode / prefill.
//
//   Y[m, n] = epilogue( sum_tap sum_c A[b, t - shift(tap), c] * W[tap][n][c] ),   m = b*T + t,  shift(tap) = (ntap-1-tap)*dil
//
// A: fp16 activations, channels-last [Bt, T, Cin]; rows with negative source time are zero-filled by TMA (causal padding).
// W: fp16 weights [ntap][N][Cin] (K-major).  Accumulation fp32 in TMEM; epilogue in registers.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "kernels.h"

namespace q3 {

enum TcAct { TC_ACT_NONE = 0, TC_ACT_GELU = 1, TC_ACT_SILU = 2 };

struct TcGemm {
  // problem
  const __half* a = nullptr;  // [Bt][T][cin]
  const __half* w = nullptr;  // [ntap][N][cin]
  int w_reps = 1;             // copies of w, w_rep_stride halves apart (codec.h ConvW::w16_reps): CTA i of the 128-row-tile kernel reads copy i % reps
  size_t w_rep_stride = 0;
  int Bt = 1, T = 0, cin = 0, N = 0, ntap = 1, dil = 1;
  // epilogue
  const float* bias = nullptr;   // [N]
  const float* res = nullptr;    // [M][ld_res]: y = res + scale[n] * (acc + bias)   (may alias out32)
  int ld_res = 0;
  const float* scale = nullptr;  // [N] or null (= 1)
  int act = TC_ACT_NONE;
  int swiglu = 0;                // columns (2i, 2i+1) = (gate_i, up_i): out column i = silu(gate) * up, N_out = N / 2
  float* out32 = nullptr;        // [M][ld32] or null
  int ld32 = 0;
  // fp16 storage of a residual stream (128-row-tile kernel only; the codec's vocoder blocks, whose fp32 stream was the largest
  // HBM consumer of a pass): res16 [M][ld_res] replaces res, outr16 [M][ld32] replaces out32 (the value BEFORE the SnakeBeta
  // transform that out16 carries); arithmetic stays fp32
  const __half* res16 = nullptr;
  __half* outr16 = nullptr;
  __half* out16 = nullptr;       // [M][ld16] or null: fp16 copy (operand of the next contraction)
  int ld16 = 0;
  const float* snake_ea = nullptr;   // SnakeBeta of the NEXT layer fused into the fp16 copy: v + ieb[ch] * sin^2(v * ea[ch]),
  const float* snake_ieb = nullptr;  // ch = n % snake_ch (Vocoder/SpeechTokenizer.swift:105-109)
  int snake_ch = 0;
  float* pcm = nullptr;              // output conv: column 0 only, clip(-1, 1) + NaN scrub, [M] (SpeechTokenizer.swift:823-840, 951)
  // RMSNorm folded around the contraction (Model/Qwen3Layers.swift:8-26 with the norm WEIGHT multiplied into the columns of W at
  // load, TalkerEngine::make_tc): the activation operand is a = fp16(x * in_scale) of the un-normalised residual stream x, and
  // row m of the accumulator is multiplied by (1 / in_scale) * rsqrt(mean(x[m]^2) + rms_eps) before bias / activation.
  //   rms_in = 1: the kernel computes the row factors itself from `a` (skinny kernel only: its epilogue warps do it while the
  //               operands stream in, in the fixed order of tc_row_sumsq_f16);
  //   row_scale : precomputed factors [M] (launch_row_scale, same summation order) for the 128-row-tile kernel.
  int rms_in = 0;
  float rms_eps = 0.0f, in_scale = 1.0f;
  const float* row_scale = nullptr;
  float out16_scale = 1.0f;          // out16 = fp16(y * out16_scale): the producer side of the same scheme
  // 0: always the 128-row-tile kernel, whatever the row count.  Prefill uses it so that a request's numbers do not depend on
  // how many rows of OTHER requests shared its GEMMs (the two kernels add the K dimension up in different orders).
  int allow_skinny = 1;
  // 0: every CTA of the 128-row-tile kernel walks K from 0 (default: from a per-CTA offset, which spreads same-address L2 reads
  // but makes the fp32 summation order -- the low bits of a row's result -- depend on the tile shape, i.e. on the row count)
  int k_rotate = 1;
  // Packed weights as the streamed operand (<= 128-row kernel, gemm_skinny_q.cu): when q_w is set and the shape qualifies
  // (tc_skinny_q_supported) the kernel reads the MLX-packed matrix [N][cin * q_bits / 32] uint32 + scales / biases [N][cin / q_group]
  // of dtype q_sdt and dequantises inside; `w` (the fp16 copy of the same matrix) is the fallback operand and may be null only if
  // the caller checked tc_skinny_q_supported first.  q_fold (fp32 [cin], may be null) is multiplied into the dequantised columns
  // before the fp16 rounding -- the RMSNorm weight in front of this linear, exactly what TalkerEngine::make_tc folds into `w`.
  // q_halves: the packed matrix is [gate ; up] (N / 2 rows each) while the kernel's tile rows are interleaved (gate_i, up_i), as in `w`.
  const uint32_t* q_w = nullptr;
  const void* q_scales = nullptr;
  const void* q_biases = nullptr;
  const float* q_fold = nullptr;
  int q_bits = 0, q_group = 64, q_sdt = Q3TTS_BF16, q_halves = 0;
};

// true when the tcgen05 path can run this shape (else the caller uses the SIMT kernel)
bool tc_gemm_supported(const TcGemm& g);
void launch_tc_gemm(const LaunchCtx& c, const TcGemm& g);
void init_tc_gemm();  // resolves cuTensorMapEncodeTiled, sets kernel attributes; once per process/device

// Skinny variant for <= 128 activation rows (batched decode steps, short codec windows), gemm_skinny.cu: the WEIGHT tile is the
// 128-row UMMA operand, the activation rows are the N dimension, K is split across a thread-block cluster and reduced through
// distributed shared memory, so a [m <= 128] x N x K linear spreads over ~all SMs instead of N/bn CTAs walking all of K.
// launch_tc_gemm routes to it when tc_skinny_supported(g).
bool tc_skinny_supported(const TcGemm& g);
void launch_tc_skinny(const LaunchCtx& c, const TcGemm& g);
void init_tc_skinny();
bool tc_skinny_q_supported(const TcGemm& g);
void launch_tc_skinny_q(const LaunchCtx& c, const TcGemm& g);
void init_tc_skinny_q();
unsigned long long* tc_skinny_trace_buf();
// measurement hook: per-CTA phase stamps (10 x u64 per CTA) of the following launches go to dev_buf (null = off)
void tc_skinny_set_trace(unsigned long long* dev_buf);
void tc_skinny_grid(const TcGemm& g, int* tiles, int* split, int* stages);

// shared host helpers (gemm_tc.cu)
void tc_resolve_encode();
typedef CUresult (*TcEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                               CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TcEncodeFn tc_encode_fn();  // cuTensorMapEncodeTiled resolved through the runtime (after tc_resolve_encode)
CUtensorMap tc_make_map(const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box);

// fp32 -> fp16 helpers used around the tensor-core contractions
void launch_f32_to_f16(const LaunchCtx& c, const float* x, size_t n, __half* y);
// RMSNorm (fp32 in) -> fp16 out
// (w may be null = ones: the norm weight lives in the consumer's folded fp16 copy)
void launch_rmsnorm_f16(const LaunchCtx& c, const float* x, int ldx, int m, int dim, const float* w, float eps, __half* y, int ldy);
// y = fp16(x * scale), elementwise (entry of a stack on the folded-RMSNorm path)
void launch_scale_to_f16(const LaunchCtx& c, const float* x, size_t n, float scale, __half* y);
// rs[m] = (1 / in_scale) * rsqrt(sum(a[m][:]^2) / (in_scale^2 * dim) + eps) for fp16 rows a = fp16(x * in_scale)
void launch_row_scale(const LaunchCtx& c, const __half* a, int m, int dim, float in_scale, float eps, float* rs);

}  // namespace q3
