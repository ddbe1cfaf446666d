// Fused DecoderResidualUnit (Vocoder/SpeechTokenizer.swift:696-718) on tcgen05: see codec_unit.cu.
#pragma once
#include <cuda_fp16.h>

#include "kernels.h"

namespace q3 {

struct CodecUnit {
  int Bt = 1, T = 0, C = 0, dil = 1;
  const __half* a = nullptr;    // [Bt][T][C] snake_act1(x): operand of the dilated 7-tap convolution
  const __half* w7 = nullptr;   // [7][C][C] fp16, K-major (conv1 of the unit)
  const float* b7 = nullptr;    // [C] or null
  const float* snake2_ea = nullptr;   // act2: v + ieb[c] * sin^2(v * ea[c])
  const float* snake2_ieb = nullptr;
  const __half* w1 = nullptr;   // [C][C] fp16 (conv2 of the unit, kernel 1)
  int w7_reps = 1, w1_reps = 1;  // copies of the weights (ConvW::w16_reps), *_rep_stride halves apart: CTA i reads copy i % reps
  size_t w7_rep_stride = 0, w1_rep_stride = 0;
  const float* b1 = nullptr;
  const __half* res16 = nullptr;  // [Bt*T][C] x, the fp16 residual stream
  __half* outr16 = nullptr;       // x' (may alias res16: a tile reads its own rows before it writes them); null: not needed
  __half* out16 = nullptr;        // snake_next(x'); must NOT alias `a` (other tiles still read their halo rows from it)
  const float* next_ea = nullptr;
  const float* next_ieb = nullptr;
};

// the shapes the fused kernel runs (C % 32 == 0, C <= 192, 128 + 6 * dil <= 192 halo rows, >= 32 row tiles)
bool codec_unit_shape_supported(int Bt, int T, int C, int dil);
// the shape is supported, every required operand is set and Q3TTS_CODEC_UNIT is not 0
bool codec_unit_supported(const CodecUnit& u);
// runs any supported shape with its operands set, whatever Q3TTS_CODEC_UNIT says: the decoder picks between this and the two-kernel
// form with codec_unit_supported
void launch_codec_unit(const LaunchCtx& c, const CodecUnit& u);
void init_codec_unit();

}  // namespace q3
