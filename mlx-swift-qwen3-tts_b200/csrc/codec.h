// Speech-tokenizer decoder (12.5 Hz codes -> 24 kHz PCM) on device.  Replaces Qwen3TTSSpeechTokenizerDecoder
// (Vocoder/SpeechTokenizer.swift:844-988) and the weight sanitiser of Vocoder/AudioDecoder.swift:196-305.
// Activations are channels-last [B, T, C] end to end (the reference transposes NCL<->NLC around every conv).
#pragma once
#include <string>
#include <vector>

#include <cuda_fp16.h>

#include "common.h"
#include "json.h"
#include "kernels.h"
#include "safetensors.h"

namespace q3 {

struct CodecConfig {  // Vocoder/SpeechTokenizer.swift:42-74
  int latent_dim = 1024, codebook_dim = 512, codebook_size = 2048, decoder_dim = 1536, hidden_size = 512;
  int intermediate_size = 1024, head_dim = 64, num_attention_heads = 16, num_hidden_layers = 8, num_key_value_heads = 16;
  int num_quantizers = 16, num_semantic_quantizers = 1, max_position_embeddings = 8000, sliding_window = 72;
  float layer_scale_initial_scale = 0.01f, rms_norm_eps = 1e-5f, rope_theta = 10000.0f;
  bool attention_bias = false;
  std::vector<int> upsample_rates{8, 5, 4, 3}, upsampling_ratios{2, 2};
  int total_upsample() const {
    int t = 1;
    for (int r : upsample_rates) t *= r;
    for (int r : upsampling_ratios) t *= r;
    return t;
  }
};
CodecConfig parse_codec_config(const Json& root);

// A causal (dilated) conv / transposed conv / linear, all as  Y[b,t,n] = bias[n] + sum_tap X[b, t-(ntap-1-tap)*dil, :] . W[tap][n][:]
struct ConvW {
  const float* w = nullptr;   // [ntap][n][cin] fp32
  const __half* w16 = nullptr;  // same, fp16: B operand of the tcgen05 path
  // Small weights that EVERY CTA re-reads once per 128-row tile are stored w16_reps times, w16_rep_stride halves apart; CTA i reads copy
  // i % reps.  One copy of a 130-520 KB matrix maps unevenly onto the 184 L2 slices, and 148 SMs x ~170 tiles of re-reads then queue on the
  // fullest slice (measured: the thin vocoder stages ran at 1 800 B/clk of the ~6 300 B/clk the L2 can deliver).
  int w16_reps = 1;
  size_t w16_rep_stride = 0;
  const float* bias = nullptr;  // [n] or null
  int ntap = 1, dil = 1, cin = 0, n = 0;
  int64_t flops_per_row() const { return 2ll * ntap * cin * n; }
};

enum ConvEpilogue { CE_STORE = 0, CE_GELU = 1, CE_RES_SCALE = 2 };

struct SnakeW { const float *alpha = nullptr, *beta = nullptr; int ch = 0; };

// bytes between the copies of an fp16 weight of `halves` elements (ConvW::w16_reps): each copy starts 256-byte aligned
inline size_t f16_rep_stride_bytes(size_t halves) { return (halves * sizeof(__half) + 255) / 256 * 256; }

class CodecDecoder {
 public:
  CodecDecoder(const std::string& dir, cudaStream_t stream, LaunchCounter* counter, int pass_frames);
  ~CodecDecoder();
  const CodecConfig& config() const { return cfg_; }
  int total_upsample() const { return up_; }
  int pass_frames() const { return pass_frames_; }
  size_t device_bytes() const { return arena_.total() + ws_bytes_; }
  int vq_dim() const { return cfg_.codebook_dim / 2; }

  // decodeImpl (Vocoder/SpeechTokenizer.swift:917-952): d_codes [B][T][Q] int32 -> d_pcm [B][T*up] fp32 (clipped to [-1,1]).
  // B*T must be <= pass_frames().  Eager launches: a CUDA graph of a pass rarely pays back its capture (DESIGN.md §7).
  void decode_pass(const int32_t* d_codes, int B, int T, float* d_pcm);
  bool uses_tensor_cores() const { return use_tc_; }
  // code -> embedding gather-sums (bit-exact probe): d_first/d_rest [B*T][vq_dim]
  void rvq_embed(const int32_t* d_codes, int B, int T, float* d_first, float* d_rest);
  int64_t flops_per_frame() const { return flops_per_frame_; }

 private:
  void ensure_workspace(int frames);
  void decode_pass_simt(const int32_t* d_codes, int B, int T, float* d_pcm);
  void decode_pass_tc(const int32_t* d_codes, int B, int T, float* d_pcm);
  void finish_weight(ConvW& w);           // uploads the fp16 copy, updates use_tc_
  const __half* upload_f16(const std::vector<float>& h, int reps = 1, size_t* rep_stride = nullptr);
  LaunchCtx ctx() const { return LaunchCtx{stream_, counter_}; }
  ConvW load_conv(const std::map<std::string, STensor>& t, const std::string& key, int cout, int cin_per_group, int k, int dil, bool bias);
  ConvW load_convT(const std::map<std::string, STensor>& t, const std::string& key, int cin, int cout, int k, int stride);
  ConvW load_linear(const std::map<std::string, STensor>& t, const std::string& key, int cout, int cin, bool bias);
  const float* load_vec(const std::map<std::string, STensor>& t, const std::string& key, int n);
  SnakeW load_snake(const std::map<std::string, STensor>& t, const std::string& prefix, int ch);

  CodecConfig cfg_;
  cudaStream_t stream_;
  LaunchCounter* counter_;
  DeviceArena arena_;
  int up_ = 1920, pass_frames_ = 0;
  int64_t flops_per_frame_ = 0;

  // weights
  std::vector<const float*> codebooks_;  // num_quantizers x [codebook_size][vq_dim]
  const float** d_codebooks_ = nullptr;
  ConvW rvq_proj_;      // [first | rest] (2*vq_dim) -> codebook_dim, no bias
  ConvW pre_conv_;
  ConvW tr_in_, tr_out_;
  struct TLayer {
    ConvW qkv, o, gate_up, down;
    ConvW gate_up_il;  // rows interleaved (gate_i, up_i) for the fused SwiGLU epilogue of the tcgen05 path
    const float *in_norm, *post_norm, *attn_scale, *mlp_scale;
  };
  std::vector<TLayer> tl_;
  const float* tr_norm_ = nullptr;
  const float* d_inv_freq_ = nullptr;
  struct Up {
    ConvW convT;  // as a 1-tap conv with n = factor * C
    int factor;
    const float *dw_w, *dw_b;  // depthwise [7][C], [C]
    const float *ln_w, *ln_b, *gamma;
    ConvW pw1, pw2;
  };
  std::vector<Up> ups_;
  ConvW init_conv_;
  struct Unit { SnakeW act1, act2; ConvW conv1, conv2; };
  struct Block { SnakeW snake; ConvW convT; int rate; int cin, cout; Unit unit[3]; };
  std::vector<Block> blocks_;
  SnakeW out_snake_;
  const float *out_w_ = nullptr, *out_b_ = nullptr;  // [7][C], [1]
  ConvW out_tc_;                                    // the same conv as a 32-column tcgen05 tile (column 0 real)
  int out_ch_ = 0;

  bool use_tc_ = true;  // every dense contraction fits the tcgen05 path (cin % 8 == 0, N % 32 == 0); else the fp32 SIMT pipeline runs
  // workspace (grow-only); the tcgen05 pipeline uses ws_[0..2] as fp32 and hs_[0..2] as fp16 operand buffers
  __half* hs_[3] = {nullptr, nullptr, nullptr};
  float* ws_[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t ws_floats_ = 0, ws_bytes_ = 0;
  int ws_frames_ = 0;
};

}  // namespace q3
