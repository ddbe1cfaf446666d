// Config + device-weight descriptors for the talker / code predictor (host side of the library).
// Shape source of truth = config.json as decoded by Qwen3TTSConfig (Model/Qwen3Config.swift:208-253).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "common.h"
#include "json.h"
#include "safetensors.h"

namespace q3 {

struct CPConfig {  // Model/Qwen3Config.swift:21-33
  int hidden_size = 1024, num_hidden_layers = 5, num_attention_heads = 16, num_key_value_heads = 8, head_dim = 128;
  int intermediate_size = 3072, max_position_embeddings = 65536, vocab_size = 2048, num_code_groups = 16;
  float rms_norm_eps = 1e-6f, rope_theta = 1000000.0f;
};

// `mode` of an MLX quantisation block; the values are those of q3tts_info.checkpoint_quant_mode
enum QuantMode { QMODE_AFFINE = 0, QMODE_MXFP4 = 1 };

struct TalkerConfig {  // Model/Qwen3Config.swift:65-128
  int hidden_size = 0, num_hidden_layers = 0, vocab_size = 0, text_vocab_size = 0, text_hidden_size = 2048;
  int num_attention_heads = 0, num_key_value_heads = 8, head_dim = 128, intermediate_size = 0;
  int max_position_embeddings = 0;
  float rms_norm_eps = 1e-6f, rope_theta = 1000000.0f;
  int tts_bos_token_id = 151672, tts_eos_token_id = 151673, tts_pad_token_id = 151671;
  int codec_bos_id = 2149, codec_eos_token_id = 2150, codec_pad_id = 2148;
  int codec_nothink_id = 2155, codec_think_bos_id = 2156, codec_think_eos_id = 2157;
  std::vector<std::pair<std::string, int>> spk_id;
  CPConfig cp;
  bool has_mrope = false;  // interleaved MRoPE == plain RoPE for the identical position streams fed (Qwen3Layers.swift:75-92)
  std::string tts_model_type;
  bool has_quantization = false, has_quantization_config = false;
  int q_bits = 0, q_group = 64;      // from `quantization`
  int qc_bits = 0, qc_group = 64;    // from `quantization_config`
  int q_mode = QMODE_AFFINE, qc_mode = QMODE_AFFINE;  // `mode` of each block (absent = affine)
};

TalkerConfig parse_talker_config(const Json& root);

// One QuantizedLayerFactory.linear leaf (Model/QuantizedLayerFactory.swift:49-66) resident in HBM.
struct Linear {
  int out = 0, in = 0;
  int bits = 0;   // 0 = dense `w`, else MLX affine packed `qw` + scales/biases
  int group = 64;
  int sdt = Q3TTS_BF16;            // dtype of scales/biases (quantised) or of `w` (dense) and of `bias`
  const uint32_t* qw = nullptr;    // [out][in*bits/32]
  const void* scales = nullptr;    // [out][in/group]
  const void* biases = nullptr;    // [out][in/group]
  const void* w = nullptr;         // [out][in]
  const float* bias = nullptr;     // [out] fp32 (Linear bias), or null
  size_t weight_bytes() const {    // algorithmic bytes streamed per invocation (SURVEY.md §8d)
    if (bits) return (size_t)out * in * bits / 8 + (size_t)out * (in / group) * 2 * dtype_size(sdt) + (bias ? out * 4 : 0);
    return (size_t)out * in * dtype_size(sdt) + (bias ? out * 4 : 0);
  }
};

// fp16 dense copy of a Linear for the tcgen05 path (rows >= 16: batched decode, prefill)
struct TcLinear {
  const void* w = nullptr;  // __half [out][in]
  int out = 0, in = 0;
  const float* bias = nullptr;
  // the packed leaf this copy was made from (bits == 0: dense checkpoint): decode steps of <= 128 rows stream THESE bytes and
  // dequantise inside the GEMM (gemm_skinny_q.cu); `w` remains the operand of prefill (128-row-tile kernel)
  const uint32_t* qw = nullptr;
  const void* qscales = nullptr;
  const void* qbiases = nullptr;
  const float* fold = nullptr;   // RMSNorm weight folded into the columns (same as in `w`), or null
  int qbits = 0, qgroup = 64, qsdt = Q3TTS_BF16;
  bool halves = false;           // packed rows are [gate ; up]; `w` rows are interleaved (gate_i, up_i)
};

struct Embedding {
  const void* w = nullptr;
  int rows = 0, dim = 0, dt = Q3TTS_BF16;
};

struct LayerWeights {
  Linear qkv;     // rows [q ; k ; v]  (three reference leaves concatenated along `out` at load)
  Linear o;
  Linear gate_up; // rows [gate ; up]
  Linear down;
  const float *in_norm = nullptr, *post_norm = nullptr, *q_norm = nullptr, *k_norm = nullptr;  // fp32
};

struct LayerTc { TcLinear qkv, o, gate_up_il /* rows interleaved (gate_i, up_i) */, down; };

struct StackWeights {  // a Qwen3 decoder stack (talker or code predictor)
  int hidden = 0, layers = 0, heads = 0, kv_heads = 0, head_dim = 128, inter = 0;
  float eps = 1e-6f, theta = 1e6f;
  std::vector<LayerWeights> layer;
  std::vector<LayerTc> tc;  // empty when the tcgen05 copies were not built
  const float* final_norm = nullptr;
};

struct TalkerWeights {
  StackWeights talker, cp;
  Embedding text_embedding, codec_embedding;
  std::vector<Embedding> cp_codec_embedding;  // 15 x [2048][H_talker]
  Linear fc1, fc2;                            // text_projection
  Linear codec_head;
  std::vector<Linear> lm_head;                // 15
  Linear small_to_mtp;                        // out == 0 when absent
  bool has_mtp = false;
  TcLinear fc1_tc, fc2_tc, codec_head_tc, small_to_mtp_tc;
  std::vector<TcLinear> lm_head_tc;
  bool has_tc = false;
  size_t talker_step_bytes = 0, cp_pass_bytes = 0;  // algorithmic weight bytes per invocation
  int checkpoint_bits = 0;  // width of the packed leaves on disk (2..8), 0 = dense; the kernels read 4 / 8-bit words (Linear::bits)
  int checkpoint_mode = QMODE_AFFINE;  // QMODE_MXFP4: E2M1 leaves held as exact 8-bit affine groups of 32 (launch_mxfp4_to_affine)
};

// Loads `model.safetensors` with the key remap of Qwen3Talker.load (Model/Qwen3Talker.swift:117-137).
void load_talker_weights(const std::string& model_dir, const TalkerConfig& cfg, DeviceArena& arena, cudaStream_t stream,  // NOLINT
                         TalkerWeights& out, int& weight_dtype, int& eff_bits, int& eff_group, bool runtime_quantization = false);

// host float conversions
inline float bf16_to_f32(uint16_t v) {
  uint32_t u = (uint32_t)v << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
float f16_to_f32(uint16_t v);
std::vector<float> to_f32_host(const STensor& t);

}  // namespace q3
