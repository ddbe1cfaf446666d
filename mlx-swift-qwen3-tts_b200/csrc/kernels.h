// Launchers of the hand-written sm_100a kernels (talker side).  Every launcher counts itself into LaunchCtx.
#pragma once
#include <cuda_fp16.h>

#include "model.h"

namespace q3 {

struct LaunchCtx {
  cudaStream_t stream = nullptr;
  LaunchCounter* counter = nullptr;
  inline void tick() const { if (counter) counter->tick(); }
};

enum Epilogue { EPI_STORE = 0, EPI_ADD = 1, EPI_SILU = 2, EPI_SWIGLU = 3 };

// MLX dequantized() — bit-exact contract in include/qwen3tts_b200.h.  dst [out][in] of out_dt.
// MLX affine quantiser (group 64, bits 4 / 6 / 8) into an 8-bit container + scales / biases in the weight dtype; `fake`: dequantised copy
void launch_mlx_quantize(const LaunchCtx& c, const void* w, int wdt, int out, int in, int bits, uint32_t* qw8, void* scales, void* biases,
                         void* fake);
void launch_dequantize(const LaunchCtx& c, const uint32_t* qw, const void* scales, const void* biases, int sdt, int out,
                       int in, int group, int bits, int out_dt, void* dst);

// The word width the kernels read a b-bit MLX checkpoint in: 2 / 3 / 4 bits -> 4-bit words, 5 / 6 / 8 bits -> 8-bit words, 0 = a width
// MLX does not write.  Codes are copied unchanged, so dequantised values do not depend on the container.
inline int container_bits(int bits) {
  return (bits == 2 || bits == 3 || bits == 4) ? 4 : ((bits == 5 || bits == 6 || bits == 8) ? 8 : 0);
}
// src: [rows][in * bits / 32] uint32 of MLX's b-bit bit stream (bits 2, 3, 5, 6; in % 32 == 0) -> dst: [rows][in * cb / 32] uint32 in the
// container_bits(bits) = cb word layout of launch_dequantize / launch_linear.  Scales and biases are untouched.
void launch_widen_bits(const LaunchCtx& c, const uint32_t* src, int rows, int in, int bits, uint32_t* dst);

// MLX mxfp4 leaves -> the exact 8-bit affine container of group 32 with bf16 scales / biases that launch_dequantize / launch_linear
// read.  packed: [rows][in / 8] uint32, E2M1 code j of a word at bits 4j; scale_bytes: [rows][in / 32] E8M0 bytes, each < 252 (the
// caller checks: larger exponents do not fit the container).  Element (c, e) = lut[c] * 2^(e - 127) becomes q = 2 lut[c] + 12 with
// scale 2^(e - 128) and bias -12 * 2^(e - 128): both are powers of two times small integers, so scale * q + bias is exact in fp32 and
// equals the E2M1 value (-0 becomes +0).  codes8_out: [rows][in / 4] uint32; scales_out / biases_out: [rows][in / 32] bf16.
constexpr int kMxfp4MaxScaleByte = 251;
void launch_mxfp4_to_affine(const LaunchCtx& c, const uint32_t* packed, const uint8_t* scale_bytes, int rows, int in, uint32_t* codes8_out,
                            uint16_t* scales_out, uint16_t* biases_out);

// y[m][*] (op)= epilogue( rmsnorm?(x[m][:]) . W^T + bias ).   x, y fp32 with row strides ldx / ldy.
// norm_w != null fuses Qwen3RMSNorm (Model/Qwen3Layers.swift:18-25) into the prologue.
// EPI_SWIGLU: W rows are [gate ; up]; y[m][r] = silu(gate_r) * up_r, r < out/2 (Model/Qwen3Layers.swift:236).
void launch_linear(const LaunchCtx& c, const Linear& L, const float* x, int ldx, int m, float* y, int ldy,
                   const float* norm_w, float eps, int epilogue);

// y = x * rsqrt(mean(x^2) + eps) * w over the last dim (Model/Qwen3Layers.swift:18-25)
void launch_rmsnorm(const LaunchCtx& c, const float* x, int ldx, int m, int dim, const float* w, float eps, float* y, int ldy);

// Per (row, head): q/k per-head RMSNorm (:174-175), rotate-half RoPE at the row's absolute position (:187-195),
// q written back in place, k and v appended to the KV ring of the row's slot (:197-201).
struct KVLayout {
  void* k = nullptr;       // base of this layer's K cache for slot 0: [kv_heads][capacity][head_dim] of float, or of __half when f16
  void* v = nullptr;
  size_t slot_stride = 0;  // ELEMENTS between consecutive slots
  int capacity = 0;        // ring size in positions
  int f16 = 0;             // element type: 0 fp32 (handles of <= 2 slots, code predictor), 1 fp16 (talker KV of batched handles)
};
void launch_qk_norm_rope_append(const LaunchCtx& c, float* qkv, int ld, int m, int heads, int kv_heads, int head_dim,
                                const float* q_norm, const float* k_norm, float eps, const float* inv_freq,
                                const int* row_slot, const int* row_pos, const KVLayout& kv);

// code-predictor pass 0 on the decode path: rows (2s, 2s+1) = positions (0, 1) of slot s; norm + RoPE + append + causal attention
void launch_cp_pass0_attention_f16(const LaunchCtx& c, const float* qkv, int ld, int n_slots, int heads, int kv_heads, const float* q_norm,
                                   const float* k_norm, float eps, const float* inv_freq, const KVLayout& kv, __half* out, int ldo);

// softmax(q k^T / sqrt(d)) v over keys [win_start[slot], row_pos] of the row's slot, GQA by head / group (:203-216)
void launch_attention(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, int head_dim,
                      const int* row_slot, const int* row_pos, const int* win_start, const KVLayout& kv, float* out,
                      int ldo);

// decode-step fusion of the two launches above (valid when every slot has ONE row in the launch)
void launch_rope_attention(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, const float* q_norm,
                           const float* k_norm, float eps, const float* inv_freq, const int* row_slot, const int* row_pos,
                           const int* win_start, const KVLayout& kv, float* out, int ldo);
void launch_rope_attention_f16(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, const float* q_norm,
                               const float* k_norm, float eps, const float* inv_freq, const int* row_slot, const int* row_pos,
                               const int* win_start, const KVLayout& kv, __half* out, int ldo);
// same attention, fp16 output (A operand of the tcgen05 o_proj)
void launch_attention_f16(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, int head_dim,
                          const int* row_slot, const int* row_pos, const int* win_start, const KVLayout& kv, __half* out, int ldo);
// dense weight (bf16 / f16 / f32) -> fp16 copy; optional row interleave of two halves ([gate ; up] -> gate_0, up_0, gate_1, ...)
// col_scale (fp32 [cols], may be null): dst[r][c] = fp16(w[r][c] * col_scale[c]) -- an RMSNorm weight folded into the consumer linear
void launch_weight_to_f16(const LaunchCtx& c, const void* w, int dt, int rows, int cols, bool interleave_halves, __half* dst,
                          const float* col_scale = nullptr);
void launch_gather_rows_f16(const LaunchCtx& c, const Embedding& e, const int* ids, int n, __half* y, int ldy);

// rows of an embedding table -> fp32: y[i][:] (= or +=) table[ids[i]][:]
void launch_gather_rows(const LaunchCtx& c, const Embedding& e, const int* ids, int n, float* y, int ldy, bool accumulate);

// prompt assembly (Model/Qwen3Talker.swift:354-433): row r = (tp >= 0 ? tp_rows[tp] : 0) + (codec >= 0 ?
// codec_embedding[codec] : 0) + (spk > 0 ? speaker_embedding[spk - 1] : 0)
void launch_assemble_rows(const LaunchCtx& c, const float* tp_rows, int H, const Embedding& codec, const float* spk,
                          const int* desc /*[n][3] = tp, codec, spk*/, int n, float* y);

// Voice prefixes (q3tts_voice): the K / V of positions [0, n_pos) of one slot's talker rings <-> a compact buffer
// [2 (K, V)][layers][kv_heads][n_pos][128] of the rings' element type (elem_bytes 2 = fp16, 4 = fp32).  Ring index = position
// (a prefix is shorter than the ring).  One launch covers every entry of the device table, every layer and every kv head.
struct KvPrefixEntry {
  void* compact;
  int slot;
  int n_pos;
};
void launch_kv_prefix_copy(const LaunchCtx& c, const KvPrefixEntry* table, int n_entries, int max_pos, void* k, void* v, size_t slot_stride,
                           size_t layer_stride, int layers, int kv_heads, int capacity, int elem_bytes, bool to_ring);

// ---- per-slot generation state living in HBM (read / written only by kernels during graph replay) ----------
struct SlotState {
  int active;           // slot holds a running utterance
  int finished;         // EOS / pad-run / max_tokens reached
  int step;             // loop counter of Model/Qwen3Talker.swift:464
  int n_frames;         // raw frames recorded
  int pos;              // absolute position of the NEXT talker input (positionOffset, :438)
  int win_start;        // first absolute position still inside the KV window (trimKVCache, Qwen3Layers.swift:111-124)
  int trailing_idx, total_text;  // :444, 462
  int consecutive_pad;  // :445
  int max_tokens;
  int n_forced;         // teacher forcing: frames to force (0 = free running)
  int stream_variant;   // 1 = no repetition penalty on code-predictor groups (:821)
  int top_k;
  int frame_alive;      // this frame is being produced (set by the code0 sampler, cleared at frame end)
  int logits_cap;       // frames of logits to dump (0 = none)
  int pad_;
  float temperature, top_p, rep_penalty, pad2_;
  unsigned long long seed;
};

struct SamplerParams {
  int vocab;             // V of this head
  int group;             // 0 = code0 (codec_head), g >= 1 = code-predictor group g-1
  int codec_vocab;       // config.vocab_size: valid-token mask applies when vocab == codec_vocab (:316-319)
  int eos_id, pad_id;
  int groups;            // 16
  int set_words;         // uint32 words per token-set bitmap
};
// One block per slot: Qwen3Talker.sampleToken (:274-322) + the loop's EOS/pad logic for group 0 (:470-494).
// What the sampler CTA of a slot writes once the group's token is known: the code predictor's next input rows
// (Model/Qwen3Talker.swift:503-510).  mode 0: nothing; 1 (after group 0): rows (2s, 2s+1) = [h_last[s], codec_embedding[code0]];
// 2 (after group g in 1..14): row s = cp_codec_embedding[g-1][code_g].  y16 (optional) = fp16(row * y16_scale).
struct NextInput {
  int mode = 0, H = 0;
  const float* h_last = nullptr;
  Embedding codec;
  const Embedding* cp_emb = nullptr;  // device array of the 15 code-predictor tables
  float* y32 = nullptr;
  __half* y16 = nullptr;
  float y16_scale = 1.0f;
};
void launch_sample(const LaunchCtx& c, const float* logits, int ld, int n_slots, SlotState* st, const SamplerParams& p,
                   unsigned* token_sets /*[slot][16][set_words]*/, int* cur_codes /*[slot][16]*/,
                   const int* forced /*[slot][max_frames][16] or null*/, int max_frames,
                   float* logits_dump /*[cap][...] of slot `dump_slot`, or null*/, int dump_stride_frame, int dump_offset,
                   int dump_slot, const NextInput& next = NextInput());

// standalone sampler probe (q3tts_sample_token)
void launch_sample_probe(const LaunchCtx& c, const float* logits, int vocab, int codec_vocab, float temperature, int top_k,
                         float top_p, float rep_penalty, const unsigned* set_bitmap, unsigned long long seed,
                         unsigned long long counter, int* id_out);

// q3tts_sampler_probe: sample_block on rows r < n_rows (logits + r * ld, V entries), one CTA per row, each row with its own
// parameters (device arrays of n_rows; sets = [n_rows][kMaxVocab / 32] bitmaps or null).  form 0 = the 512-thread form of
// sample_kernel, 1 = the 480-thread named-barrier form of frame_megakernel.  processed (or null): [n_rows][V], the row just before the
// Gumbel step (greedy rows: after the penalty).
struct SamplerProbeRows {
  const float* temperature;
  const int* top_k;
  const float* top_p;
  const float* rep_penalty;
  const unsigned* sets;
  const unsigned long long* seed;
  const unsigned long long* counter;
};
void launch_sampler_probe(const LaunchCtx& c, int form, const float* logits, int ld, int n_rows, int V, int codec_vocab,
                          const SamplerProbeRows& rows, int* ids, float* processed);
// launch_sample's work (NextInput mode 0) in the form frame_megakernel's sample_phase runs it: sample_slot<1, 480> (q3tts_sampler_slot_probe)
void launch_sample_frame_form(const LaunchCtx& c, const float* logits, int ld, int n_slots, SlotState* st, const SamplerParams& p,
                              unsigned* token_sets, int* cur_codes, const int* forced, int max_frames, float* logits_dump,
                              int dump_stride_frame, int dump_offset, int dump_slot);

// code-predictor input rows (Model/Qwen3Talker.swift:503-510): pass 0 -> rows (2s, 2s+1) = [h_last[s], codec_embedding[code0]];
// pass g >= 1 -> row s = cp_codec_embedding[g-1][codes[s][g]]
void launch_cp_input(const LaunchCtx& c, int pass, int n_slots, const float* h_last, int H, const Embedding& codec,
                     const Embedding* cp_emb_dev /*[15] device array*/, const int* cur_codes, float* y);

// frame end (Model/Qwen3Talker.swift:526-549, 554-558): record the frame, add code0 to its set, build the next talker
// input = (trailing text row | tts_pad) + sum of the 16 code embeddings, advance trailing_idx.
void launch_frame_finalize(const LaunchCtx& c, int n_slots, SlotState* st, const int* cur_codes, int* frames_out,
                           int max_frames, unsigned* token_sets, int set_words, const float* trailing /*[slot][max_trailing][H]*/,
                           int max_trailing, const float* tts_pad /*[H]*/, const Embedding& codec,
                           const Embedding* cp_emb_dev, int H, float* x_next, __half* x16_next = nullptr, float x16_scale = 1.0f);
// after the talker step: pos++, step++, window trim every 15th step, max_tokens stop
void launch_step_advance(const LaunchCtx& c, int n_slots, SlotState* st, int window);
// row metadata for the talker step: row s -> (slot s, pos[s])
void launch_step_rows(const LaunchCtx& c, int n_slots, const SlotState* st, int* row_slot, int* row_pos, int* win_start);

}  // namespace q3
