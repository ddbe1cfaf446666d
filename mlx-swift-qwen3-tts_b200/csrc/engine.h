// The handle behind the C ABI: talker engine (slots, KV rings, frame-step graphs) + codec decoder.
#pragma once
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "frame_kernel.h"
#include "kernels.h"

namespace q3 {

class CodecDecoder;  // codec.h
class AudioEncoder;       // audio_encoder.h
class SpeakerEncoderDev;  // speaker_encoder.h

struct EngineOptions {
  int device = 0;
  cudaStream_t stream = nullptr;
  int max_batch = 1, kv_capacity = 512, max_frames = 2400, use_cuda_graph = 1;
  int load_codec = 1, load_talker = 1, codec_max_frames = 2400, codec_max_batch = 8;
  int lanes = 1;  // q3tts_options.lanes
  int max_trailing = 1024;
  int packed_gemm = 0;  // q3tts_options::packed_gemm
  int runtime_quantization = 0;  // q3tts_options::runtime_quantization
};

// Result of admitting one request into a slot.
struct Admission {
  bool too_short = false;  // < 9 text ids: the reference returns [] (Model/Qwen3Talker.swift:348-352)
  int prefill_len = 0;
};

struct TalkerShared;

// q3tts_voice: the talker K / V of a voice's prompt prefix (positions [0, prefix_len)), prefilled once on the handle that created it.
// Immutable; holds a reference on the weights, so it may outlive that handle.  Accepted by every handle with the same weights and
// options (the creator and its clones): same numeric path, same ring element type.
struct VoicePrefix {
  std::shared_ptr<TalkerShared> shared;
  int device = 0, max_batch = 0, kv_capacity = 0, kv_f16 = 0, handle_tc = 0;
  int prefix_len = 0;  // P - 1 of every request in this voice
  int role[3] = {0, 0, 0};
  void* kv = nullptr;  // [2 (K, V)][layers][kv_heads][prefix_len][128], fp16 when kv_f16 else fp32 (cudaMalloc: outlives arenas)
  size_t bytes = 0;
  ~VoicePrefix();
};

// Immutable after load: the checkpoint's tensors (packed / dense, runtime-quantised when asked) and the fp16 tensor-core copies.  Shared
// by a handle and its clones (q3tts_clone): every handle owns its stream, KV rings, slot state and activation buffers, none owns the weights.
struct TalkerShared {
  DeviceArena arena;
  TalkerWeights w;
  int weight_dtype = Q3TTS_BF16, eff_bits = 0, eff_group = 64;
  std::mutex mu;  // building the tensor-core copies (first handle of >= 3 slots)
};

class TalkerEngine {
 public:
  TalkerEngine(const std::string& model_dir, const TalkerConfig& cfg, const EngineOptions& opt, cudaStream_t stream,
               LaunchCounter* counter, std::shared_ptr<TalkerShared> shared = nullptr);  // shared: a clone (weights are not loaded again)
  ~TalkerEngine();

  // Prompt assembly + prefill of `req` into `slot` (Model/Qwen3Talker.swift:344-462).
  Admission admit(int slot, const q3tts_request& req);
  struct AdmitItem { int slot; const q3tts_request* req; };
  // Several utterances at once: one concatenated prefill pass (rows carry their own slot / position).
  void admit_batch(const std::vector<AdmitItem>& items, std::vector<Admission>& out);
  // q3tts_voice_create: prefills the voice part of `r` (rows [0, P-1)) in a scratch slot and copies its K / V out into v.kv
  void create_voice(const q3tts_request& r, VoicePrefix& v);
  // the voice rules of a request (q3tts_request::voice): exclusive fields, role ids, a voice this handle accepts; host only
  void check_voice_request(const q3tts_request& r) const;
  int max_prefill_rows() const { return max_rows_; }
  // slot count a frame step is issued for when `hi` slots are in use: the row bucket of the tensor-core GEMMs (32 / 64 / 128 ...)
  // on batched handles, `hi` itself on the <= 2-slot handles of the persistent frame kernel
  int step_slots(int hi) const {
    if (!handle_tc_) return hi;
    int b = hi <= 32 ? 32 : (hi <= 64 ? 64 : (hi + 127) / 128 * 128);
    return b < opt_.max_batch ? b : opt_.max_batch;
  }
  // Run `n` frame steps for slots [0, n_slots) — CUDA-graph replay when enabled.
  void run_frames(int n_slots, int n);
  // Read back slot states (synchronises the stream).
  void fetch_states(int n_slots, std::vector<SlotState>& out);
  // Copy raw frames [first, first+count) of `slot` into host memory (synchronises).
  void fetch_frames(int slot, int first, int count, int32_t* dst);
  void fetch_logits(int frames, float* code0_out, float* cp_out);
  int dump_slot() const { return dump_enabled_ ? dump_slot_ : -1; }
  void release(int slot);
  void drop_graphs();

  const TalkerConfig& config() const { return cfg_; }
  const TalkerWeights& weights() const { return w_; }
  int max_batch() const { return opt_.max_batch; }
  int kv_capacity() const { return opt_.kv_capacity; }
  int max_frames() const { return opt_.max_frames; }
  int weight_dtype() const { return shared_->weight_dtype; }
  int quant_bits() const { return shared_->eff_bits; }
  int checkpoint_quant_bits() const { return w_.checkpoint_bits; }
  int checkpoint_quant_mode() const { return w_.checkpoint_mode; }
  int quant_group() const { return shared_->eff_group; }
  size_t device_bytes() const { return arena_.total() + (owns_weights_ ? shared_->arena.total() : 0); }  // a clone reports its own state only
  const std::shared_ptr<TalkerShared>& shared() const { return shared_; }
  size_t weight_bytes_per_frame() const { return w_.talker_step_bytes + 15 * w_.cp_pass_bytes; }
  int64_t graph_replays = 0, graph_nodes_replayed = 0, mega_launches = 0;
  bool megakernel_enabled() const { return mega_.ok; }
  double last_prefill_ms = 0;
  int64_t last_prefill_rows = 0;

  // measurement hook (q3tts_profile_linear)
  double profile_linears(int which, int m, int iters, int64_t& launches, int64_t& bytes_per_iter);
  // probe used by q3tts_sample_token
  int sample_probe(const float* logits, int vocab, float temperature, int top_k, float top_p, float rep_penalty,
                   const int32_t* token_set, int n_set, uint64_t seed, uint64_t counter);

 private:
  // one_row_per_slot: decode steps may fuse norm+RoPE+append into the attention launch (prefill / CP pass 0 may not);
  // decode_step: rows <= 128 may take the split-K cluster GEMM (prefill stays on the 128-row-tile kernel: batch invariance)
  void forward_stack(const StackWeights& S, float* x, int m, const int* row_slot, const int* row_pos, const int* win_start,
                     const float* inv_freq, void* kbase, void* vbase, int kv_f16, size_t slot_stride, size_t layer_stride, int capacity,
                     bool one_row_per_slot, bool decode_step, bool x16_ready);
  void issue_frame(int n_slots);
  // Prompt assembly (Model/Qwen3Talker.swift:338-433), ONE copy for admission and voice creation.  A PromptBatch collects the rows of
  // several prompts: text ids to project ([0, 3) = tts bos / eos / pad), one (tp, codec, speaker) descriptor per prefill row with its
  // (slot, position), and the speaker vectors.
  struct PromptBatch {
    std::vector<int> ids, desc, row_slot, row_pos;
    std::vector<float> spk;
  };
  PromptBatch new_prompt_batch() const;
  // the voice rows [0, P-1) of `r` at positions 0.. of `slot` (validated as admission validates them); returns P - 1
  int voice_rows(PromptBatch& b, int slot, const q3tts_request& r);
  // firstText row of `r` at position `pos` (codec bos + text_ids[3]) and its trailing text ids; returns the first trailing id's index
  int text_rows(PromptBatch& b, int slot, int pos, const q3tts_request& r);
  // uploads a PromptBatch, runs text_projection over its ids and assembles its rows into d_x_ (d_tp_ keeps the projected ids)
  void assemble_prompt(const PromptBatch& b);
  KvPrefixEntry* d_voice_tab_ = nullptr;  // [max_batch] voice prefixes to install in one admission round
  void build_tc_weights();
  void build_mega_plan();
  TcLinear make_tc(const Linear& L, bool interleave_halves, const float* fold = nullptr);
  // prefill / prompt assembly: the SAME per-handle rule as decode steps, never the row count of the call -- a request prefilled
  // alone and the same request prefilled next to others must see the same arithmetic.  Batched handles prefill on the 128-row-tile
  // tcgen05 kernel (row-count invariant); handles of <= 2 slots keep fp32 activations end to end (dequant-fused SIMT linears)
  bool use_tc(int) const { return handle_tc_; }
  // decode steps: ONE numeric path per handle, fixed at creation from max_batch (not from how many slots happen to be live in a
  // frame), so a request's codes do not depend on what it is co-batched with or on utterances finishing around it:
  //   max_batch >= tc_min_rows_ (3)  -> every decode step on the tcgen05 GEMMs (fp16 operands, fp32 accumulate)
  //   max_batch <= 2                 -> the persistent frame kernel (fp32 activations), else the SIMT graph path
  bool use_tc_step(int) const { return handle_tc_; }
  bool use_mega(int n_slots) const { return mega_.ok && !handle_tc_ && opt_.max_batch <= mega_.max_slots && n_slots <= mega_.max_slots; }
  // y = epilogue(x16 . W^T): one tcgen05 GEMM launch over m rows
  void linear_tc(const TcLinear& L, const void* x16, int m, float* out32, int ld32, void* out16, int ld16, const float* res, int act, int swiglu, bool row_count_invariant = false);
  LaunchCtx ctx() { return LaunchCtx{stream_, counter_}; }

  TalkerConfig cfg_;
  EngineOptions opt_;
  cudaStream_t stream_;
  LaunchCounter* counter_;
  DeviceArena arena_;                     // this handle's state: KV rings, slots, activations, plans
  std::shared_ptr<TalkerShared> shared_;  // the weights (declared before w_: w_ refers into it)
  bool owns_weights_ = false;
  TalkerWeights& w_;

  int max_rows_ = 0, max_tp_rows_ = 0, set_words_ = 0;
  // max_batch from which a handle runs on tensor cores and keeps fp16 KV rings (env Q3TTS_TC_MIN_ROWS; 0 disables).  Decode steps
  // switch at 3 utterances: measured per frame-step (0.6B 4-bit) 6.5 / 10.3 / 17.2 ms at 3 / 8 / 12 rows on the SIMT path against a
  // flat 3.45-3.5 ms on the split-K cluster GEMM; 1-2 utterances stay on the persistent frame kernel (2.2 ms).
  int tc_min_rows_ = 3;
  bool step_tc_ = false;  // set by issue_frame for the launches of the current frame step
  bool handle_tc_ = false;  // decode steps of this handle run on tensor cores (see use_tc_step)
  // 3..128-row GEMMs of a quantised checkpoint read the packed weights (gemm_skinny_q.cu) instead of the fp16 copies: q3tts_options::
  // packed_gemm.  Off by default: at 64 rows the frame step is a chain of ~570 dependent launches, not a bandwidth problem, and the
  // dequantisation in front of the MMAs lengthens every link (measured 4.95-5.4 ms against 4.18 ms per frame-step; DESIGN.md 3.2).
  bool packed_gemm_ = false;
  void attach_packed(struct TcGemm& g, const TcLinear& L) const;
  float* d_rs_ = nullptr;                     // [max_rows] RMSNorm row factors for the 128-row-tile kernel (prefill)
  static constexpr float kX16Div = 16.0f;     // the fp16 copy of the residual stream is x / 16 (range headroom; exact power of two)
  void *d_h16_ = nullptr, *d_attn16_ = nullptr, *d_act16_ = nullptr, *d_tpe16_ = nullptr, *d_tph16_ = nullptr;
  // device buffers
  // talker KV rings: fp16 on handles whose decode steps run on tensor cores (half the bytes of every window walk; K / V rounded once
  // at append, like every other fp16 operand of that path), fp32 on the <= 2-slot handles of the persistent frame kernel
  void *kcache_ = nullptr, *vcache_ = nullptr;
  int kv_f16_ = 0;
  float *cp_k_ = nullptr, *cp_v_ = nullptr;
  size_t kv_slot_stride_ = 0, kv_layer_stride_ = 0, cpkv_slot_stride_ = 0, cpkv_layer_stride_ = 0;
  static constexpr int kCpCapacity = 32;
  SlotState* d_state_ = nullptr;
  int *d_step_slot_ = nullptr, *d_step_pos_ = nullptr, *d_win_ = nullptr;
  int *d_cp_slot2_ = nullptr, *d_cp_pos2_ = nullptr, *d_iota_ = nullptr, *d_cp_pos_ = nullptr;  // cp_pos [16][B]
  int *d_pf_slot_ = nullptr, *d_pf_pos_ = nullptr, *d_pf_win_ = nullptr;
  float *d_x_ = nullptr, *d_qkv_ = nullptr, *d_attn_ = nullptr, *d_act_ = nullptr;
  float *d_hlast_ = nullptr, *d_logits0_ = nullptr, *d_cplogits_ = nullptr, *d_cpin_ = nullptr, *d_cpx_ = nullptr, *d_xstep_ = nullptr;
  int *d_cur_codes_ = nullptr, *d_frames_ = nullptr, *d_forced_ = nullptr;
  unsigned* d_sets_ = nullptr;
  float *d_trailing_ = nullptr, *d_tts_ = nullptr;  // tts rows: bos, eos, pad
  float *d_tpe_ = nullptr, *d_tph_ = nullptr, *d_tp_ = nullptr, *d_spk_ = nullptr;
  int *d_ids_ = nullptr, *d_desc_ = nullptr;
  Embedding* d_cp_emb_ = nullptr;
  float *d_inv_freq_ = nullptr, *d_cp_inv_freq_ = nullptr;
  float *d_dump0_ = nullptr, *d_dumpcp_ = nullptr;  // logits dumps of slot 0 (allocated on first use)
  int dump_cap_ = 0, dump_slot_ = 0;  // the slot whose logits are dumped (one request per handle at a time)
  bool dump_enabled_ = false;
  float* d_probe_logits_ = nullptr;
  unsigned* d_probe_set_ = nullptr;
  int* d_probe_out_ = nullptr;
  // pinned staging
  int* h_stage_ = nullptr;
  size_t h_stage_ints_ = 0;
  SlotState* h_state_ = nullptr;
  cudaEvent_t ev_a_ = nullptr, ev_b_ = nullptr;

  struct Graph {
    cudaGraphExec_t exec = nullptr;
    int64_t nodes = 0;
  };
  std::map<long long, Graph> graphs_;  // key: n_slots * 8192 + (dump_enabled ? 1 + dump_slot : 0)
  MegaPlan mega_;                // persistent frame kernel (batch-1 decode); !ok -> graph path
};

struct Handle {
  std::mutex mu;
  std::string model_dir;
  std::string last_error;
  bool poisoned = false;  // a kernel fault (trap, illegal address) left the CUDA context unusable: every later call fails the same way
  EngineOptions opt;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  LaunchCounter counter;
  TalkerConfig cfg;
  bool has_talker = false;
  std::unique_ptr<TalkerEngine> talker;
  std::unique_ptr<CodecDecoder> codec;
  std::unique_ptr<AudioEncoder> audio_encoder;  // ICL reference-audio encoder, when the checkpoint carries one
  std::unique_ptr<SpeakerEncoderDev> speaker_encoder;  // ECAPA-TDNN speaker encoder, when model.safetensors carries `speaker_encoder.*`
  q3tts_timing timing{};
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
  float* h_pcm = nullptr;  // pinned staging for PCM read-back
  size_t h_pcm_floats = 0;
  int32_t* h_codes = nullptr;
  size_t h_codes_ints = 0;
  int32_t* d_codes = nullptr;  // grow-only device staging of the codec passes
  size_t d_codes_ints = 0;
  float* d_pcm = nullptr;
  size_t d_pcm_floats = 0;
  // A stream owns talker slot 0 from q3tts_stream_begin to q3tts_stream_free: while it is open, every other talker call on
  // the handle (and a second stream) fails with Q3TTS_ERR_INVALID_ARG instead of silently re-admitting the slot.
  void* open_stream = nullptr;
  // q3tts_options.lanes > 1: clones of this handle (created on the first call that needs them), destroyed with it
  std::mutex lanes_mu;
  std::vector<Handle*> lanes;
  ~Handle();
};

}  // namespace q3

struct q3tts_voice : q3::VoicePrefix {};
