// Talker engine: slot state in HBM, KV rings, prompt assembly + prefill, and the device-resident frame step
// (code0 sample -> 15 code-predictor passes -> frame finalize -> talker step) replayed as one CUDA graph so the 16
// host syncs per frame of the reference loop (Model/Qwen3Talker.swift:482, 520) disappear.
#include <algorithm>
#include <cmath>

#include "engine.h"
#include "frame_kernel.h"
#include "gemm_tc.h"

namespace q3 {

void init_talker_kernels();  // talker_kernels.cu: opt-in shared-memory attributes, once per device
int mega_max_blocks_per_sm(int fmt, int slots, size_t smem);  // frame_kernel.cu

TalkerEngine::TalkerEngine(const std::string& model_dir, const TalkerConfig& cfg, const EngineOptions& opt, cudaStream_t stream,
                           LaunchCounter* counter, std::shared_ptr<TalkerShared> shared)
    : cfg_(cfg), opt_(opt), stream_(stream), counter_(counter), shared_(shared ? shared : std::make_shared<TalkerShared>()),
      owns_weights_(!shared), w_(shared_->w) {
  init_talker_kernels();
  if (owns_weights_)
    load_talker_weights(model_dir, cfg_, shared_->arena, stream_, w_, shared_->weight_dtype, shared_->eff_bits, shared_->eff_group,
                        opt_.runtime_quantization != 0);
  const int B = opt_.max_batch, C = opt_.kv_capacity, F = opt_.max_frames;
  const int H = cfg_.hidden_size, Hcp = cfg_.cp.hidden_size;
  Q3_CHECK(B >= 1 && C >= 208 && F >= 1, Q3TTS_ERR_INVALID_ARG, "bad options: max_batch %d kv_capacity %d max_frames %d", B, C, F);
  const StackWeights &T = w_.talker, &P = w_.cp;
  // rows of one batched pass: a decode step (<= 2B), one prompt (<= C), or the prefill of a whole admission batch
  max_rows_ = std::max(std::max(2 * B, C), std::min(B * 96, 8192));
  max_tp_rows_ = std::max(C + opt_.max_trailing + 8, std::min(B * 128, 16384));
  set_words_ = (std::max(cfg_.vocab_size, cfg_.cp.vocab_size) + 31) / 32;

  kv_layer_stride_ = (size_t)T.kv_heads * C * 128;
  kv_slot_stride_ = kv_layer_stride_ * T.layers;
  // decided here (before the tensor-core copies exist) from the same inputs handle_tc_ is decided from below
  if (const char* e = getenv("Q3TTS_TC_MIN_ROWS")) tc_min_rows_ = atoi(e);
  {
    const char* e16 = getenv("Q3TTS_KV_F16");
    kv_f16_ = (tc_min_rows_ > 0 && B >= tc_min_rows_ && !(e16 && atoi(e16) == 0)) ? 1 : 0;
  }
  const size_t kv_elem = kv_f16_ ? 2 : 4;
  kcache_ = arena_.alloc(kv_slot_stride_ * B * kv_elem);
  vcache_ = arena_.alloc(kv_slot_stride_ * B * kv_elem);
  cpkv_layer_stride_ = (size_t)P.kv_heads * kCpCapacity * 128;
  cpkv_slot_stride_ = cpkv_layer_stride_ * P.layers;
  cp_k_ = arena_.alloc_n<float>(cpkv_slot_stride_ * B);
  cp_v_ = arena_.alloc_n<float>(cpkv_slot_stride_ * B);

  d_state_ = arena_.alloc_n<SlotState>(B);
  Q3_CUDA(cudaMemsetAsync(d_state_, 0, sizeof(SlotState) * B, stream_));
  d_step_slot_ = arena_.alloc_n<int>(B); d_step_pos_ = arena_.alloc_n<int>(B); d_win_ = arena_.alloc_n<int>(B);
  d_cp_slot2_ = arena_.alloc_n<int>(2 * B); d_cp_pos2_ = arena_.alloc_n<int>(2 * B);
  d_iota_ = arena_.alloc_n<int>(B); d_cp_pos_ = arena_.alloc_n<int>(16 * B);
  d_pf_slot_ = arena_.alloc_n<int>(max_rows_); d_pf_pos_ = arena_.alloc_n<int>(max_rows_); d_pf_win_ = arena_.alloc_n<int>(B);
  Q3_CUDA(cudaMemsetAsync(d_pf_win_, 0, sizeof(int) * B, stream_));
  Q3_CUDA(cudaMemsetAsync(d_win_, 0, sizeof(int) * B, stream_));

  const int wide_h = std::max(H, Hcp);
  const int qkv_w = std::max((T.heads + 2 * T.kv_heads) * 128, (P.heads + 2 * P.kv_heads) * 128);
  const int attn_w = std::max(T.heads, P.heads) * 128;
  const int act_w = std::max(T.inter, P.inter);
  d_x_ = arena_.alloc_n<float>((size_t)max_rows_ * wide_h);
  d_qkv_ = arena_.alloc_n<float>((size_t)max_rows_ * qkv_w);
  d_attn_ = arena_.alloc_n<float>((size_t)max_rows_ * attn_w);
  d_act_ = arena_.alloc_n<float>((size_t)max_rows_ * act_w);
  d_hlast_ = arena_.alloc_n<float>((size_t)B * H);
  d_logits0_ = arena_.alloc_n<float>((size_t)B * cfg_.vocab_size);
  d_cplogits_ = arena_.alloc_n<float>((size_t)B * cfg_.cp.vocab_size);
  d_cpin_ = arena_.alloc_n<float>((size_t)2 * B * H);
  d_cpx_ = arena_.alloc_n<float>((size_t)2 * B * Hcp);
  d_xstep_ = arena_.alloc_n<float>((size_t)B * H);
  d_cur_codes_ = arena_.alloc_n<int>((size_t)B * 16);
  Q3_CUDA(cudaMemsetAsync(d_cur_codes_, 0, sizeof(int) * B * 16, stream_));
  d_frames_ = arena_.alloc_n<int>((size_t)B * F * 16);
  d_forced_ = arena_.alloc_n<int>((size_t)B * F * 16);
  d_sets_ = arena_.alloc_n<unsigned>((size_t)B * 16 * set_words_);
  d_trailing_ = arena_.alloc_n<float>((size_t)B * opt_.max_trailing * H);
  d_tts_ = arena_.alloc_n<float>((size_t)3 * H);
  d_tpe_ = arena_.alloc_n<float>((size_t)max_tp_rows_ * cfg_.text_hidden_size);
  d_tph_ = arena_.alloc_n<float>((size_t)max_tp_rows_ * cfg_.text_hidden_size);
  d_tp_ = arena_.alloc_n<float>((size_t)max_tp_rows_ * H);
  d_spk_ = arena_.alloc_n<float>((size_t)B * H);
  d_ids_ = arena_.alloc_n<int>(max_tp_rows_);
  d_desc_ = arena_.alloc_n<int>((size_t)3 * max_rows_);
  // tensor-core copies: built when the handle can see >= tc_min_rows_ rows at once (batched decode, or any prefill)
  if (tc_min_rows_ > 0 && B >= tc_min_rows_) {  // batched handle: fp16 copies for prefill, packed weights for decode steps
    init_tc_gemm();
    {
      std::lock_guard<std::mutex> lk(shared_->mu);
      if (!w_.has_tc) build_tc_weights();  // a clone finds them built
    }
    d_h16_ = arena_.alloc((size_t)max_rows_ * std::max(wide_h, cfg_.text_hidden_size) * 2);
    d_attn16_ = arena_.alloc((size_t)max_rows_ * attn_w * 2);
    d_act16_ = arena_.alloc((size_t)max_rows_ * act_w * 2);
    d_rs_ = arena_.alloc_n<float>((size_t)max_rows_);
    d_tpe16_ = arena_.alloc((size_t)max_tp_rows_ * cfg_.text_hidden_size * 2);
    d_tph16_ = arena_.alloc((size_t)max_tp_rows_ * cfg_.text_hidden_size * 2);
  }
  handle_tc_ = w_.has_tc && tc_min_rows_ > 0 && B >= tc_min_rows_;
  {
    const char* e = getenv("Q3TTS_SKINNY_Q");
    packed_gemm_ = opt_.packed_gemm == 1 || (opt_.packed_gemm == 0 && e && atoi(e) != 0);
  }
  Q3_CHECK(!kv_f16_ || handle_tc_ || !w_.has_tc, Q3TTS_ERR_BAD_CONFIG, "internal: fp16 KV rings on a handle without the tensor-core step");
  d_probe_logits_ = arena_.alloc_n<float>(4096);
  d_probe_set_ = arena_.alloc_n<unsigned>(128);
  d_probe_out_ = arena_.alloc_n<int>(1);

  // static row metadata for the code-predictor passes
  std::vector<int> slot2(2 * B), pos2(2 * B), iota(B), cpos(16 * B);
  for (int s = 0; s < B; ++s) {
    slot2[2 * s] = slot2[2 * s + 1] = s;
    pos2[2 * s] = 0; pos2[2 * s + 1] = 1;
    iota[s] = s;
    for (int g = 0; g < 16; ++g) cpos[g * B + s] = g + 1;
  }
  Q3_CUDA(cudaMemcpy(d_cp_slot2_, slot2.data(), slot2.size() * 4, cudaMemcpyHostToDevice));
  Q3_CUDA(cudaMemcpy(d_cp_pos2_, pos2.data(), pos2.size() * 4, cudaMemcpyHostToDevice));
  Q3_CUDA(cudaMemcpy(d_iota_, iota.data(), iota.size() * 4, cudaMemcpyHostToDevice));
  Q3_CUDA(cudaMemcpy(d_cp_pos_, cpos.data(), cpos.size() * 4, cudaMemcpyHostToDevice));

  // inv_freq = 1 / pow(base, Float(2i) / Float(dim))  in fp32 (Model/Qwen3Layers.swift:45; Qwen3CodePredictor.swift:16)
  std::vector<float> f(64), fc(64);
  for (int i = 0; i < 64; ++i) {
    f[i] = 1.0f / powf(cfg_.rope_theta, (float)(2 * i) / 128.0f);
    fc[i] = 1.0f / powf(cfg_.cp.rope_theta, (float)(2 * i) / 128.0f);
  }
  d_inv_freq_ = arena_.alloc_n<float>(64); d_cp_inv_freq_ = arena_.alloc_n<float>(64);
  Q3_CUDA(cudaMemcpy(d_inv_freq_, f.data(), 256, cudaMemcpyHostToDevice));
  Q3_CUDA(cudaMemcpy(d_cp_inv_freq_, fc.data(), 256, cudaMemcpyHostToDevice));

  d_cp_emb_ = arena_.alloc_n<Embedding>(15);
  Q3_CUDA(cudaMemcpy(d_cp_emb_, w_.cp_codec_embedding.data(), sizeof(Embedding) * 15, cudaMemcpyHostToDevice));

  h_stage_ints_ = (size_t)max_tp_rows_ + 3 * (size_t)C + 64;
  Q3_CUDA(cudaMallocHost(&h_stage_, h_stage_ints_ * sizeof(int)));
  Q3_CUDA(cudaMallocHost(&h_state_, sizeof(SlotState) * B));
  Q3_CUDA(cudaEventCreate(&ev_a_));
  Q3_CUDA(cudaEventCreate(&ev_b_));

  // tts_{bos,eos,pad} rows through text_projection(text_embedding(.)) (Model/Qwen3Talker.swift:354-358)
  h_stage_[0] = cfg_.tts_bos_token_id; h_stage_[1] = cfg_.tts_eos_token_id; h_stage_[2] = cfg_.tts_pad_token_id;
  for (int i = 0; i < 3; ++i)
    Q3_CHECK(h_stage_[i] >= 0 && h_stage_[i] < cfg_.text_vocab_size, Q3TTS_ERR_BAD_CONFIG, "tts special token id %d outside text vocab", h_stage_[i]);
  Q3_CUDA(cudaMemcpyAsync(d_ids_, h_stage_, 12, cudaMemcpyHostToDevice, stream_));
  LaunchCtx c{stream_, nullptr};
  launch_gather_rows(c, w_.text_embedding, d_ids_, 3, d_tpe_, cfg_.text_hidden_size, false);
  launch_linear(c, w_.fc1, d_tpe_, cfg_.text_hidden_size, 3, d_tph_, cfg_.text_hidden_size, nullptr, 0.f, EPI_SILU);
  launch_linear(c, w_.fc2, d_tph_, cfg_.text_hidden_size, 3, d_tts_, H, nullptr, 0.f, EPI_STORE);
  Q3_CUDA(cudaStreamSynchronize(stream_));
  build_mega_plan();
}

// Plan of the persistent frame kernel (frame_kernel.cu): the frame's linears in execution order, the shared-memory
// layout, and the envelope checks.  Anything outside the envelope keeps the CUDA-graph path (mega_.ok stays false).
void TalkerEngine::build_mega_plan() {
  mega_ = MegaPlan{};
  if (const char* e = getenv("Q3TTS_MEGAKERNEL"))
    if (atoi(e) == 0) return;
  if (!opt_.use_cuda_graph) return;
  const StackWeights &T = w_.talker, &P = w_.cp;
  std::vector<const Linear*> order;
  std::vector<int> swiglu;
  struct Norms { const float *norm_w, *q_norm, *k_norm; };
  struct PhaseInfo { int in_kind, pass, epi, out_sel, flags, layer, unit, tkind; };
  std::vector<Norms> norms;
  std::vector<PhaseInfo> phase;
  // InKind / EpiKind values of frame_kernel.cu
  enum { IN_GX = 0, IN_GX_LAST, IN_CP0, IN_CPG, IN_TALKER, IN_ATTN, IN_ACT };
  enum { E_STORE = 0, E_ADD_RAW = 1, E_SWIGLU = 2 };
  auto push = [&](const Linear& L, bool sw, PhaseInfo ph, const float* nw = nullptr, const float* qn = nullptr, const float* kn = nullptr) {
    order.push_back(&L); swiglu.push_back(sw ? 1 : 0); norms.push_back({nw, qn, kn}); phase.push_back(ph);
  };
  for (int u = 0; u < 16; ++u) {  // units 0..14: code-predictor passes, 15: the talker step
    const bool talker = (u == 15);
    const StackWeights& S = talker ? T : P;
    const int base = (talker ? MF_TALKER : 0) | (u == 0 ? MF_ROWS2 : 0);
    const int first_kind = talker ? IN_TALKER : (u == 0 ? IN_CP0 : IN_CPG);
    bool first = true;
    auto flags_of = [&](int extra) { const int f = base | extra | (first ? MF_UNIT_START : 0); first = false; return f; };
    const bool mtp = !talker && w_.has_mtp;
    if (mtp) push(w_.small_to_mtp, false, {first_kind, u, E_STORE, 0, flags_of(0), 0, u, 0});
    for (int l = 0; l < S.layers; ++l) {
      const LayerWeights& lw = S.layer[l];
      const int qkv_in = (l == 0 && !mtp) ? first_kind : IN_GX;
      push(lw.qkv, false, {qkv_in, u, E_STORE, 1, flags_of(MF_ATTN | MF_KEEP_RAW | ((talker && l == 0) ? MF_FINALIZE : 0)), l, u, 1}, lw.in_norm, lw.q_norm, lw.k_norm);
      push(lw.o, false, {IN_ATTN, u, E_ADD_RAW, 0, flags_of(0), l, u, 2});
      push(lw.gate_up, true, {IN_GX, u, E_SWIGLU, 2, flags_of(MF_KEEP_RAW), l, u, 3}, lw.post_norm);
      push(lw.down, false, {IN_ACT, u, E_ADD_RAW, 0, flags_of(0), l, u, 4});
    }
    if (talker) push(w_.codec_head, false, {IN_GX, u, E_STORE, 3, flags_of(MF_HEAD | MF_KEEP_RAW), 0, u, 5}, T.final_norm);
    else push(w_.lm_head[u], false, {IN_GX_LAST, u == 0 ? 2 : 1, E_STORE, 3, flags_of(MF_HEAD), 0, u, 5}, P.final_norm);
  }
  // one weight format for the whole frame
  const Linear& L0 = *order[0];
  int fmt = -1;
  if (L0.bits == 4) fmt = 0; else if (L0.bits == 8) fmt = 1;
  else if (L0.bits == 0) fmt = L0.sdt == Q3TTS_BF16 ? 2 : (L0.sdt == Q3TTS_F16 ? 3 : 4);
  if (fmt < 0) return;
  const int vpl = fmt == 0 ? 32 : (fmt == 1 ? 16 : (fmt == 4 ? 4 : 8));
  const int kc = 32 * vpl;
  std::vector<MegaLinear> lin;
  int kmax = 0, need_slot = 0;
  for (size_t i = 0; i < order.size(); ++i) {
    const Linear& L = *order[i];
    if (L.bits != L0.bits || (L.bits == 0 && L.sdt != L0.sdt)) return;
    if (L.bits && (L.group % vpl != 0 || L.in % L.group != 0)) return;
    if (L.in % vpl != 0 || L.in % 4 != 0) return;
    MegaLinear m{};
    m.w = L.bits ? (const void*)L.qw : L.w; m.scales = L.scales; m.biases = L.biases; m.bias = L.bias;
    m.nsub = swiglu[i] ? 2 : 1;
    m.out_eff = L.out / m.nsub;
    m.in = L.in;
    m.row_bytes = L.bits ? L.in * L.bits / 8 : L.in * (int)dtype_size(L.sdt);
    m.srow_bytes = L.bits ? (L.in / L.group) * (int)dtype_size(L.sdt) : 0;
    m.sdt = L.sdt; m.group = L.bits ? L.group : 1;
    if (m.group & (m.group - 1)) return;  // power-of-two groups only
    m.group_shift = 0;
    while ((1 << m.group_shift) < m.group) ++m.group_shift;
    int u = 1;
    while (u <= 16 && ((u * m.row_bytes) % 16 != 0 || (u * m.srow_bytes) % 16 != 0)) u <<= 1;
    if (u > 16 || m.out_eff % u != 0) return;
    m.unit = u;
    m.norm_w = norms[i].norm_w; m.q_norm = norms[i].q_norm; m.k_norm = norms[i].k_norm;
    m.in_kind = phase[i].in_kind; m.pass = phase[i].pass; m.epi = phase[i].epi; m.out_sel = phase[i].out_sel; m.flags = phase[i].flags;
    m.layer = phase[i].layer; m.uidx = phase[i].unit; m.tkind = phase[i].tkind;
    need_slot = std::max(need_slot, u * m.nsub * (m.row_bytes + 2 * m.srow_bytes));
    kmax = std::max(kmax, L.in);
    lin.push_back(m);
  }
  const int G_tk = T.heads / T.kv_heads, G_cp = P.heads / P.kv_heads;
  auto g_ok = [](int g) { return g == 1 || g == 2 || g == 4; };
  if (!g_ok(G_tk) || !g_ok(G_cp) || T.head_dim != 128 || P.head_dim != 128) return;
  if (T.heads % T.kv_heads || P.heads % P.kv_heads) return;
  if (cfg_.vocab_size > 4096 || cfg_.cp.vocab_size > 4096) return;
  if (T.hidden % 4 || P.hidden % 4 || T.inter % 4 || P.inter % 4) return;
  int slot_bytes = 32 * 1024;
  while (slot_bytes < need_slot) slot_bytes += 8 * 1024;
  const int nchunk = (kmax + kc - 1) / kc;
  const int hmax = std::max(T.hidden, P.hidden);
  auto up = [](int v, int a) { return (v + a - 1) / a * a; };
  // Handles that can hold >= 2 utterances (packed formats) run the tensor-core GEMV: kMegaMaxSlots utterances per launch;
  // single-utterance handles keep the fp32 SIMT GEMV (lower latency at one row).
  const bool mma = (fmt == 0 || fmt == 1);
  int gmin = 1 << 30, gmax = 0, max_tiles = 0;
  for (const MegaLinear& m : lin) {
    gmin = std::min(gmin, m.group); gmax = std::max(gmax, m.group);
    const int rch = (slot_bytes / (m.nsub * (m.row_bytes + 2 * m.srow_bytes))) / m.unit * m.unit;
    max_tiles = std::max(max_tiles, ((rch + 15) / 16) * m.nsub);
  }
  if (mma && (gmin < 32 || gmax > 128 || kmax % 32 != 0)) return;
  const int budget = 226 * 1024;
  int NS = 0, MT = 0, n_ring = 0, xs_bytes = 0, xsum_bytes = 0, xraw_bytes = 0, red_bytes = 0, hl_bytes = 0, rope_bytes = 0, part_bytes = 0;
  const int scratch = (4096 + 64 + 4096) * 4;  // sampler: ids + reductions + staged logits of the CTA's slot; attention tiles fit too
  for (int cand : {kMegaMaxSlots, 1}) {
    if (cand > 1 && (!mma || opt_.max_batch < 2)) continue;
    NS = cand; MT = 2 * NS;
    const bool tc = mma && cand > 1;  // one utterance: fp32 SIMT GEMV; several: tensor-core GEMV with hi/lo fp16 columns (8 columns)
    xs_bytes = up(std::max(tc ? 8 * (kmax * 2 + 64) : MT * nchunk * kc * 4, scratch), 128);
    xsum_bytes = up(tc ? MT * (kmax / gmin) * 4 : MT * nchunk * 32 * 4, 128);
    xraw_bytes = up(MT * hmax * 4, 128);
    red_bytes = up(MT * 16 * 4, 128);
    hl_bytes = up(NS * hmax * 4, 128);
    rope_bytes = up(NS * 128 * 2 * 4, 128);
    part_bytes = tc ? up(std::max(32, max_tiles) * 128 * 4, 128) : 0;
    const int fixed = xs_bytes + xsum_bytes + xraw_bytes + red_bytes + 256 + 512 + hl_bytes + rope_bytes + part_bytes + 128;
    n_ring = std::min(8, (budget - fixed) / slot_bytes);
    if (n_ring >= 3 || (cand == 1 && n_ring >= 2)) break;
    NS = 0;
  }
  if (NS == 0) return;
  mega_.max_slots = NS;
  MegaParams& p = mega_.p;
  p.slot_bytes = slot_bytes; p.n_ring = n_ring;
  p.off_xs = n_ring * slot_bytes;
  p.off_xsum = p.off_xs + xs_bytes;
  p.off_xraw = p.off_xsum + xsum_bytes;
  p.off_red = p.off_xraw + xraw_bytes;
  p.off_bar = p.off_red + red_bytes;
  p.off_dsc = p.off_bar + 256;
  static_assert(2 * sizeof(MegaLinear) <= 512, "descriptor slots");
  p.off_hl = p.off_dsc + 512;
  p.raw_ld = hmax;
  p.off_rope = p.off_hl + hl_bytes;
  p.off_part = p.off_rope + rope_bytes;
  p.xh_stride = kmax + 32;
  mega_.smem = (size_t)p.off_part + part_bytes + 128;
  mega_.fmt = fmt; mega_.G_cp = G_cp; mega_.G_tk = G_tk;
  int dev = 0, sms = 0, coop = 0;
  Q3_CUDA(cudaGetDevice(&dev));
  Q3_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  Q3_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
  if (!coop || sms < 1) return;
  init_mega_kernels();
  if (mega_max_blocks_per_sm(fmt, mega_.max_slots, mega_.smem) < 1) return;
  // every CTA must own rows of every linear: the tagged exchange relies on all CTAs writing in every linear phase
  int min_units = 1 << 30;
  for (const MegaLinear& m : lin) min_units = std::min(min_units, m.out_eff / m.unit);
  mega_.grid = std::min(sms, min_units);
  if (mega_.grid < 1 || opt_.kv_capacity > 4 * 128) return;
  for (MegaLinear& m : lin) {
    const int U = m.out_eff / m.unit;
    m.ubase = U / mega_.grid; m.urem = U % mega_.grid;
    m.rch = (slot_bytes / (m.nsub * (m.row_bytes + 2 * m.srow_bytes))) / m.unit * m.unit;
  }
  // device tables
  MegaLinear* d_lin = arena_.alloc_n<MegaLinear>(lin.size());
  Q3_CUDA(cudaMemcpy(d_lin, lin.data(), sizeof(MegaLinear) * lin.size(), cudaMemcpyHostToDevice));
  auto stack_of = [&](const StackWeights& S, const float* inv_freq, float* k, float* v, size_t slot_stride, size_t layer_stride, int cap, int nsplit) {
    MegaStack s{};
    s.hidden = S.hidden; s.layers = S.layers; s.heads = S.heads; s.kv_heads = S.kv_heads; s.inter = S.inter; s.eps = S.eps;
    s.final_norm = S.final_norm; s.inv_freq = inv_freq; s.k = k; s.v = v;
    s.slot_stride = slot_stride; s.layer_stride = layer_stride; s.capacity = cap; s.nsplit = nsplit;
    return s;
  };
  const int nsplit_tk = 4;  // key splits of a talker attention item (each <= 128 keys: kv_capacity <= 512)
  p.lin = d_lin; p.n_lin = (int)lin.size();
  p.cp = stack_of(P, d_cp_inv_freq_, cp_k_, cp_v_, cpkv_slot_stride_, cpkv_layer_stride_, kCpCapacity, 1);
  if (kv_f16_) return;  // the persistent frame kernel reads fp32 rings (it only ever runs on handles of <= 2 slots, which keep them)
  p.tk = stack_of(T, d_inv_freq_, (float*)kcache_, (float*)vcache_, kv_slot_stride_, kv_layer_stride_, opt_.kv_capacity, nsplit_tk);
  p.has_mtp = w_.has_mtp ? 1 : 0; p.H = cfg_.hidden_size; p.Hcp = cfg_.cp.hidden_size; p.V = cfg_.vocab_size; p.Vc = cfg_.cp.vocab_size;
  p.codec = w_.codec_embedding; p.cp_emb = d_cp_emb_;
  p.st = d_state_; p.cur_codes = d_cur_codes_; p.frames = d_frames_; p.forced = d_forced_; p.max_frames = opt_.max_frames;
  p.sets = d_sets_; p.set_words = set_words_;
  p.trailing = d_trailing_; p.max_trailing = opt_.max_trailing; p.tts_pad = d_tts_ + (size_t)2 * cfg_.hidden_size;
  p.hlast = d_hlast_; p.logits0 = d_logits0_; p.cplogits = d_cplogits_;
  p.part_stride = up(std::max(T.heads, P.heads) * 130, 4);
  p.ld_x = up(hmax, 4);
  p.ld_qkv = up(std::max((T.heads + 2 * T.kv_heads) * 128, (P.heads + 2 * P.kv_heads) * 128), 4);
  p.ld_act = up(std::max(T.inter, P.inter), 4);
  p.ld_logit = up(std::max(cfg_.vocab_size, cfg_.cp.vocab_size), 4);
  const size_t n_x = (size_t)MT * p.ld_x, n_qkv = (size_t)MT * p.ld_qkv, n_part = (size_t)MT * nsplit_tk * p.part_stride;
  const size_t n_act = (size_t)MT * p.ld_act, n_logit = (size_t)NS * p.ld_logit, n_msg = (size_t)2 * 16 * kMegaMaxSlots * 4;
  p.ex_bytes = (n_x + n_qkv + n_part + n_act + n_logit + n_msg) * sizeof(unsigned long long);
  unsigned long long* ex = arena_.alloc_n<unsigned long long>(n_x + n_qkv + n_part + n_act + n_logit + n_msg);
  p.ex_base = ex;
  p.ex_x = ex; ex += n_x;
  p.ex_qkv = ex; ex += n_qkv;
  p.ex_part = ex; ex += n_part;
  p.ex_act = ex; ex += n_act;
  p.ex_logit = ex; ex += n_logit;
  p.ex_msg = ex;
  p.window = 192;  // maxKVCacheWindow (Model/Qwen3Layers.swift:108)
  p.eos_id = cfg_.codec_eos_token_id; p.pad_id = cfg_.codec_pad_id;
  if (getenv("Q3TTS_MEGA_TRACE")) {  // diagnostics: per-phase cycle stamps of one launch (frame_kernel.cu), dumped by run_frames
    p.trace_stride = 8 * 1024 * 8;
    p.trace = arena_.alloc_n<long long>((size_t)2 * p.trace_stride);
  }
  mega_.ok = true;
}

TalkerEngine::~TalkerEngine() {
  drop_graphs();
  if (h_stage_) cudaFreeHost(h_stage_);
  if (h_state_) cudaFreeHost(h_state_);
  if (ev_a_) cudaEventDestroy(ev_a_);
  if (ev_b_) cudaEventDestroy(ev_b_);
  if (d_dump0_) cudaFree(d_dump0_);
  if (d_dumpcp_) cudaFree(d_dumpcp_);
}

void TalkerEngine::drop_graphs() {
  for (auto& g : graphs_)
    if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
  graphs_.clear();
}

// fp16 dense copy of one Linear for the tcgen05 path.  Packed leaves go through the bit-exact dequant kernel (deq16 =
// round(fp32(scale) * q + fp32(bias))), float leaves are rounded to fp16.
// `fold` (fp32 [in], may be null): the RMSNorm weight that precedes this linear, multiplied into its columns in fp32 before the
// fp16 rounding (Model/Qwen3Layers.swift:8-26, 246-257: norm(x) * w feeds exactly this linear), so the norm's row factor can be
// applied to the accumulator instead (TcGemm::ss_in).
TcLinear TalkerEngine::make_tc(const Linear& L, bool interleave_halves, const float* fold) {
  const LaunchCtx c{stream_, nullptr};
  TcLinear t;
  t.out = L.out; t.in = L.in; t.bias = L.bias;
  if (L.bits) { t.qw = L.qw; t.qscales = L.scales; t.qbiases = L.biases; t.qbits = L.bits; t.qgroup = L.group; t.qsdt = L.sdt; t.fold = fold; t.halves = interleave_halves; }
  __half* dst = (__half*)shared_->arena.alloc((size_t)L.out * L.in * 2);
  if (L.bits && fold) {
    float* tmp = nullptr;
    Q3_CUDA(cudaMalloc(&tmp, (size_t)L.out * L.in * 4));
    launch_dequantize(c, L.qw, L.scales, L.biases, L.sdt, L.out, L.in, L.group, L.bits, Q3TTS_F32, tmp);
    launch_weight_to_f16(c, tmp, Q3TTS_F32, L.out, L.in, interleave_halves, dst, fold);
    Q3_CUDA(cudaStreamSynchronize(stream_));
    cudaFree(tmp);
  } else if (L.bits) {
    if (!interleave_halves) {
      launch_dequantize(c, L.qw, L.scales, L.biases, L.sdt, L.out, L.in, L.group, L.bits, Q3TTS_F16, dst);
    } else {
      __half* tmp = nullptr;
      Q3_CUDA(cudaMalloc(&tmp, (size_t)L.out * L.in * 2));
      launch_dequantize(c, L.qw, L.scales, L.biases, L.sdt, L.out, L.in, L.group, L.bits, Q3TTS_F16, tmp);
      launch_weight_to_f16(c, tmp, Q3TTS_F16, L.out, L.in, true, dst);
      Q3_CUDA(cudaStreamSynchronize(stream_));
      cudaFree(tmp);
    }
  } else {
    launch_weight_to_f16(c, L.w, L.sdt, L.out, L.in, interleave_halves, dst, fold);
  }
  t.w = dst;
  return t;
}

void TalkerEngine::build_tc_weights() {
  auto ok = [](const Linear& L) { return L.in % 8 == 0 && L.out % 32 == 0; };
  bool all = ok(w_.fc1) && ok(w_.fc2) && ok(w_.codec_head) && (!w_.has_mtp || ok(w_.small_to_mtp));
  for (StackWeights* S : {&w_.talker, &w_.cp})
    for (auto& l : S->layer) all = all && ok(l.qkv) && ok(l.o) && ok(l.gate_up) && ok(l.down) && (l.gate_up.out / 2) % 16 == 0;
  for (auto& h : w_.lm_head) all = all && ok(h);
  if (!all) return;  // shapes outside the tcgen05 path: every row count stays on the SIMT kernels
  for (StackWeights* S : {&w_.talker, &w_.cp}) {
    S->tc.resize(S->layers);
    for (int l = 0; l < S->layers; ++l) {
      S->tc[l].qkv = make_tc(S->layer[l].qkv, false, S->layer[l].in_norm);         // input_layernorm folded in
      S->tc[l].o = make_tc(S->layer[l].o, false);
      S->tc[l].gate_up_il = make_tc(S->layer[l].gate_up, true, S->layer[l].post_norm);  // post_attention_layernorm folded in
      S->tc[l].down = make_tc(S->layer[l].down, false);
    }
  }
  w_.fc1_tc = make_tc(w_.fc1, false);
  w_.fc2_tc = make_tc(w_.fc2, false);
  w_.codec_head_tc = make_tc(w_.codec_head, false);
  for (auto& h : w_.lm_head) w_.lm_head_tc.push_back(make_tc(h, false, w_.cp.final_norm));  // code predictor's final norm folded in
  if (w_.has_mtp) w_.small_to_mtp_tc = make_tc(w_.small_to_mtp, false);
  Q3_CUDA(cudaStreamSynchronize(stream_));
  w_.has_tc = true;
}

// decode-step GEMMs read the checkpoint's packed bytes when the leaf is quantised (a9: dequant fused into the GEMM)
void TalkerEngine::attach_packed(TcGemm& g, const TcLinear& L) const {
  if (!L.qbits || !packed_gemm_) return;
  g.q_w = L.qw; g.q_scales = L.qscales; g.q_biases = L.qbiases; g.q_fold = L.fold;
  g.q_bits = L.qbits; g.q_group = L.qgroup; g.q_sdt = L.qsdt; g.q_halves = L.halves ? 1 : 0;
}

void TalkerEngine::linear_tc(const TcLinear& L, const void* x16, int m, float* out32, int ld32, void* out16, int ld16, const float* res,
                             int act, int swiglu, bool row_count_invariant) {
  TcGemm g;
  if (row_count_invariant) { g.allow_skinny = 0; g.k_rotate = 0; }  // prefill: see forward_stack
  g.a = (const __half*)x16; g.w = (const __half*)L.w; g.Bt = 1; g.T = m; g.cin = L.in; g.N = L.out; g.ntap = 1; g.dil = 1;
  g.bias = L.bias; g.res = res; g.ld_res = ld32; g.act = act; g.swiglu = swiglu;
  g.out32 = out32; g.ld32 = ld32; g.out16 = (__half*)out16; g.ld16 = ld16;
  if (!row_count_invariant) attach_packed(g, L);
  launch_tc_gemm(ctx(), g);
}

// Qwen3DecoderLayer x layers (Model/Qwen3Layers.swift:242-262; Qwen3CodePredictor.swift:118-138): 6 launches per layer.
void TalkerEngine::forward_stack(const StackWeights& S, float* x, int m, const int* row_slot, const int* row_pos,
                                 const int* win_start, const float* inv_freq, void* kbase, void* vbase, int kv_f16, size_t slot_stride,
                                 size_t layer_stride, int capacity, bool one_row_per_slot, bool decode_step, bool x16_ready) {
  const size_t kv_elem = kv_f16 ? 2 : 4;
  const LaunchCtx c = ctx();
  const int qkv_ld = (S.heads + 2 * S.kv_heads) * 128, attn_ld = S.heads * 128;
  if ((decode_step ? step_tc_ : use_tc(m)) && !S.tc.empty()) {
    // tcgen05 path (rows >= tc_min_rows_): fp16 operands, fp32 accumulate, fp32 residual stream.  RMSNorm is folded around the
    // contractions: its WEIGHT lives in the fp16 copies of qkv / gate|up (make_tc), its per-row factor is applied to the
    // accumulator, and the activation operand is d_h16_ = fp16(x / 16) of the un-normalised stream.
    //   <= 128 rows (decode steps): 5 launches per layer -- the o / down GEMMs write fp16(x / 16) next to x, the qkv / gate|up
    //      GEMMs derive the row factors from their own operand (TcGemm::rms_in);
    //   prefill (any row count): the same arithmetic on the 128-row-tile kernel with precomputed factors (launch_row_scale).
    //      Every output row of either kernel depends only on its own input row and on the weight shape, so a request's
    //      result does not depend on which other requests shared its launches (tests: batched == single, bit for bit).
    const bool fused = decode_step && m <= 128;
    // decode step with two rows per slot and no window = code-predictor pass 0: rows (2s, 2s+1) at positions (0, 1)
    const bool pass0_pairs = decode_step && !one_row_per_slot && win_start == nullptr && row_pos == d_cp_pos2_ && (m % 2) == 0;
    const float inv16 = 1.0f / kX16Div;
    auto consumer = [&](const TcLinear& L, float* out32, int ld32, void* out16, int ld16, int swiglu) {
      TcGemm g;
      g.a = (const __half*)d_h16_; g.w = (const __half*)L.w; g.Bt = 1; g.T = m; g.cin = L.in; g.N = L.out;
      g.bias = L.bias; g.swiglu = swiglu; g.out32 = out32; g.ld32 = ld32; g.out16 = (__half*)out16; g.ld16 = ld16;
      g.rms_eps = S.eps; g.in_scale = inv16; g.allow_skinny = fused; g.k_rotate = fused;
      if (fused) {
        g.rms_in = 1;
        attach_packed(g, L);
      } else {
        launch_row_scale(c, (const __half*)d_h16_, m, S.hidden, inv16, S.eps, d_rs_);
        g.row_scale = d_rs_;
      }
      launch_tc_gemm(c, g);
    };
    auto producer = [&](const TcLinear& L, const void* a16) {  // x += a . W^T, and refresh d_h16_ = fp16(x / 16)
      TcGemm g;
      g.a = (const __half*)a16; g.w = (const __half*)L.w; g.Bt = 1; g.T = m; g.cin = L.in; g.N = L.out;
      g.bias = L.bias; g.res = x; g.ld_res = S.hidden; g.out32 = x; g.ld32 = S.hidden; g.allow_skinny = fused; g.k_rotate = fused;
      if (fused) {
        g.out16 = (__half*)d_h16_; g.ld16 = S.hidden; g.out16_scale = inv16;
        attach_packed(g, L);
        launch_tc_gemm(c, g);
      } else {
        launch_tc_gemm(c, g);
        launch_scale_to_f16(c, x, (size_t)m * S.hidden, inv16, (__half*)d_h16_);
      }
    };
    if (!x16_ready) launch_scale_to_f16(c, x, (size_t)m * S.hidden, inv16, (__half*)d_h16_);  // else the producer of x wrote it
    for (int l = 0; l < S.layers; ++l) {
      const LayerWeights& L = S.layer[l];
      const LayerTc& Tc = S.tc[l];
      KVLayout kv;
      kv.k = static_cast<char*>(kbase) + l * layer_stride * kv_elem; kv.v = static_cast<char*>(vbase) + l * layer_stride * kv_elem;
      kv.slot_stride = slot_stride; kv.capacity = capacity; kv.f16 = kv_f16;
      consumer(Tc.qkv, d_qkv_, qkv_ld, nullptr, 0, 0);
      if (one_row_per_slot) {
        launch_rope_attention_f16(c, d_qkv_, qkv_ld, m, S.heads, S.kv_heads, L.q_norm, L.k_norm, S.eps, inv_freq, row_slot, row_pos, win_start, kv,
                                  (__half*)d_attn16_, attn_ld);
      } else if (pass0_pairs) {
        launch_cp_pass0_attention_f16(c, d_qkv_, qkv_ld, m / 2, S.heads, S.kv_heads, L.q_norm, L.k_norm, S.eps, inv_freq, kv, (__half*)d_attn16_, attn_ld);
      } else {
        launch_qk_norm_rope_append(c, d_qkv_, qkv_ld, m, S.heads, S.kv_heads, S.head_dim, L.q_norm, L.k_norm, S.eps, inv_freq, row_slot,
                                   row_pos, kv);
        launch_attention_f16(c, d_qkv_, qkv_ld, m, S.heads, S.kv_heads, S.head_dim, row_slot, row_pos, win_start, kv, (__half*)d_attn16_, attn_ld);
      }
      producer(Tc.o, d_attn16_);
      consumer(Tc.gate_up_il, nullptr, 0, d_act16_, S.inter, 1);
      producer(Tc.down, d_act16_);
    }
    return;
  }
  for (int l = 0; l < S.layers; ++l) {
    const LayerWeights& L = S.layer[l];
    KVLayout kv;
    kv.k = static_cast<char*>(kbase) + l * layer_stride * kv_elem; kv.v = static_cast<char*>(vbase) + l * layer_stride * kv_elem;
    kv.slot_stride = slot_stride; kv.capacity = capacity; kv.f16 = kv_f16;
    launch_linear(c, L.qkv, x, S.hidden, m, d_qkv_, qkv_ld, L.in_norm, S.eps, EPI_STORE);
    if (one_row_per_slot) {
      launch_rope_attention(c, d_qkv_, qkv_ld, m, S.heads, S.kv_heads, L.q_norm, L.k_norm, S.eps, inv_freq, row_slot, row_pos, win_start, kv,
                            d_attn_, attn_ld);
    } else {
      launch_qk_norm_rope_append(c, d_qkv_, qkv_ld, m, S.heads, S.kv_heads, S.head_dim, L.q_norm, L.k_norm, S.eps, inv_freq, row_slot,
                                 row_pos, kv);
      launch_attention(c, d_qkv_, qkv_ld, m, S.heads, S.kv_heads, S.head_dim, row_slot, row_pos, win_start, kv, d_attn_, attn_ld);
    }
    launch_linear(c, L.o, d_attn_, attn_ld, m, x, S.hidden, nullptr, 0.f, EPI_ADD);
    launch_linear(c, L.gate_up, x, S.hidden, m, d_act_, S.inter, L.post_norm, S.eps, EPI_SWIGLU);
    launch_linear(c, L.down, d_act_, S.inter, m, x, S.hidden, nullptr, 0.f, EPI_ADD);
  }
}

Admission TalkerEngine::admit(int slot, const q3tts_request& r) {
  std::vector<AdmitItem> items{{slot, &r}};
  std::vector<Admission> out;
  admit_batch(items, out);
  return out[0];
}

// Prompt assembly + prefill of several utterances at once (Model/Qwen3Talker.swift:344-462 for each): their prefill rows
// are concatenated into one [R, H] activation matrix so the 28-layer prefill is ONE pass of (tensor-core) GEMMs; rows carry
// (slot, position) so RoPE / KV append / causal attention stay per utterance.
void TalkerEngine::admit_batch(const std::vector<AdmitItem>& items, std::vector<Admission>& out) {
  const int H = cfg_.hidden_size, C = opt_.kv_capacity, F = opt_.max_frames, TH = cfg_.text_hidden_size;
  out.assign(items.size(), Admission{});
  std::vector<int> ids{cfg_.tts_bos_token_id, cfg_.tts_eos_token_id, cfg_.tts_pad_token_id};
  const int TP_BOS = 0, TP_EOS = 1, TP_PAD = 2;
  std::vector<int> desc, meta_slot, meta_pos;
  std::vector<float> spk_host;
  struct Plan { int slot, row0, P, tp_trailing, n_trailing; const q3tts_request* r; };
  std::vector<Plan> plans;
  auto check_text = [&](const int32_t* p, int n, const char* what) {
    for (int i = 0; i < n; ++i)
      Q3_CHECK(p[i] >= 0 && p[i] < cfg_.text_vocab_size, Q3TTS_ERR_INVALID_ARG, "%s id %d outside the text vocabulary", what, p[i]);
  };
  for (size_t it = 0; it < items.size(); ++it) {
    const int slot = items[it].slot;
    const q3tts_request& r = *items[it].req;
    Q3_CHECK(slot >= 0 && slot < opt_.max_batch, Q3TTS_ERR_INVALID_ARG, "slot %d out of range", slot);
    Q3_CHECK(r.text_ids != nullptr || r.n_text_ids == 0, Q3TTS_ERR_INVALID_ARG, "text_ids is NULL");
    if (r.n_text_ids < 9) {  // minTokens (Model/Qwen3Talker.swift:348-352)
      out[it].too_short = true;
      continue;
    }
    check_text(r.text_ids, r.n_text_ids, "text");
    const bool has_instruct = r.instruct_ids != nullptr && r.n_instruct_ids > 0;
    const bool use_icl = !has_instruct && r.ref_codes != nullptr && r.ref_text_ids != nullptr && r.n_ref_text_ids > 0;  // :338, 395
    if (has_instruct) check_text(r.instruct_ids, r.n_instruct_ids, "instruct");
    if (use_icl) check_text(r.ref_text_ids, r.n_ref_text_ids, "reference transcript");
    const bool spk_by_id = r.speaker_id >= 0;
    const bool spk_by_vec = !spk_by_id && r.speaker_embedding != nullptr;
    if (spk_by_id) Q3_CHECK(r.speaker_id < cfg_.vocab_size, Q3TTS_ERR_INVALID_ARG, "speaker_id %d outside codec vocabulary", r.speaker_id);
    if (spk_by_vec) Q3_CHECK(r.speaker_embedding_dim == H, Q3TTS_ERR_INVALID_ARG, "speaker embedding has %d dims, model hidden size is %d", r.speaker_embedding_dim, H);
    const int n_front_text = has_instruct ? r.n_instruct_ids : (use_icl ? r.n_ref_text_ids : 0);
    const int n_ref_audio = (use_icl && r.ref_frames > 0) ? r.ref_frames : 0;
    const int trailing_len = r.n_text_ids - 4 - 5;  // :426
    const int n_trailing = trailing_len > 0 ? trailing_len : 0;
    Q3_CHECK(n_trailing + 1 <= opt_.max_trailing, Q3TTS_ERR_CAPACITY, "text too long: %d trailing tokens > %d", n_trailing + 1, opt_.max_trailing);
    const int n_codec = 5 + ((spk_by_id || spk_by_vec) ? 1 : 0);
    const int P = n_front_text + n_ref_audio + 3 + (n_codec - 1) + 1;
    Q3_CHECK(P <= C - 16, Q3TTS_ERR_CAPACITY, "prefill of %d positions exceeds kv_capacity %d - 16; raise q3tts_options.kv_capacity", P, C);
    Q3_CHECK((int)ids.size() + n_front_text + 4 + n_trailing <= max_tp_rows_ && (int)meta_slot.size() + P <= max_rows_, Q3TTS_ERR_CAPACITY,
             "prompt batch too large for this handle");
    // text rows to project: [instruct | ref-text ..., role(3), first text, trailing ...]
    const int tp_front = (int)ids.size();
    for (int i = 0; i < n_front_text; ++i) ids.push_back(has_instruct ? r.instruct_ids[i] : r.ref_text_ids[i]);
    const int tp_role = (int)ids.size();
    for (int i = 0; i < 3; ++i) ids.push_back(r.text_ids[i]);
    const int tp_first = (int)ids.size();
    ids.push_back(r.text_ids[3]);
    const int tp_trailing = (int)ids.size();
    for (int i = 0; i < n_trailing; ++i) ids.push_back(r.text_ids[4 + i]);
    // prefill row descriptors (tp index, codec row, speaker-vector index + 1)
    int spk_ref = 0;
    if (spk_by_vec) {
      spk_host.insert(spk_host.end(), r.speaker_embedding, r.speaker_embedding + H);
      spk_ref = (int)(spk_host.size() / H);
    }
    const int row0 = (int)meta_slot.size();
    auto row = [&](int tp, int codec, int spk) {
      desc.push_back(tp); desc.push_back(codec); desc.push_back(spk);
      meta_slot.push_back(slot); meta_pos.push_back((int)meta_slot.size() - 1 - row0);
    };
    for (int i = 0; i < n_front_text; ++i) row(tp_front + i, -1, 0);
    for (int i = 0; i < n_ref_audio; ++i) {  // codec_embedding(refCodes[0]) — first codebook only (:402-403)
      const int code = r.ref_codes[i];
      Q3_CHECK(code >= 0 && code < cfg_.vocab_size, Q3TTS_ERR_INVALID_ARG, "reference code %d outside codec vocabulary", code);
      row(-1, code, 0);
    }
    for (int i = 0; i < 3; ++i) row(tp_role + i, -1, 0);
    // codecEmbed = [nothink, think_bos, think_eos, (speaker), pad, bos] (:360-379);
    // combined = [tts_pad x (n-2), tts_bos] + codecEmbed[0 ..< n-1] (:383-386)
    int codec_ids[6], codec_spk[6] = {0, 0, 0, 0, 0, 0};
    int k = 0;
    codec_ids[k++] = cfg_.codec_nothink_id; codec_ids[k++] = cfg_.codec_think_bos_id; codec_ids[k++] = cfg_.codec_think_eos_id;
    if (spk_by_id) codec_ids[k++] = r.speaker_id;
    else if (spk_by_vec) { codec_ids[k] = -1; codec_spk[k] = spk_ref; ++k; }
    codec_ids[k++] = cfg_.codec_pad_id; codec_ids[k++] = cfg_.codec_bos_id;
    for (int i = 0; i < n_codec - 1; ++i) row(i < n_codec - 2 ? TP_PAD : TP_BOS, codec_ids[i], codec_spk[i]);
    row(tp_first, codec_ids[n_codec - 1], 0);  // firstTextEmbed (:423)
    out[it].prefill_len = P;
    plans.push_back({slot, row0, P, tp_trailing, n_trailing, &r});
  }
  if (plans.empty()) return;
  const int n_tp = (int)ids.size(), R = (int)meta_slot.size();
  Q3_CHECK((int)(spk_host.size() / H) <= opt_.max_batch, Q3TTS_ERR_CAPACITY, "too many speaker embeddings in one admission batch");

  const LaunchCtx c = ctx();
  Q3_CUDA(cudaEventRecord(ev_a_, stream_));
  Q3_CUDA(cudaMemcpyAsync(d_ids_, ids.data(), sizeof(int) * n_tp, cudaMemcpyHostToDevice, stream_));
  Q3_CUDA(cudaMemcpyAsync(d_desc_, desc.data(), sizeof(int) * 3 * R, cudaMemcpyHostToDevice, stream_));
  Q3_CUDA(cudaMemcpyAsync(d_pf_slot_, meta_slot.data(), sizeof(int) * R, cudaMemcpyHostToDevice, stream_));
  Q3_CUDA(cudaMemcpyAsync(d_pf_pos_, meta_pos.data(), sizeof(int) * R, cudaMemcpyHostToDevice, stream_));
  if (!spk_host.empty()) Q3_CUDA(cudaMemcpyAsync(d_spk_, spk_host.data(), sizeof(float) * spk_host.size(), cudaMemcpyHostToDevice, stream_));
  // text_projection(text_embedding(ids)) (Model/Qwen3Talker.swift:103-106; Qwen3Layers.swift:276-279)
  if (use_tc(n_tp)) {
    launch_gather_rows_f16(c, w_.text_embedding, d_ids_, n_tp, (__half*)d_tpe16_, TH);
    linear_tc(w_.fc1_tc, d_tpe16_, n_tp, nullptr, 0, d_tph16_, TH, nullptr, TC_ACT_SILU, 0, true);
    linear_tc(w_.fc2_tc, d_tph16_, n_tp, d_tp_, H, nullptr, 0, nullptr, TC_ACT_NONE, 0, true);
  } else {
    launch_gather_rows(c, w_.text_embedding, d_ids_, n_tp, d_tpe_, TH, false);
    launch_linear(c, w_.fc1, d_tpe_, TH, n_tp, d_tph_, TH, nullptr, 0.f, EPI_SILU);
    launch_linear(c, w_.fc2, d_tph_, TH, n_tp, d_tp_, H, nullptr, 0.f, EPI_STORE);
  }
  launch_assemble_rows(c, d_tp_, H, w_.codec_embedding, d_spk_, d_desc_, R, d_x_);
  for (const Plan& p : plans) {  // trailingTextHidden = textproj(ids[4 ..< len-5]) ++ tts_eos (:426-433)
    float* tr = d_trailing_ + (size_t)p.slot * opt_.max_trailing * H;
    if (p.n_trailing > 0)
      Q3_CUDA(cudaMemcpyAsync(tr, d_tp_ + (size_t)p.tp_trailing * H, sizeof(float) * p.n_trailing * H, cudaMemcpyDeviceToDevice, stream_));
    Q3_CUDA(cudaMemcpyAsync(tr + (size_t)p.n_trailing * H, d_tp_ + (size_t)TP_EOS * H, sizeof(float) * H, cudaMemcpyDeviceToDevice, stream_));
  }
  // prefill: every row at its own (slot, position) (Model/Qwen3Talker.swift:437)
  forward_stack(w_.talker, d_x_, R, d_pf_slot_, d_pf_pos_, d_pf_win_, d_inv_freq_, kcache_, vcache_, kv_f16_, kv_slot_stride_, kv_layer_stride_, C, false, false, false);
  // final norm + codec_head on the last position only (the reference computes all, :449, and samples the last, :284-286)
  for (const Plan& p : plans) {
    launch_rmsnorm(c, d_x_ + (size_t)(p.row0 + p.P - 1) * H, H, 1, H, w_.talker.final_norm, w_.talker.eps, d_hlast_ + (size_t)p.slot * H, H);
    launch_linear(c, w_.codec_head, d_hlast_ + (size_t)p.slot * H, H, 1, d_logits0_ + (size_t)p.slot * cfg_.vocab_size, cfg_.vocab_size, nullptr, 0.f, EPI_STORE);
  }
  for (const Plan& p : plans) {
    const q3tts_request& r = *p.r;
    const int slot = p.slot;
    const bool forced = r.forced_codes != nullptr && r.n_forced_frames > 0;
    if (forced) {
      Q3_CHECK(r.n_forced_frames <= F, Q3TTS_ERR_CAPACITY, "n_forced_frames %d > max_frames %d", r.n_forced_frames, F);
      Q3_CUDA(cudaMemcpyAsync(d_forced_ + (size_t)slot * F * 16, r.forced_codes, sizeof(int) * 16 * r.n_forced_frames, cudaMemcpyHostToDevice, stream_));
    }
    int logits_cap = 0;
    if ((r.code0_logits_out != nullptr || r.cp_logits_out != nullptr) && r.logits_capacity_frames > 0) {
      Q3_CHECK(slot == 0 || !use_mega(opt_.max_batch), Q3TTS_ERR_INVALID_ARG, "logit dumps on a handle of <= 2 slots are only available for slot 0");
      Q3_CHECK(slot < 4096, Q3TTS_ERR_INVALID_ARG, "logit dumps are limited to slots < 4096");
      logits_cap = std::min(r.logits_capacity_frames, F);
      if (logits_cap > dump_cap_) {
        Q3_CUDA(cudaStreamSynchronize(stream_));
        if (d_dump0_) cudaFree(d_dump0_);
        if (d_dumpcp_) cudaFree(d_dumpcp_);
        Q3_CUDA(cudaMalloc(&d_dump0_, sizeof(float) * (size_t)logits_cap * cfg_.vocab_size));
        Q3_CUDA(cudaMalloc(&d_dumpcp_, sizeof(float) * (size_t)logits_cap * 15 * cfg_.cp.vocab_size));
        dump_cap_ = logits_cap;
        drop_graphs();  // dump pointers are baked into captured graphs
      }
      Q3_CUDA(cudaMemsetAsync(d_dump0_, 0, sizeof(float) * (size_t)logits_cap * cfg_.vocab_size, stream_));
      Q3_CUDA(cudaMemsetAsync(d_dumpcp_, 0, sizeof(float) * (size_t)logits_cap * 15 * cfg_.cp.vocab_size, stream_));
    }
    if (logits_cap > 0) { dump_slot_ = slot; dump_enabled_ = true; }
    else if (slot == dump_slot_) dump_enabled_ = false;
    SlotState s{};
    s.active = 1;
    s.pos = p.P;  // positionOffset = inputEmbeds.shape[1] (:438)
    s.total_text = p.n_trailing + 1;
    s.max_tokens = forced ? r.n_forced_frames : std::min(std::max(r.max_tokens, 0), F);
    s.n_forced = forced ? r.n_forced_frames : 0;
    s.stream_variant = r.stream_variant ? 1 : 0;
    s.top_k = r.top_k;
    s.logits_cap = logits_cap;
    s.temperature = r.temperature;
    s.top_p = (r.top_p > 0.f) ? r.top_p : 1.0f;
    s.rep_penalty = (r.repetition_penalty > 0.f) ? r.repetition_penalty : 1.0f;
    s.seed = r.seed;
    if (s.max_tokens <= 0) s.finished = 1;
    h_state_[slot] = s;
    Q3_CUDA(cudaMemsetAsync(d_sets_ + (size_t)slot * 16 * set_words_, 0, sizeof(unsigned) * 16 * set_words_, stream_));
  }
  Q3_CUDA(cudaStreamSynchronize(stream_));  // pinned h_state_ entries were written after earlier async reads completed
  for (const Plan& p : plans)
    Q3_CUDA(cudaMemcpyAsync(d_state_ + p.slot, h_state_ + p.slot, sizeof(SlotState), cudaMemcpyHostToDevice, stream_));
  Q3_CUDA(cudaEventRecord(ev_b_, stream_));
  Q3_CUDA(cudaStreamSynchronize(stream_));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ev_a_, ev_b_);
  last_prefill_ms += ms;
}

void TalkerEngine::release(int slot) {
  Q3_CUDA(cudaMemsetAsync(d_state_ + slot, 0, sizeof(SlotState), stream_));
}

// One 12.5 Hz frame for slots [0, n_slots): the loop body of Model/Qwen3Talker.swift:464-562 with every decision on device.
void TalkerEngine::issue_frame(int n_slots) {
  step_tc_ = use_tc_step(n_slots);  // one decision per frame step (by utterances, not by the rows of each launch)
  const LaunchCtx c = ctx();
  const int H = cfg_.hidden_size, Hcp = cfg_.cp.hidden_size, V = cfg_.vocab_size, Vc = cfg_.cp.vocab_size;
  const int B = opt_.max_batch, F = opt_.max_frames;
  SamplerParams p{};
  p.vocab = V; p.group = 0; p.codec_vocab = V; p.eos_id = cfg_.codec_eos_token_id; p.pad_id = cfg_.codec_pad_id;
  p.groups = 16; p.set_words = set_words_;
  float* dump0 = dump_enabled_ ? d_dump0_ : nullptr;
  float* dumpcp = dump_enabled_ ? d_dumpcp_ : nullptr;
  // The sampler of group g also writes the code predictor's input rows of pass g (and, on the tensor-core path, their fp16
  // operand copy: fp16(x) for the small_to_mtp GEMM, fp16(x / 16) when the rows enter the stack directly).
  const bool x16_direct = step_tc_ && !w_.has_mtp;
  auto next_input = [&](int mode) {
    NextInput ni;
    ni.mode = mode; ni.H = H; ni.h_last = d_hlast_; ni.codec = w_.codec_embedding; ni.cp_emb = d_cp_emb_; ni.y32 = d_cpin_;
    if (step_tc_) { ni.y16 = (__half*)d_h16_; ni.y16_scale = w_.has_mtp ? 1.0f : 1.0f / kX16Div; }
    return ni;
  };
  launch_sample(c, d_logits0_, V, n_slots, d_state_, p, d_sets_, d_cur_codes_, d_forced_, F, dump0, V, 0, dump_slot_, next_input(1));
  for (int g = 0; g < 15; ++g) {  // code predictor, strictly sequential (:501-523)
    const int m = g == 0 ? 2 * n_slots : n_slots;
    float* x = d_cpin_;
    if (w_.has_mtp) {  // small_to_mtp_projection (Qwen3CodePredictor.swift:183-185)
      if (step_tc_) {
        linear_tc(w_.small_to_mtp_tc, d_h16_, m, d_cpx_, Hcp, nullptr, 0, nullptr, TC_ACT_NONE, 0);
      } else {
        launch_linear(c, w_.small_to_mtp, d_cpin_, H, m, d_cpx_, Hcp, nullptr, 0.f, EPI_STORE);
      }
      x = d_cpx_;
    }
    forward_stack(w_.cp, x, m, g == 0 ? d_cp_slot2_ : d_iota_, g == 0 ? d_cp_pos2_ : d_cp_pos_ + (size_t)g * B, nullptr,
                  d_cp_inv_freq_, cp_k_, cp_v_, 0, cpkv_slot_stride_, cpkv_layer_stride_, kCpCapacity, g != 0, true, x16_direct);
    // norm + lm_head[g] on the last position of each slot (Qwen3CodePredictor.swift:207-212)
    if (step_tc_ && g != 0 && n_slots <= 128) {
      // the last layer's down GEMM left fp16(x / 16) in d_h16_: lm_head (final norm folded in) takes it as is
      TcGemm hg;
      hg.a = (const __half*)d_h16_; hg.w = (const __half*)w_.lm_head_tc[g].w; hg.Bt = 1; hg.T = n_slots; hg.cin = Hcp; hg.N = Vc;
      hg.bias = w_.lm_head_tc[g].bias; hg.out32 = d_cplogits_; hg.ld32 = Vc;
      hg.rms_in = 1; hg.rms_eps = w_.cp.eps; hg.in_scale = 1.0f / kX16Div;
      attach_packed(hg, w_.lm_head_tc[g]);
      launch_tc_gemm(c, hg);
    } else if (step_tc_) {
      launch_rmsnorm_f16(c, g == 0 ? x + Hcp : x, g == 0 ? 2 * Hcp : Hcp, n_slots, Hcp, nullptr, w_.cp.eps, (__half*)d_h16_, Hcp);
      linear_tc(w_.lm_head_tc[g], d_h16_, n_slots, d_cplogits_, Vc, nullptr, 0, nullptr, TC_ACT_NONE, 0);
    } else if (g == 0) {
      launch_linear(c, w_.lm_head[0], x + Hcp, 2 * Hcp, n_slots, d_cplogits_, Vc, w_.cp.final_norm, w_.cp.eps, EPI_STORE);
    } else {
      launch_linear(c, w_.lm_head[g], x, Hcp, n_slots, d_cplogits_, Vc, w_.cp.final_norm, w_.cp.eps, EPI_STORE);
    }
    SamplerParams pg = p;
    pg.vocab = Vc; pg.group = g + 1;
    launch_sample(c, d_cplogits_, Vc, n_slots, d_state_, pg, d_sets_, d_cur_codes_, d_forced_, F, dumpcp, 15 * Vc, g * Vc, dump_slot_,
                  g < 14 ? next_input(2) : NextInput());
  }
  launch_frame_finalize(c, n_slots, d_state_, d_cur_codes_, d_frames_, F, d_sets_, set_words_, d_trailing_, opt_.max_trailing,
                        d_tts_ + (size_t)2 * H, w_.codec_embedding, d_cp_emb_, H, d_xstep_, step_tc_ ? (__half*)d_h16_ : nullptr, 1.0f / kX16Div);
  launch_step_rows(c, n_slots, d_state_, d_step_slot_, d_step_pos_, d_win_);
  forward_stack(w_.talker, d_xstep_, n_slots, d_step_slot_, d_step_pos_, d_win_, d_inv_freq_, kcache_, vcache_, kv_f16_, kv_slot_stride_,
                kv_layer_stride_, opt_.kv_capacity, true, true, step_tc_);
  launch_rmsnorm(c, d_xstep_, H, n_slots, H, w_.talker.final_norm, w_.talker.eps, d_hlast_, H);
  if (step_tc_) {
    launch_f32_to_f16(c, d_hlast_, (size_t)n_slots * H, (__half*)d_h16_);
    linear_tc(w_.codec_head_tc, d_h16_, n_slots, d_logits0_, V, nullptr, 0, nullptr, TC_ACT_NONE, 0);
  } else {
    launch_linear(c, w_.codec_head, d_hlast_, H, n_slots, d_logits0_, V, nullptr, 0.f, EPI_STORE);
  }
  launch_step_advance(c, n_slots, d_state_, 192);  // maxKVCacheWindow (Model/Qwen3Layers.swift:108)
}

void TalkerEngine::run_frames(int n_slots, int n) {
  if (n <= 0 || n_slots <= 0) return;
  if (!opt_.use_cuda_graph) {
    for (int i = 0; i < n; ++i) issue_frame(n_slots);
    return;
  }
  if (use_mega(n_slots)) {  // handles of <= 2 slots: one persistent cooperative launch for all n frames
    if (mega_.p.trace) Q3_CUDA(cudaMemsetAsync(mega_.p.trace, 0, sizeof(long long) * 2 * mega_.p.trace_stride, stream_));
    launch_frame_megakernel(ctx(), mega_, n_slots, n, dump_enabled_ ? d_dump0_ : nullptr, dump_enabled_ ? d_dumpcp_ : nullptr);
    ++mega_launches;
    if (mega_.p.trace) {
      std::vector<long long> t((size_t)2 * mega_.p.trace_stride);
      Q3_CUDA(cudaMemcpyAsync(t.data(), mega_.p.trace, sizeof(long long) * t.size(), cudaMemcpyDeviceToHost, stream_));
      Q3_CUDA(cudaStreamSynchronize(stream_));
      if (FILE* f = fopen(getenv("Q3TTS_MEGA_TRACE"), "wb")) { fwrite(t.data(), sizeof(long long), t.size(), f); fclose(f); }
    }
    return;
  }
  const long long key = (long long)n_slots * 8192 + (dump_enabled_ ? 1 + dump_slot_ : 0);
  auto it = graphs_.find(key);
  if (it == graphs_.end()) {
    cudaGraph_t g = nullptr;
    if (counter_) { counter_->capturing = true; counter_->captured = 0; }
    Q3_CUDA(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal));
    try {
      issue_frame(n_slots);
    } catch (...) {
      cudaStreamEndCapture(stream_, &g);
      if (g) cudaGraphDestroy(g);
      if (counter_) counter_->capturing = false;
      throw;
    }
    cudaError_t e = cudaStreamEndCapture(stream_, &g);
    if (counter_) counter_->capturing = false;
    if (e != cudaSuccess) fail(Q3TTS_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
    Graph gr;
    gr.nodes = counter_ ? counter_->captured : 0;
    e = cudaGraphInstantiate(&gr.exec, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) fail(Q3TTS_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
    it = graphs_.emplace(key, gr).first;
  }
  for (int i = 0; i < n; ++i) {
    Q3_CUDA(cudaGraphLaunch(it->second.exec, stream_));
    if (counter_) counter_->n += it->second.nodes;
    ++graph_replays;
  }
}

void TalkerEngine::fetch_states(int n_slots, std::vector<SlotState>& out) {
  Q3_CUDA(cudaMemcpyAsync(h_state_, d_state_, sizeof(SlotState) * n_slots, cudaMemcpyDeviceToHost, stream_));
  Q3_CUDA(cudaStreamSynchronize(stream_));
  out.assign(h_state_, h_state_ + n_slots);
}

void TalkerEngine::fetch_frames(int slot, int first, int count, int32_t* dst) {
  if (count <= 0) return;
  Q3_CUDA(cudaMemcpyAsync(dst, d_frames_ + ((size_t)slot * opt_.max_frames + first) * 16, sizeof(int) * 16 * count,
                          cudaMemcpyDeviceToHost, stream_));
  Q3_CUDA(cudaStreamSynchronize(stream_));
}

void TalkerEngine::fetch_logits(int frames, float* code0_out, float* cp_out) {
  frames = std::min(frames, dump_cap_);
  if (frames <= 0) return;
  if (code0_out) Q3_CUDA(cudaMemcpyAsync(code0_out, d_dump0_, sizeof(float) * (size_t)frames * cfg_.vocab_size, cudaMemcpyDeviceToHost, stream_));
  if (cp_out) Q3_CUDA(cudaMemcpyAsync(cp_out, d_dumpcp_, sizeof(float) * (size_t)frames * 15 * cfg_.cp.vocab_size, cudaMemcpyDeviceToHost, stream_));
  Q3_CUDA(cudaStreamSynchronize(stream_));
}

double TalkerEngine::profile_linears(int which, int m, int iters, int64_t& launches, int64_t& bytes_per_iter) {
  const StackWeights& S = which == 0 ? w_.talker : w_.cp;
  Q3_CHECK(m >= 1 && m <= max_rows_, Q3TTS_ERR_INVALID_ARG, "m %d out of range (1..%d)", m, max_rows_);
  const LaunchCtx c{stream_, nullptr};
  const int qkv_ld = (S.heads + 2 * S.kv_heads) * 128, attn_ld = S.heads * 128;
  Q3_CUDA(cudaMemsetAsync(d_x_, 0, sizeof(float) * (size_t)m * S.hidden, stream_));
  Q3_CUDA(cudaMemsetAsync(d_attn_, 0, sizeof(float) * (size_t)m * attn_ld, stream_));
  if (d_h16_) {
    Q3_CUDA(cudaMemsetAsync(d_h16_, 0, (size_t)m * S.hidden * 2, stream_));
    Q3_CUDA(cudaMemsetAsync(d_attn16_, 0, (size_t)m * attn_ld * 2, stream_));
    Q3_CUDA(cudaMemsetAsync(d_act16_, 0, (size_t)m * S.inter * 2, stream_));
  }
  launches = 0;
  bytes_per_iter = 0;
  const bool tc = handle_tc_ && m >= tc_min_rows_ && !S.tc.empty();  // the launches a decode step of this handle issues at m rows
  auto pass = [&](bool count) {
    for (int l = 0; l < S.layers; ++l) {
      const LayerWeights& L = S.layer[l];
      if (tc) {  // the launches batched decode actually issues (fp16 dense copies through tcgen05)
        const LayerTc& T = S.tc[l];
        linear_tc(T.qkv, d_h16_, m, d_qkv_, qkv_ld, nullptr, 0, nullptr, TC_ACT_NONE, 0);
        linear_tc(T.o, d_attn16_, m, d_x_, S.hidden, nullptr, 0, nullptr, TC_ACT_NONE, 0);
        linear_tc(T.gate_up_il, d_h16_, m, nullptr, 0, d_act16_, S.inter, nullptr, TC_ACT_NONE, 1);
        linear_tc(T.down, d_act16_, m, d_x_, S.hidden, nullptr, 0, nullptr, TC_ACT_NONE, 0);
        // algorithmic bytes (SURVEY.md §8d): the weights as the checkpoint stores them (packed codes + scales + biases)
        if (count) { launches += 4; bytes_per_iter += (int64_t)(L.qkv.weight_bytes() + L.o.weight_bytes() + L.gate_up.weight_bytes() + L.down.weight_bytes()); }
        continue;
      }
      launch_linear(c, L.qkv, d_x_, S.hidden, m, d_qkv_, qkv_ld, L.in_norm, S.eps, EPI_STORE);
      launch_linear(c, L.o, d_attn_, attn_ld, m, d_x_, S.hidden, nullptr, 0.f, EPI_ADD);
      launch_linear(c, L.gate_up, d_x_, S.hidden, m, d_act_, S.inter, L.post_norm, S.eps, EPI_SWIGLU);
      launch_linear(c, L.down, d_act_, S.inter, m, d_x_, S.hidden, nullptr, 0.f, EPI_ADD);
      if (count) { launches += 4; bytes_per_iter += (int64_t)(L.qkv.weight_bytes() + L.o.weight_bytes() + L.gate_up.weight_bytes() + L.down.weight_bytes()); }
    }
    if (tc) {
      const TcLinear& head = which == 0 ? w_.codec_head_tc : w_.lm_head_tc[0];
      linear_tc(head, d_h16_, m, which == 0 ? d_logits0_ : d_cplogits_, head.out, nullptr, 0, nullptr, TC_ACT_NONE, 0);
      if (count) { launches += 1; bytes_per_iter += (int64_t)(which == 0 ? w_.codec_head : w_.lm_head[0]).weight_bytes(); }
      return;
    }
    const Linear& head = which == 0 ? w_.codec_head : w_.lm_head[0];
    launch_linear(c, head, d_x_, S.hidden, m, which == 0 ? d_logits0_ : d_cplogits_, head.out, S.final_norm, S.eps, EPI_STORE);
    if (count) { launches += 1; bytes_per_iter += (int64_t)head.weight_bytes(); }
  };
  pass(true);  // warm-up (and the per-iteration accounting)
  // One pass as a CUDA graph, replayed `iters` times: the same submission path as the frame step (stream launches would add a
  // host-side tensor-map encode + launch per kernel and measure the CPU instead of the kernels).
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  Q3_CUDA(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal));
  pass(false);
  Q3_CUDA(cudaStreamEndCapture(stream_, &graph));
  Q3_CUDA(cudaGraphInstantiate(&exec, graph, 0));
  Q3_CUDA(cudaGraphLaunch(exec, stream_));
  Q3_CUDA(cudaEventRecord(ev_a_, stream_));
  for (int i = 0; i < iters; ++i) Q3_CUDA(cudaGraphLaunch(exec, stream_));
  Q3_CUDA(cudaEventRecord(ev_b_, stream_));
  Q3_CUDA(cudaStreamSynchronize(stream_));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ev_a_, ev_b_);
  cudaGraphExecDestroy(exec);
  cudaGraphDestroy(graph);
  launches *= iters;
  return ms;
}

int TalkerEngine::sample_probe(const float* logits, int vocab, float temperature, int top_k, float top_p, float rep_penalty,
                               const int32_t* token_set, int n_set, uint64_t seed, uint64_t counter) {
  Q3_CHECK(vocab > 0 && vocab <= 4096, Q3TTS_ERR_INVALID_ARG, "vocab %d out of range", vocab);
  std::vector<unsigned> bm(128, 0u);
  for (int i = 0; i < n_set; ++i)
    if (token_set[i] >= 0 && token_set[i] < vocab) bm[token_set[i] >> 5] |= 1u << (token_set[i] & 31);
  Q3_CUDA(cudaMemcpyAsync(d_probe_logits_, logits, sizeof(float) * vocab, cudaMemcpyHostToDevice, stream_));
  Q3_CUDA(cudaMemcpyAsync(d_probe_set_, bm.data(), sizeof(unsigned) * 128, cudaMemcpyHostToDevice, stream_));
  launch_sample_probe(ctx(), d_probe_logits_, vocab, cfg_.vocab_size, temperature, top_k, top_p > 0.f ? top_p : 1.f,
                      rep_penalty > 0.f ? rep_penalty : 1.f, n_set > 0 ? d_probe_set_ : nullptr, seed, counter, d_probe_out_);
  int id = -1;
  Q3_CUDA(cudaMemcpyAsync(&id, d_probe_out_, sizeof(int), cudaMemcpyDeviceToHost, stream_));
  Q3_CUDA(cudaStreamSynchronize(stream_));
  return id;
}

}  // namespace q3
