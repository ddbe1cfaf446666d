// Codec decoder: weight loading in the on-disk (PyTorch) layouts + the decode graph of decodeImpl.
#include <algorithm>
#include <cmath>

#include "codec_kernels.h"
#include "codec_unit.h"
#include "gemm_tc.h"

namespace q3 {

CodecConfig parse_codec_config(const Json& root) {
  // AudioDecoderConfig -> decoder_config -> toQwen3Config (Vocoder/AudioDecoder.swift:33-57, 137)
  CodecConfig c;
  const Json* d = root.find("decoder_config");
  if (d && d->type == Json::Obj) {
    c.upsample_rates = d->int_array_or("upsample_rates", c.upsample_rates);
    c.upsampling_ratios = d->int_array_or("upsampling_ratios", c.upsampling_ratios);
    c.decoder_dim = d->integer_or("decoder_dim", c.decoder_dim);
    c.codebook_size = d->integer_or("codebook_size", c.codebook_size);
    c.codebook_dim = d->integer_or("codebook_dim", c.codebook_dim);
    c.num_hidden_layers = d->integer_or("num_hidden_layers", c.num_hidden_layers);
    c.num_attention_heads = d->integer_or("num_attention_heads", c.num_attention_heads);
    c.num_key_value_heads = d->integer_or("num_key_value_heads", c.num_key_value_heads);
    c.hidden_size = d->integer_or("hidden_size", c.hidden_size);
    c.intermediate_size = d->integer_or("intermediate_size", c.intermediate_size);
    c.latent_dim = d->integer_or("latent_dim", c.latent_dim);
    c.num_quantizers = d->integer_or("num_quantizers", c.num_quantizers);
    c.num_semantic_quantizers = d->integer_or("num_semantic_quantizers", c.num_semantic_quantizers);
    c.head_dim = d->integer_or("head_dim", c.head_dim);
    c.rms_norm_eps = (float)d->number_or("rms_norm_eps", c.rms_norm_eps);
    c.rope_theta = (float)d->number_or("rope_theta", c.rope_theta);
    c.layer_scale_initial_scale = (float)d->number_or("layer_scale_initial_scale", c.layer_scale_initial_scale);
    c.max_position_embeddings = d->integer_or("max_position_embeddings", c.max_position_embeddings);
    c.attention_bias = d->bool_or("attention_bias", c.attention_bias);
    c.sliding_window = d->integer_or("sliding_window", c.sliding_window);  // parsed, never applied (quirk 7)
    Q3_CHECK(!d->has("quantization") || d->at("quantization").type == Json::Null, Q3TTS_ERR_BAD_CONFIG,
             "quantised speech_tokenizer checkpoints are out of scope (fp32/fp16/bf16 codec weights only)");
  }
  Q3_CHECK(c.head_dim == 64, Q3TTS_ERR_BAD_CONFIG, "codec attention kernels are specialised for head_dim 64 (got %d)", c.head_dim);
  Q3_CHECK(c.num_quantizers >= 1 && c.num_quantizers <= 64 && c.num_semantic_quantizers >= 1, Q3TTS_ERR_BAD_CONFIG, "bad quantizer counts");
  return c;
}

namespace {
const STensor& need(const std::map<std::string, STensor>& t, const std::string& k) {
  auto it = t.find(k);
  if (it == t.end()) fail(Q3TTS_ERR_DECODER_LOAD_FAILED, "speech_tokenizer/model.safetensors: missing tensor '%s'", k.c_str());
  return it->second;
}
}  // namespace

const __half* CodecDecoder::upload_f16(const std::vector<float>& h, int reps, size_t* rep_stride) {
  std::vector<__half> r(h.size());
  for (size_t i = 0; i < h.size(); ++i) r[i] = __float2half_rn(h[i]);
  const size_t stride = f16_rep_stride_bytes(r.size());  // bytes between copies
  __half* d = (__half*)arena_.alloc(stride * (size_t)reps);
  for (int i = 0; i < reps; ++i)
    Q3_CUDA(cudaMemcpy(reinterpret_cast<uint8_t*>(d) + (size_t)i * stride, r.data(), r.size() * sizeof(__half), cudaMemcpyHostToDevice));
  if (rep_stride) *rep_stride = stride / sizeof(__half);
  return d;
}

// copies of a conv weight for the L2-slice spreading described at ConvW::w16_reps: only matrices small enough that the re-reads matter
static int weight_reps(size_t halves) {
  constexpr int kReps = 8;
  return halves * 2 <= (size_t)(2u << 20) ? kReps : 1;
}

// A contraction can take the tcgen05 path when its K rows are 16-byte multiples (TMA) and N is a multiple of 32 (epilogue chunks).
void CodecDecoder::finish_weight(ConvW& w) {
  if (w.cin % 8 != 0 || w.n % 32 != 0) use_tc_ = false;
}

const float* CodecDecoder::load_vec(const std::map<std::string, STensor>& t, const std::string& key, int n) {
  std::vector<float> h = to_f32_host(need(t, key));
  Q3_CHECK((int)h.size() == n, Q3TTS_ERR_DECODER_LOAD_FAILED, "tensor '%s' has %zu elements, expected %d", key.c_str(), h.size(), n);
  float* d = arena_.alloc_n<float>(h.size());
  Q3_CUDA(cudaMemcpy(d, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
  return d;
}

// disk [C_out, C_in/g, K] -> device [K][C_out][C_in/g]   (the reference permutes to MLX [C_out, K, C_in], AudioDecoder.swift:276-277)
ConvW CodecDecoder::load_conv(const std::map<std::string, STensor>& t, const std::string& key, int cout, int cin, int k, int dil, bool bias) {
  const STensor& s = need(t, key + ".weight");
  Q3_CHECK(s.shape.size() == 3 && s.shape[0] == cout && s.shape[1] == cin && s.shape[2] == k, Q3TTS_ERR_DECODER_LOAD_FAILED,
           "conv weight '%s' has the wrong shape", key.c_str());
  std::vector<float> h = to_f32_host(s), r((size_t)k * cout * cin);
  for (int o = 0; o < cout; ++o)
    for (int i = 0; i < cin; ++i)
      for (int kk = 0; kk < k; ++kk) r[((size_t)kk * cout + o) * cin + i] = h[((size_t)o * cin + i) * k + kk];
  float* d = arena_.alloc_n<float>(r.size());
  Q3_CUDA(cudaMemcpy(d, r.data(), r.size() * 4, cudaMemcpyHostToDevice));
  ConvW w;
  w.w16_reps = weight_reps(r.size());
  w.w = d; w.w16 = upload_f16(r, w.w16_reps, &w.w16_rep_stride); w.ntap = k; w.dil = dil; w.cin = cin; w.n = cout;
  if (bias) w.bias = load_vec(t, key + ".bias", cout);
  finish_weight(w);
  return w;
}

// Transposed conv, disk [C_in, C_out, K] (AudioDecoder.swift:271-275), stride s, K in {s, 2s}, output trimmed to T*s
// (SpeechTokenizer.swift:174-204, 720-751).  Polyphase form: output sample t*s + j = x[t] . w[:,:,j] (+ x[t-1] . w[:,:,j+s] when
// K = 2s), i.e. a causal conv with K/s taps and n = s * C_out whose output [B, T, s*C_out] IS [B, T*s, C_out] in memory.
ConvW CodecDecoder::load_convT(const std::map<std::string, STensor>& t, const std::string& key, int cin, int cout, int k, int stride) {
  const STensor& s = need(t, key + ".weight");
  Q3_CHECK(s.shape.size() == 3 && s.shape[0] == cin && s.shape[1] == cout && s.shape[2] == k, Q3TTS_ERR_DECODER_LOAD_FAILED,
           "transposed-conv weight '%s' has the wrong shape", key.c_str());
  Q3_CHECK(k == stride || k == 2 * stride, Q3TTS_ERR_BAD_CONFIG, "transposed conv kernel %d / stride %d unsupported", k, stride);
  const int ntap = k / stride, n = stride * cout;
  std::vector<float> h = to_f32_host(s), r((size_t)ntap * n * cin);
  for (int tap = 0; tap < ntap; ++tap) {
    const int shift = ntap - 1 - tap;  // tap reads x[t - shift]
    for (int j = 0; j < stride; ++j)
      for (int o = 0; o < cout; ++o)
        for (int i = 0; i < cin; ++i)
          r[((size_t)tap * n + (size_t)j * cout + o) * cin + i] = h[((size_t)i * cout + o) * k + (j + shift * stride)];
  }
  float* d = arena_.alloc_n<float>(r.size());
  Q3_CUDA(cudaMemcpy(d, r.data(), r.size() * 4, cudaMemcpyHostToDevice));
  std::vector<float> hb = to_f32_host(need(t, key + ".bias")), rb((size_t)n);
  Q3_CHECK((int)hb.size() == cout, Q3TTS_ERR_DECODER_LOAD_FAILED, "bias of '%s' has the wrong size", key.c_str());
  for (int j = 0; j < stride; ++j)
    for (int o = 0; o < cout; ++o) rb[(size_t)j * cout + o] = hb[o];
  float* db = arena_.alloc_n<float>(rb.size());
  Q3_CUDA(cudaMemcpy(db, rb.data(), rb.size() * 4, cudaMemcpyHostToDevice));
  ConvW w;
  w.w16_reps = weight_reps(r.size());
  w.w = d; w.w16 = upload_f16(r, w.w16_reps, &w.w16_rep_stride); w.bias = db; w.ntap = ntap; w.dil = 1; w.cin = cin; w.n = n;
  finish_weight(w);
  return w;
}

ConvW CodecDecoder::load_linear(const std::map<std::string, STensor>& t, const std::string& key, int cout, int cin, bool bias) {
  const STensor& s = need(t, key + ".weight");
  Q3_CHECK(s.numel() == (int64_t)cout * cin, Q3TTS_ERR_DECODER_LOAD_FAILED, "linear weight '%s' has the wrong size", key.c_str());
  std::vector<float> h = to_f32_host(s);
  float* d = arena_.alloc_n<float>(h.size());
  Q3_CUDA(cudaMemcpy(d, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
  ConvW w;
  w.w = d; w.w16 = upload_f16(h); w.ntap = 1; w.dil = 1; w.cin = cin; w.n = cout;
  if (bias) w.bias = load_vec(t, key + ".bias", cout);
  finish_weight(w);
  return w;
}

SnakeW CodecDecoder::load_snake(const std::map<std::string, STensor>& t, const std::string& prefix, int ch) {
  std::vector<float> a = to_f32_host(need(t, prefix + ".alpha")), b = to_f32_host(need(t, prefix + ".beta"));
  Q3_CHECK((int)a.size() == ch && (int)b.size() == ch, Q3TTS_ERR_DECODER_LOAD_FAILED, "snake '%s' has the wrong size", prefix.c_str());
  for (int i = 0; i < ch; ++i) {
    a[i] = expf(a[i]);                    // exp(alpha)
    b[i] = 1.0f / (expf(b[i]) + 1e-9f);   // 1 / (exp(beta) + eps)   (SpeechTokenizer.swift:105-108)
  }
  float* da = arena_.alloc_n<float>(ch);
  float* db = arena_.alloc_n<float>(ch);
  Q3_CUDA(cudaMemcpy(da, a.data(), ch * 4, cudaMemcpyHostToDevice));
  Q3_CUDA(cudaMemcpy(db, b.data(), ch * 4, cudaMemcpyHostToDevice));
  SnakeW s;
  s.alpha = da; s.beta = db; s.ch = ch;
  return s;
}

CodecDecoder::CodecDecoder(const std::string& dir, cudaStream_t stream, LaunchCounter* counter, int pass_frames)
    : stream_(stream), counter_(counter), pass_frames_(pass_frames) {
  init_codec_kernels();
  init_tc_gemm();
  init_codec_unit();
  // config candidates (Qwen3TTSPipeline.swift:191-199)
  std::string cfg_path;
  for (const char* name : {"config.json", "configuration.json", "speech_tokenizer_config.json"}) {
    std::string p = dir + "/" + name;
    if (FILE* f = fopen(p.c_str(), "rb")) { fclose(f); cfg_path = p; break; }
  }
  if (cfg_path.empty()) fail(Q3TTS_ERR_FILE_NOT_FOUND, "Required file not found: speech_tokenizer/config.json");
  cfg_ = parse_codec_config(parse_json_file(cfg_path));
  up_ = cfg_.total_upsample();
  SafeTensors st(dir + "/model.safetensors", Q3TTS_ERR_DECODER_LOAD_FAILED);
  std::map<std::string, STensor> t;
  for (auto& kv : st.tensors()) {  // AudioDecoder.sanitize: strip "audio_decoder.", drop encoder.* (:204-216)
    std::string k = kv.first;
    if (k.rfind("audio_decoder.", 0) == 0) k = k.substr(14);
    if (k.rfind("encoder.", 0) == 0 || k.find(".encoder.") != std::string::npos) continue;
    t[k] = kv.second;
  }
  const CodecConfig& c = cfg_;
  const int D = c.codebook_dim / 2, L = c.latent_dim, hs = c.hidden_size, hd = c.head_dim;
  // codebook = embedding_sum / clip(cluster_usage, 1e-5, inf)[:, None]  in fp32 (AudioDecoder.swift:285-302)
  const int n_sem = c.num_semantic_quantizers;
  for (int q = 0; q < c.num_quantizers; ++q) {
    const std::string p = std::string("decoder.quantizer.") + (q < n_sem ? "rvq_first" : "rvq_rest") + ".vq.layers." +
                          std::to_string(q < n_sem ? q : q - n_sem) + "._codebook";
    std::vector<float> es = to_f32_host(need(t, p + ".embedding_sum")), cu = to_f32_host(need(t, p + ".cluster_usage"));
    Q3_CHECK((int)cu.size() == c.codebook_size && es.size() == (size_t)c.codebook_size * D, Q3TTS_ERR_DECODER_LOAD_FAILED,
             "codebook '%s' has the wrong shape", p.c_str());
    for (int i = 0; i < c.codebook_size; ++i) {
      const float u = cu[i] < 1e-5f ? 1e-5f : cu[i];
      for (int d = 0; d < D; ++d) es[(size_t)i * D + d] = es[(size_t)i * D + d] / u;
    }
    float* d = arena_.alloc_n<float>(es.size());
    Q3_CUDA(cudaMemcpy(d, es.data(), es.size() * 4, cudaMemcpyHostToDevice));
    codebooks_.push_back(d);
  }
  d_codebooks_ = (const float**)arena_.alloc(sizeof(float*) * codebooks_.size());
  Q3_CUDA(cudaMemcpy((void*)d_codebooks_, codebooks_.data(), sizeof(float*) * codebooks_.size(), cudaMemcpyHostToDevice));
  {  // [W_first | W_rest]: out = first . W1^T + rest . W2^T (SpeechTokenizer.swift:629-639, 684-691); 1x1 convs, no bias (:616-622)
    std::vector<float> w1 = to_f32_host(need(t, "decoder.quantizer.rvq_first.output_proj.weight"));
    std::vector<float> w2((size_t)c.codebook_dim * D, 0.f);
    if (c.num_quantizers > n_sem) w2 = to_f32_host(need(t, "decoder.quantizer.rvq_rest.output_proj.weight"));
    Q3_CHECK(w1.size() == (size_t)c.codebook_dim * D && w2.size() == w1.size(), Q3TTS_ERR_DECODER_LOAD_FAILED, "rvq output_proj has the wrong shape");
    std::vector<float> r((size_t)c.codebook_dim * 2 * D);
    for (int o = 0; o < c.codebook_dim; ++o)
      for (int i = 0; i < D; ++i) {
        r[(size_t)o * 2 * D + i] = w1[(size_t)o * D + i];
        r[(size_t)o * 2 * D + D + i] = w2[(size_t)o * D + i];
      }
    float* d = arena_.alloc_n<float>(r.size());
    Q3_CUDA(cudaMemcpy(d, r.data(), r.size() * 4, cudaMemcpyHostToDevice));
    rvq_proj_.w = d; rvq_proj_.w16 = upload_f16(r); rvq_proj_.ntap = 1; rvq_proj_.dil = 1; rvq_proj_.cin = 2 * D; rvq_proj_.n = c.codebook_dim;
    finish_weight(rvq_proj_);
  }
  pre_conv_ = load_conv(t, "decoder.pre_conv.conv", L, c.codebook_dim, 3, 1, true);
  const std::string pt = "decoder.pre_transformer";
  tr_in_ = load_linear(t, pt + ".input_proj", hs, L, true);
  tr_out_ = load_linear(t, pt + ".output_proj", L, hs, true);
  tr_norm_ = load_vec(t, pt + ".norm.weight", hs);
  const int qd = c.num_attention_heads * hd, kvd = c.num_key_value_heads * hd;
  auto concat_linear = [&](const std::vector<std::string>& keys, const std::vector<int>& outs, int cin, bool bias) {
    std::vector<float> w, b;
    int n = 0;
    for (size_t i = 0; i < keys.size(); ++i) {
      std::vector<float> h = to_f32_host(need(t, keys[i] + ".weight"));
      Q3_CHECK(h.size() == (size_t)outs[i] * cin, Q3TTS_ERR_DECODER_LOAD_FAILED, "linear '%s' has the wrong size", keys[i].c_str());
      w.insert(w.end(), h.begin(), h.end());
      if (bias) { std::vector<float> hb = to_f32_host(need(t, keys[i] + ".bias")); b.insert(b.end(), hb.begin(), hb.end()); }
      n += outs[i];
    }
    float* d = arena_.alloc_n<float>(w.size());
    Q3_CUDA(cudaMemcpy(d, w.data(), w.size() * 4, cudaMemcpyHostToDevice));
    ConvW cw;
    cw.w = d; cw.w16 = upload_f16(w); cw.ntap = 1; cw.dil = 1; cw.cin = cin; cw.n = n;
    if (bias) {
      float* db = arena_.alloc_n<float>(b.size());
      Q3_CUDA(cudaMemcpy(db, b.data(), b.size() * 4, cudaMemcpyHostToDevice));
      cw.bias = db;
    }
    finish_weight(cw);
    return cw;
  };
  // (gate_i, up_i) row-interleaved copy: the tcgen05 epilogue pairs adjacent columns for SwiGLU
  auto interleaved_gate_up = [&](const std::string& gate_key, const std::string& up_key, int inter, int cin) {
    std::vector<float> g = to_f32_host(need(t, gate_key + ".weight")), u = to_f32_host(need(t, up_key + ".weight")), r((size_t)2 * inter * cin);
    for (int i = 0; i < inter; ++i)
      for (int k = 0; k < cin; ++k) {
        r[((size_t)2 * i) * cin + k] = g[(size_t)i * cin + k];
        r[((size_t)2 * i + 1) * cin + k] = u[(size_t)i * cin + k];
      }
    ConvW cw;
    cw.w16 = upload_f16(r); cw.ntap = 1; cw.dil = 1; cw.cin = cin; cw.n = 2 * inter;
    finish_weight(cw);
    return cw;
  };
  for (int i = 0; i < c.num_hidden_layers; ++i) {
    const std::string lp = pt + ".layers." + std::to_string(i);
    TLayer l;
    l.qkv = concat_linear({lp + ".self_attn.q_proj", lp + ".self_attn.k_proj", lp + ".self_attn.v_proj"}, {qd, kvd, kvd}, hs, c.attention_bias);
    l.o = load_linear(t, lp + ".self_attn.o_proj", hs, qd, c.attention_bias);
    l.gate_up = concat_linear({lp + ".mlp.gate_proj", lp + ".mlp.up_proj"}, {c.intermediate_size, c.intermediate_size}, hs, false);
    l.gate_up_il = interleaved_gate_up(lp + ".mlp.gate_proj", lp + ".mlp.up_proj", c.intermediate_size, hs);
    l.down = load_linear(t, lp + ".mlp.down_proj", hs, c.intermediate_size, false);
    l.in_norm = load_vec(t, lp + ".input_layernorm.weight", hs);
    l.post_norm = load_vec(t, lp + ".post_attention_layernorm.weight", hs);
    l.attn_scale = load_vec(t, lp + ".self_attn_layer_scale.scale", hs);
    l.mlp_scale = load_vec(t, lp + ".mlp_layer_scale.scale", hs);
    tl_.push_back(l);
  }
  {  // inv_freq = 1 / pow(theta, (0,2,..)/dim) (SpeechTokenizer.swift:286-287)
    std::vector<float> f(hd / 2);
    for (int i = 0; i < hd / 2; ++i) f[i] = 1.0f / powf(c.rope_theta, (float)(2 * i) / (float)hd);
    float* d = arena_.alloc_n<float>(f.size());
    Q3_CUDA(cudaMemcpy(d, f.data(), f.size() * 4, cudaMemcpyHostToDevice));
    d_inv_freq_ = d;
  }
  for (size_t i = 0; i < c.upsampling_ratios.size(); ++i) {
    const int f = c.upsampling_ratios[i];
    const std::string p = "decoder.upsample." + std::to_string(i);
    Up u;
    u.factor = f;
    u.convT = load_convT(t, p + ".0.conv", L, L, f, f);
    {
      const STensor& s = need(t, p + ".1.dwconv.conv.weight");  // [C, 1, 7] -> [7][C]
      Q3_CHECK(s.numel() == (int64_t)L * 7, Q3TTS_ERR_DECODER_LOAD_FAILED, "dwconv weight has the wrong shape");
      std::vector<float> h = to_f32_host(s), r((size_t)7 * L);
      for (int ch = 0; ch < L; ++ch)
        for (int k = 0; k < 7; ++k) r[(size_t)k * L + ch] = h[(size_t)ch * 7 + k];
      float* d = arena_.alloc_n<float>(r.size());
      Q3_CUDA(cudaMemcpy(d, r.data(), r.size() * 4, cudaMemcpyHostToDevice));
      u.dw_w = d;
      u.dw_b = load_vec(t, p + ".1.dwconv.conv.bias", L);
    }
    u.ln_w = load_vec(t, p + ".1.norm.weight", L);
    u.ln_b = load_vec(t, p + ".1.norm.bias", L);
    u.pw1 = load_linear(t, p + ".1.pwconv1", 4 * L, L, true);
    u.pw2 = load_linear(t, p + ".1.pwconv2", L, 4 * L, true);
    u.gamma = load_vec(t, p + ".1.gamma", L);
    ups_.push_back(u);
  }
  init_conv_ = load_conv(t, "decoder.decoder.0.conv", c.decoder_dim, L, 7, 1, true);
  const int dils[3] = {1, 3, 9};
  for (size_t i = 0; i < c.upsample_rates.size(); ++i) {
    Block b;
    b.rate = c.upsample_rates[i];
    b.cin = c.decoder_dim >> i;
    b.cout = c.decoder_dim >> (i + 1);
    const std::string p = "decoder.decoder." + std::to_string(i + 1) + ".block";
    b.snake = load_snake(t, p + ".0", b.cin);
    b.convT = load_convT(t, p + ".1.conv", b.cin, b.cout, 2 * b.rate, b.rate);
    for (int j = 0; j < 3; ++j) {
      const std::string up = p + "." + std::to_string(j + 2);
      b.unit[j].act1 = load_snake(t, up + ".act1", b.cout);
      b.unit[j].conv1 = load_conv(t, up + ".conv1.conv", b.cout, b.cout, 7, dils[j], true);
      b.unit[j].act2 = load_snake(t, up + ".act2", b.cout);
      b.unit[j].conv2 = load_conv(t, up + ".conv2.conv", b.cout, b.cout, 1, 1, true);
    }
    blocks_.push_back(b);
  }
  const int n_out = (int)c.upsample_rates.size() + 1;
  out_ch_ = c.decoder_dim >> c.upsample_rates.size();
  out_snake_ = load_snake(t, "decoder.decoder." + std::to_string(n_out), out_ch_);
  {
    const STensor& s = need(t, "decoder.decoder." + std::to_string(n_out + 1) + ".conv.weight");  // [1, C, 7] -> [7][C]
    Q3_CHECK(s.numel() == (int64_t)out_ch_ * 7, Q3TTS_ERR_DECODER_LOAD_FAILED, "output conv has the wrong shape");
    std::vector<float> h = to_f32_host(s), r((size_t)7 * out_ch_);
    for (int ch = 0; ch < out_ch_; ++ch)
      for (int k = 0; k < 7; ++k) r[(size_t)k * out_ch_ + ch] = h[(size_t)ch * 7 + k];
    float* d = arena_.alloc_n<float>(r.size());
    Q3_CUDA(cudaMemcpy(d, r.data(), r.size() * 4, cudaMemcpyHostToDevice));
    out_w_ = d;
    out_b_ = load_vec(t, "decoder.decoder." + std::to_string(n_out + 1) + ".conv.bias", 1);
    // tensor-core form: the single output channel padded to a 32-column tile ([7][32][C] fp16, bias [32]); 31 columns of
    // zeros cost nothing next to streaming the activations once through the TMA pipeline instead of a SIMT smem loop
    std::vector<float> wp((size_t)7 * 32 * out_ch_, 0.f);
    for (int k = 0; k < 7; ++k)
      for (int ch = 0; ch < out_ch_; ++ch) wp[((size_t)k * 32) * out_ch_ + ch] = r[(size_t)k * out_ch_ + ch];
    std::vector<float> hb(32, 0.f);
    Q3_CUDA(cudaMemcpy(hb.data(), out_b_, 4, cudaMemcpyDeviceToHost));
    float* db = arena_.alloc_n<float>(32);
    Q3_CUDA(cudaMemcpy(db, hb.data(), 32 * 4, cudaMemcpyHostToDevice));
    out_tc_.w16_reps = weight_reps(wp.size());
    out_tc_.w16 = upload_f16(wp, out_tc_.w16_reps, &out_tc_.w16_rep_stride); out_tc_.bias = db; out_tc_.n = 32; out_tc_.cin = out_ch_; out_tc_.ntap = 7; out_tc_.dil = 1;
  }
  // algorithmic flops per 12.5 Hz frame (SURVEY.md §8d): 2 * MACs of every dense contraction
  int64_t fl = rvq_proj_.flops_per_row() + pre_conv_.flops_per_row() + tr_in_.flops_per_row() + tr_out_.flops_per_row();
  for (auto& l : tl_) fl += l.qkv.flops_per_row() + l.o.flops_per_row() + l.gate_up.flops_per_row() + l.down.flops_per_row();
  int64_t rate = 1;
  for (auto& u : ups_) {
    fl += rate * u.convT.flops_per_row();
    rate *= u.factor;
    fl += rate * (u.pw1.flops_per_row() + u.pw2.flops_per_row() + 2ll * 7 * L);
  }
  fl += rate * init_conv_.flops_per_row();
  for (auto& b : blocks_) {
    fl += rate * b.convT.flops_per_row();
    rate *= b.rate;
    for (int j = 0; j < 3; ++j) fl += rate * (b.unit[j].conv1.flops_per_row() + b.unit[j].conv2.flops_per_row());
  }
  fl += rate * 2ll * 7 * out_ch_;
  flops_per_frame_ = fl;
  if ((c.num_attention_heads * hd) % 8 != 0 || c.intermediate_size % 16 != 0 || hs % 8 != 0 || L % 8 != 0 || out_ch_ % 8 != 0) use_tc_ = false;
  if (const char* e = getenv("Q3TTS_CODEC_SIMT"))
    if (e[0] == '1') use_tc_ = false;  // A/B switch: run the fp32 SIMT pipeline
}

CodecDecoder::~CodecDecoder() {
  for (float*& p : ws_)
    if (p) { cudaFree(p); p = nullptr; }
  for (__half*& p : hs_)
    if (p) { cudaFree(p); p = nullptr; }
}

void CodecDecoder::ensure_workspace(int frames) {
  if (frames <= ws_frames_) return;
  // Regrowing frees and reallocates GBs behind a stream synchronize (measured: a 64 x 26-frame window after 63 x 26-frame ones
  // cost 390 ms): grow in steps of 512 frames so that batches of nearly equal size share one allocation.
  frames = std::min(std::max(pass_frames_, frames), (frames + 511) / 512 * 512);
  const CodecConfig& c = cfg_;
  // widest per-frame activation over all stages, in floats
  int64_t per = std::max<int64_t>({(int64_t)c.codebook_dim, (int64_t)c.latent_dim,
                                   (int64_t)(c.num_attention_heads + 2 * c.num_key_value_heads) * c.head_dim,
                                   (int64_t)2 * c.intermediate_size});
  int64_t rate = 1;
  for (auto& u : ups_) { rate *= u.factor; per = std::max(per, rate * 4 * c.latent_dim); }
  per = std::max(per, rate * c.decoder_dim);
  for (auto& b : blocks_) { per = std::max(per, rate * b.cin); rate *= b.rate; per = std::max(per, rate * b.cout); }
  Q3_CUDA(cudaStreamSynchronize(stream_));
  for (float*& p : ws_)
    if (p) { cudaFree(p); p = nullptr; }
  for (__half*& p : hs_)
    if (p) { cudaFree(p); p = nullptr; }
  ws_floats_ = (size_t)per * frames;
  ws_bytes_ = 0;
  const int n32 = use_tc_ ? 3 : 4;
  for (int i = 0; i < n32; ++i) { Q3_CUDA(cudaMalloc(&ws_[i], ws_floats_ * sizeof(float))); ws_bytes_ += ws_floats_ * sizeof(float); }
  if (use_tc_)
    for (__half*& p : hs_) { Q3_CUDA(cudaMalloc(&p, ws_floats_ * sizeof(__half))); ws_bytes_ += ws_floats_ * sizeof(__half); }
  ws_frames_ = frames;
}

void CodecDecoder::rvq_embed(const int32_t* d_codes, int B, int T, float* d_first, float* d_rest) {
  const int M = B * T, D = vq_dim();
  ensure_workspace(std::max(M, 1));
  launch_rvq_embed(ctx(), d_codes, d_codebooks_, cfg_.num_quantizers, cfg_.num_semantic_quantizers, D, cfg_.codebook_size, M, ws_[0]);
  Q3_CUDA(cudaMemcpy2DAsync(d_first, D * 4, ws_[0], 2 * D * 4, D * 4, M, cudaMemcpyDeviceToDevice, stream_));
  Q3_CUDA(cudaMemcpy2DAsync(d_rest, D * 4, ws_[0] + D, 2 * D * 4, D * 4, M, cudaMemcpyDeviceToDevice, stream_));
}

void CodecDecoder::decode_pass(const int32_t* d_codes, int B, int T, float* d_pcm) {
  if (use_tc_) decode_pass_tc(d_codes, B, T, d_pcm);
  else decode_pass_simt(d_codes, B, T, d_pcm);
}

// tcgen05 pipeline: every dense contraction is one launch of the implicit-GEMM kernel with its elementwise neighbours fused
// into the epilogue (bias, GELU, SwiGLU, LayerScale/gamma + residual, and the SnakeBeta of the NEXT layer applied to the fp16
// operand copy), fp32 residual streams, fp16 operands.
void CodecDecoder::decode_pass_tc(const int32_t* d_codes, int B, int T, float* d_pcm) {
  const CodecConfig& c = cfg_;
  const LaunchCtx lc = ctx();
  const int N = B * T;
  if (N <= 0) return;
  Q3_CHECK(N <= pass_frames_, Q3TTS_ERR_CAPACITY, "codec pass of %d frames exceeds pass capacity %d", N, pass_frames_);
  ensure_workspace(N);
  float *F0 = ws_[0], *F1 = ws_[1];
  __half *H0 = hs_[0], *H1 = hs_[1], *H2 = hs_[2];
  const int hs = c.hidden_size, nh = c.num_attention_heads, nkv = c.num_key_value_heads, hd = c.head_dim, I = c.intermediate_size, L = c.latent_dim;
  const int qkvw = (nh + 2 * nkv) * hd;
  auto gemm = [&](const ConvW& w, const __half* a, int Bt, int Tt) {
    TcGemm g;
    g.a = a; g.w = w.w16; g.Bt = Bt; g.T = Tt; g.cin = w.cin; g.N = w.n; g.ntap = w.ntap; g.dil = w.dil; g.bias = w.bias;
    g.w_reps = w.w16_reps; g.w_rep_stride = w.w16_rep_stride;
    return g;
  };
  auto with_snake = [](TcGemm& g, const SnakeW& s) { g.snake_ea = s.alpha; g.snake_ieb = s.beta; g.snake_ch = s.ch; };
  // quantizer.decode -> preConv (SpeechTokenizer.swift:922-923)
  launch_rvq_embed_f16(lc, d_codes, d_codebooks_, c.num_quantizers, c.num_semantic_quantizers, vq_dim(), c.codebook_size, N, H0);
  { TcGemm g = gemm(rvq_proj_, H0, B, T); g.out16 = H1; g.ld16 = c.codebook_dim; launch_tc_gemm(lc, g); }
  { TcGemm g = gemm(pre_conv_, H1, B, T); g.out16 = H0; g.ld16 = L; launch_tc_gemm(lc, g); }
  // preTransformer (:464-487): fp32 residual stream in F0
  { TcGemm g = gemm(tr_in_, H0, B, T); g.out32 = F0; g.ld32 = hs; launch_tc_gemm(lc, g); }
  for (auto& l : tl_) {
    launch_rmsnorm_f16(lc, F0, hs, N, hs, l.in_norm, c.rms_norm_eps, H0, hs);
    { TcGemm g = gemm(l.qkv, H0, B, T); g.out32 = F1; g.ld32 = qkvw; launch_tc_gemm(lc, g); }
    launch_codec_rope(lc, F1, qkvw, N, T, nh + nkv, d_inv_freq_);
    launch_codec_attention_f16(lc, F1, qkvw, B, T, nh, nkv, H1, nh * hd);
    { TcGemm g = gemm(l.o, H1, B, T); g.res = F0; g.ld_res = hs; g.scale = l.attn_scale; g.out32 = F0; g.ld32 = hs; launch_tc_gemm(lc, g); }
    launch_rmsnorm_f16(lc, F0, hs, N, hs, l.post_norm, c.rms_norm_eps, H0, hs);
    { TcGemm g = gemm(l.gate_up_il, H0, B, T); g.swiglu = 1; g.out16 = H1; g.ld16 = I; launch_tc_gemm(lc, g); }
    { TcGemm g = gemm(l.down, H1, B, T); g.res = F0; g.ld_res = hs; g.scale = l.mlp_scale; g.out32 = F0; g.ld32 = hs; launch_tc_gemm(lc, g); }
  }
  launch_rmsnorm_f16(lc, F0, hs, N, hs, tr_norm_, c.rms_norm_eps, H0, hs);
  { TcGemm g = gemm(tr_out_, H0, B, T); g.out16 = H1; g.ld16 = L; launch_tc_gemm(lc, g); }
  // upsample stages (:928-936): cur16 = H1
  int Tc = T;
  __half *cur = H1, *oa = H0, *ob = H2;
  for (auto& u : ups_) {
    { TcGemm g = gemm(u.convT, cur, B, Tc); g.out32 = F0; g.ld32 = u.convT.n; launch_tc_gemm(lc, g); }  // [B, Tc, f*L] == [B, Tc*f, L]
    Tc *= u.factor;
    const int M = B * Tc;
    launch_dwconv7(lc, F0, u.dw_w, u.dw_b, L, Tc, M, F1);
    launch_layernorm_f16(lc, F1, M, L, u.ln_w, u.ln_b, 1e-6f, oa);
    { TcGemm g = gemm(u.pw1, oa, B, Tc); g.act = TC_ACT_GELU; g.out16 = ob; g.ld16 = 4 * L; launch_tc_gemm(lc, g); }
    { TcGemm g = gemm(u.pw2, ob, B, Tc); g.res = F0; g.ld_res = L; g.scale = u.gamma; g.out16 = cur; g.ld16 = L; launch_tc_gemm(lc, g); }
  }
  // decoder[0] initial conv (:786-803) with block 0's SnakeBeta fused into its fp16 output
  {
    TcGemm g = gemm(init_conv_, cur, B, Tc);
    g.out16 = oa; g.ld16 = c.decoder_dim;
    if (!blocks_.empty()) with_snake(g, blocks_[0].snake); else with_snake(g, out_snake_);
    launch_tc_gemm(lc, g);
  }
  std::swap(cur, oa);  // cur = snake(init conv output)
  // The blocks' residual stream lives in fp16 (R0, carved out of the fp32 buffer F0): at 96-192 channels and 640-1920 samples per
  // frame it was the largest HBM stream of the pass (fp32: 1.2 GB read + 1.2 GB written per 1x1 conv at 64 x 26 frames); the
  // arithmetic stays fp32, one more fp16 rounding per unit.
  __half* R0 = reinterpret_cast<__half*>(F0);
  for (size_t bi = 0; bi < blocks_.size(); ++bi) {  // DecoderBlock (:753-784)
    Block& b = blocks_[bi];
    // polyphase transposed conv: y (residual stream) and snake_act1(y) (fp16 operand)
    {
      TcGemm g = gemm(b.convT, cur, B, Tc);
      g.outr16 = R0; g.allow_skinny = 0;
      g.ld32 = b.convT.n; g.out16 = oa; g.ld16 = b.convT.n; with_snake(g, b.unit[0].act1);
      launch_tc_gemm(lc, g);
    }
    Tc *= b.rate;
    for (int j = 0; j < 3; ++j) {  // DecoderResidualUnit (:696-718)
      const bool last = j == 2;
      const SnakeW& nxt = !last ? b.unit[j + 1].act1 : (bi + 1 < blocks_.size() ? blocks_[bi + 1].snake : out_snake_);
      {  // thin stages: the whole unit in one persistent kernel (codec_unit.cu), the intermediate never leaves the SM
        CodecUnit u;
        u.Bt = B; u.T = Tc; u.C = b.cout; u.dil = b.unit[j].conv1.dil;
        u.a = oa; u.w7 = b.unit[j].conv1.w16; u.b7 = b.unit[j].conv1.bias;
        u.snake2_ea = b.unit[j].act2.alpha; u.snake2_ieb = b.unit[j].act2.beta;
        u.w1 = b.unit[j].conv2.w16; u.b1 = b.unit[j].conv2.bias;
        u.w7_reps = b.unit[j].conv1.w16_reps; u.w7_rep_stride = b.unit[j].conv1.w16_rep_stride;
        u.w1_reps = b.unit[j].conv2.w16_reps; u.w1_rep_stride = b.unit[j].conv2.w16_rep_stride;
        u.res16 = R0; u.outr16 = last ? nullptr : R0;
        u.out16 = last ? cur : ob;  // never in place: other tiles still read their halo rows from `oa`
        u.next_ea = nxt.alpha; u.next_ieb = nxt.beta;
        if (b.unit[j].conv1.ntap == 7 && b.unit[j].conv2.ntap == 1 && b.unit[j].conv1.cin == b.cout && nxt.ch == b.cout && codec_unit_supported(u)) {
          launch_codec_unit(lc, u);
          if (!last) std::swap(oa, ob);
          continue;
        }
      }
      { TcGemm g = gemm(b.unit[j].conv1, oa, B, Tc); g.out16 = ob; g.ld16 = b.cout; with_snake(g, b.unit[j].act2); launch_tc_gemm(lc, g); }
      TcGemm g = gemm(b.unit[j].conv2, ob, B, Tc);
      g.ld_res = b.cout; g.ld32 = b.cout;
      g.res16 = R0; g.allow_skinny = 0;
      if (!last) g.outr16 = R0;
      g.out16 = last ? cur : oa; g.ld16 = b.cout;
      with_snake(g, nxt);
      launch_tc_gemm(lc, g);
    }
  }
  if (out_conv_stream_supported(out_ch_)) {
    launch_out_conv_stream_f16(lc, cur, out_w_, out_b_, out_ch_, B, Tc, d_pcm);  // HBM-bound: streamed once, fp32 weights in registers
  } else {
    TcGemm g = gemm(out_tc_, cur, B, Tc); g.pcm = d_pcm; launch_tc_gemm(lc, g);
  }
}

void CodecDecoder::decode_pass_simt(const int32_t* d_codes, int B, int T, float* d_pcm) {
  const CodecConfig& c = cfg_;
  const LaunchCtx lc = ctx();
  const int N = B * T;
  if (N <= 0) return;
  Q3_CHECK(N <= pass_frames_, Q3TTS_ERR_CAPACITY, "codec pass of %d frames exceeds pass capacity %d", N, pass_frames_);
  ensure_workspace(N);
  float *A = ws_[0], *Bf = ws_[1], *C = ws_[2], *D = ws_[3];
  const int hs = c.hidden_size, nh = c.num_attention_heads, nkv = c.num_key_value_heads, hd = c.head_dim, I = c.intermediate_size;
  const int qkvw = (nh + 2 * nkv) * hd;
  // quantizer.decode (SpeechTokenizer.swift:922) -> preConv (:923)
  launch_rvq_embed(lc, d_codes, d_codebooks_, c.num_quantizers, c.num_semantic_quantizers, vq_dim(), c.codebook_size, N, A);
  launch_conv_gemm(lc, A, rvq_proj_, Bf, nullptr, nullptr, N, T, CE_STORE);
  launch_conv_gemm(lc, Bf, pre_conv_, A, nullptr, nullptr, N, T, CE_STORE);
  // preTransformer (:464-487)
  launch_conv_gemm(lc, A, tr_in_, Bf, nullptr, nullptr, N, T, CE_STORE);
  for (auto& l : tl_) {
    launch_rmsnorm(lc, Bf, hs, N, hs, l.in_norm, c.rms_norm_eps, C, hs);
    launch_conv_gemm(lc, C, l.qkv, D, nullptr, nullptr, N, T, CE_STORE);
    launch_codec_rope(lc, D, qkvw, N, T, nh + nkv, d_inv_freq_);
    launch_codec_attention(lc, D, qkvw, B, T, nh, nkv, C, nh * hd);
    launch_conv_gemm(lc, C, l.o, Bf, Bf, l.attn_scale, N, T, CE_RES_SCALE);  // residual + LayerScale(attn) (:426)
    launch_rmsnorm(lc, Bf, hs, N, hs, l.post_norm, c.rms_norm_eps, C, hs);
    launch_conv_gemm(lc, C, l.gate_up, D, nullptr, nullptr, N, T, CE_STORE);
    launch_silu_mul(lc, D, N, I, C);
    launch_conv_gemm(lc, C, l.down, Bf, Bf, l.mlp_scale, N, T, CE_RES_SCALE);  // residual + LayerScale(mlp) (:431)
  }
  launch_rmsnorm(lc, Bf, hs, N, hs, tr_norm_, c.rms_norm_eps, C, hs);
  launch_conv_gemm(lc, C, tr_out_, A, nullptr, nullptr, N, T, CE_STORE);
  // upsample: [CausalTransposeConv1d k=f s=f, ConvNeXtBlock] x 2 (:928-936)
  int Tc = T;
  float *cur = A, *o1 = Bf, *o2 = C, *o3 = D;
  for (auto& u : ups_) {
    launch_conv_gemm(lc, cur, u.convT, o1, nullptr, nullptr, B * Tc, Tc, CE_STORE);
    Tc *= u.factor;
    const int M = B * Tc, L = c.latent_dim;
    launch_dwconv7(lc, o1, u.dw_w, u.dw_b, L, Tc, M, o2);
    launch_layernorm(lc, o2, M, L, u.ln_w, u.ln_b, 1e-6f, o3);
    launch_conv_gemm(lc, o3, u.pw1, o2, nullptr, nullptr, M, Tc, CE_GELU);
    launch_conv_gemm(lc, o2, u.pw2, o1, o1, u.gamma, M, Tc, CE_RES_SCALE);  // residual + gamma * h (:232-234)
    std::swap(cur, o1);
  }
  // decoder[0]: initial conv k7 (:786-803)
  launch_conv_gemm(lc, cur, init_conv_, o1, nullptr, nullptr, B * Tc, Tc, CE_STORE);
  std::swap(cur, o1);
  // DecoderBlocks (:753-784)
  for (auto& b : blocks_) {
    launch_snake(lc, cur, b.snake, (size_t)B * Tc, o1);
    launch_conv_gemm(lc, o1, b.convT, o2, nullptr, nullptr, B * Tc, Tc, CE_STORE);
    Tc *= b.rate;
    const size_t M = (size_t)B * Tc;
    for (int j = 0; j < 3; ++j) {  // DecoderResidualUnit (:696-718)
      launch_snake(lc, o2, b.unit[j].act1, M, o1);
      launch_conv_gemm(lc, o1, b.unit[j].conv1, o3, nullptr, nullptr, (int)M, Tc, CE_STORE);
      launch_snake(lc, o3, b.unit[j].act2, M, o1);
      launch_conv_gemm(lc, o1, b.unit[j].conv2, o2, o2, nullptr, (int)M, Tc, CE_RES_SCALE);
    }
    std::swap(cur, o2);
  }
  launch_snake(lc, cur, out_snake_, (size_t)B * Tc, o1);
  launch_out_conv(lc, o1, out_w_, out_b_, out_ch_, B, Tc, d_pcm);
}

}  // namespace q3
