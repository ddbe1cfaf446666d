// config.json + model.safetensors -> device weights.  Replaces Qwen3TTSConfig.init(from:) (Model/Qwen3Config.swift:208-253)
// and Qwen3Talker.load (Model/Qwen3Talker.swift:114-270).
#include <cuda_fp16.h>

#include "kernels.h"

namespace q3 {

float f16_to_f32(uint16_t v) {
  const uint32_t sign = (uint32_t)(v & 0x8000) << 16;
  uint32_t exp = (v >> 10) & 0x1F, man = v & 0x3FF, u;
  if (exp == 0) {
    if (man == 0) u = sign;
    else {
      int e = -1;
      do { man <<= 1; ++e; } while (!(man & 0x400));
      u = sign | ((uint32_t)(127 - 15 - e) << 23) | ((man & 0x3FF) << 13);
    }
  } else if (exp == 31) {
    u = sign | 0x7F800000u | (man << 13);
  } else {
    u = sign | ((exp + 112) << 23) | (man << 13);
  }
  float f;
  memcpy(&f, &u, 4);
  return f;
}

std::vector<float> to_f32_host(const STensor& t) {
  const int64_t n = t.numel();
  std::vector<float> r((size_t)n);
  if (t.dtype == "F32") {
    Q3_CHECK(t.nbytes == (size_t)n * 4, Q3TTS_ERR_BAD_WEIGHTS, "tensor byte size mismatch");
    memcpy(r.data(), t.data, (size_t)n * 4);
  } else if (t.dtype == "BF16" || t.dtype == "F16") {
    Q3_CHECK(t.nbytes == (size_t)n * 2, Q3TTS_ERR_BAD_WEIGHTS, "tensor byte size mismatch");
    const uint16_t* p = reinterpret_cast<const uint16_t*>(t.data);
    const bool bf = t.dtype == "BF16";
    for (int64_t i = 0; i < n; ++i) {
      uint16_t v;
      memcpy(&v, p + i, 2);
      r[(size_t)i] = bf ? bf16_to_f32(v) : f16_to_f32(v);
    }
  } else {
    fail(Q3TTS_ERR_BAD_WEIGHTS, "expected a float tensor, got %s", t.dtype.c_str());
  }
  return r;
}

TalkerConfig parse_talker_config(const Json& root) {
  TalkerConfig c;
  // nested `talker_config` wins for the model dims (Qwen3Config.swift:211-216)
  const Json& src = root.has("talker_config") ? root.at("talker_config") : root;
  c.hidden_size = src.integer("hidden_size");
  c.num_hidden_layers = src.integer("num_hidden_layers");
  c.vocab_size = src.integer("vocab_size");
  c.text_vocab_size = src.integer("text_vocab_size");
  c.text_hidden_size = src.integer_or("text_hidden_size", 2048);
  c.num_attention_heads = src.integer("num_attention_heads");
  c.num_key_value_heads = src.integer_or("num_key_value_heads", 8);
  c.head_dim = src.integer_or("head_dim", 128);
  c.intermediate_size = src.integer("intermediate_size");
  c.rms_norm_eps = (float)src.number("rms_norm_eps");
  c.max_position_embeddings = src.integer("max_position_embeddings");
  c.rope_theta = (float)src.number("rope_theta");
  c.tts_bos_token_id = root.integer_or("tts_bos_token_id", 151672);  // top level (:231-233)
  c.tts_eos_token_id = root.integer_or("tts_eos_token_id", 151673);
  c.tts_pad_token_id = root.integer_or("tts_pad_token_id", 151671);
  c.codec_bos_id = src.integer_or("codec_bos_id", 2149);
  c.codec_eos_token_id = src.integer_or("codec_eos_token_id", 2150);
  c.codec_pad_id = src.integer_or("codec_pad_id", 2148);
  c.codec_nothink_id = src.integer_or("codec_nothink_id", 2155);
  c.codec_think_bos_id = src.integer_or("codec_think_bos_id", 2156);
  c.codec_think_eos_id = src.integer_or("codec_think_eos_id", 2157);
  if (const Json* s = src.find("spk_id"))
    if (s->type == Json::Obj)
      for (auto& kv : s->obj)
        if (kv.second.type == Json::Num) c.spk_id.emplace_back(kv.first, (int)llround(kv.second.num));
  if (const Json* cp = src.find("code_predictor_config")) {
    if (cp->type == Json::Obj) {
      CPConfig d;
      c.cp.hidden_size = cp->integer_or("hidden_size", d.hidden_size);
      c.cp.num_hidden_layers = cp->integer_or("num_hidden_layers", d.num_hidden_layers);
      c.cp.num_attention_heads = cp->integer_or("num_attention_heads", d.num_attention_heads);
      c.cp.num_key_value_heads = cp->integer_or("num_key_value_heads", d.num_key_value_heads);
      c.cp.head_dim = cp->integer_or("head_dim", d.head_dim);
      c.cp.intermediate_size = cp->integer_or("intermediate_size", d.intermediate_size);
      c.cp.rms_norm_eps = (float)cp->number_or("rms_norm_eps", d.rms_norm_eps);
      c.cp.max_position_embeddings = cp->integer_or("max_position_embeddings", d.max_position_embeddings);
      c.cp.rope_theta = (float)cp->number_or("rope_theta", d.rope_theta);
      c.cp.vocab_size = cp->integer_or("vocab_size", d.vocab_size);
      c.cp.num_code_groups = cp->integer_or("num_code_groups", d.num_code_groups);
    }
  }
  if (const Json* rs = src.find("rope_scaling"))
    c.has_mrope = rs->type == Json::Obj && rs->has("mrope_section") && rs->at("mrope_section").type == Json::Arr;
  c.tts_model_type = root.string_or("tts_model_type", "");
  // MLX's `mode` of a quantisation block: "affine" (the default) or "mxfp4", whose bits and group_size default to 4 and 32 and must be
  // those.  nvfp4, mxfp8 and every other mode are refused here, before any weight is read (DESIGN.md §8).
  auto quant_block = [](const Json& q, const char* key, int& bits, int& group, int& mode) {
    const std::string m = q.string_or("mode", "affine");
    Q3_CHECK(m == "affine" || m == "mxfp4", Q3TTS_ERR_BAD_CONFIG, "%s.mode \"%s\" is not supported (affine or mxfp4)", key, m.c_str());
    mode = m == "mxfp4" ? QMODE_MXFP4 : QMODE_AFFINE;
    bits = q.integer_or("bits", mode == QMODE_MXFP4 ? 4 : 0);
    group = q.integer_or("group_size", mode == QMODE_MXFP4 ? 32 : 64);
    if (mode == QMODE_MXFP4)
      Q3_CHECK(bits == 4 && group == 32, Q3TTS_ERR_BAD_CONFIG, "%s: mode mxfp4 needs bits 4 and group_size 32 (got %d / %d)", key, bits, group);
  };
  if (const Json* q = root.find("quantization")) {
    if (q->type == Json::Obj) {
      c.has_quantization = true;
      quant_block(*q, "quantization", c.q_bits, c.q_group, c.q_mode);
    }
  }
  if (const Json* q = root.find("quantization_config")) {
    if (q->type == Json::Obj) {
      c.has_quantization_config = true;
      quant_block(*q, "quantization_config", c.qc_bits, c.qc_group, c.qc_mode);
    }
  }
  Q3_CHECK(c.hidden_size > 0 && c.num_hidden_layers > 0 && c.num_attention_heads > 0 && c.intermediate_size > 0,
           Q3TTS_ERR_BAD_CONFIG, "config.json: non-positive model dimension");
  Q3_CHECK(c.head_dim == 128 && c.cp.head_dim == 128, Q3TTS_ERR_BAD_CONFIG, "head_dim must be 128 (got %d / %d)", c.head_dim, c.cp.head_dim);
  Q3_CHECK(c.cp.num_code_groups == 16, Q3TTS_ERR_BAD_CONFIG, "num_code_groups must be 16 (got %d)", c.cp.num_code_groups);
  Q3_CHECK(c.num_attention_heads % c.num_key_value_heads == 0 && c.cp.num_attention_heads % c.cp.num_key_value_heads == 0,
           Q3TTS_ERR_BAD_CONFIG, "heads must be a multiple of kv heads");
  return c;
}

namespace {

struct Loader {
  const std::map<std::string, STensor>& t;  // remapped keys
  DeviceArena& arena;
  cudaStream_t stream;
  bool packed;          // use uint32 leaves as they are
  bool offline_dequant; // uint32 leaves -> fp16 dense at load (Qwen3Talker.swift:139-175)
  int bits, group;
  bool mxfp4;           // packed leaves are MLX mxfp4 (E2M1 codes + E8M0 scale bytes), converted to 8-bit affine groups of 32 at load
  // Qwen3TTSPipeline.applyMixedQuantization (:961-980): every dense Linear / Embedding is MLX-quantised at load, group 64, 6 bits for
  // embeddings, q/k/v projections and the heads, 4 bits for the rest; the codes live in an 8-bit container (launch_mlx_quantize)
  bool runtime_quant = false;
  int weight_dtype = -1;
  int ckpt_bits = 0;  // width of the packed leaves on disk (q3tts_info.checkpoint_quant_bits)
  static bool six_bit(const std::string& path) {
    std::string p = path;
    for (char& ch : p) ch = (char)tolower((unsigned char)ch);
    for (const char* k : {"embed", "qproj", "kproj", "vproj", "q_proj", "k_proj", "v_proj", "lm_head", "codec_head"})
      if (p.find(k) != std::string::npos) return true;
    return false;
  }

  const STensor& get(const std::string& k) const {
    auto it = t.find(k);
    if (it == t.end()) fail(Q3TTS_ERR_BAD_WEIGHTS, "model.safetensors: missing tensor '%s'", k.c_str());
    return it->second;
  }
  bool has(const std::string& k) const { return t.count(k) != 0; }

  void* upload(const void* src, size_t bytes) {
    void* d = arena.alloc(bytes);
    Q3_CUDA(cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, stream));
    return d;
  }
  const float* upload_f32(const std::string& k, int64_t expect) {
    const STensor& s = get(k);
    Q3_CHECK(s.numel() == expect, Q3TTS_ERR_BAD_WEIGHTS, "tensor '%s' has %lld elements, expected %lld", k.c_str(),
             (long long)s.numel(), (long long)expect);
    std::vector<float> h = to_f32_host(s);
    void* d = arena.alloc(h.size() * 4);
    Q3_CUDA(cudaMemcpyAsync(d, h.data(), h.size() * 4, cudaMemcpyHostToDevice, stream));
    Q3_CUDA(cudaStreamSynchronize(stream));  // h is a temporary
    return (const float*)d;
  }
  Embedding embedding(const std::string& k, int rows, int dim) {
    const STensor& s = get(k);
    Q3_CHECK(s.shape.size() == 2 && s.shape[0] == rows && s.shape[1] == dim, Q3TTS_ERR_BAD_WEIGHTS,
             "embedding '%s' has the wrong shape", k.c_str());
    Embedding e;
    e.rows = rows; e.dim = dim; e.dt = s.q3_dtype();
    const size_t bytes = (size_t)rows * dim * dtype_size(e.dt);
    Q3_CHECK(s.nbytes == bytes, Q3TTS_ERR_BAD_WEIGHTS, "embedding '%s' has the wrong byte size", k.c_str());
    void* d = upload(s.data, bytes);
    if (runtime_quant && dim % 64 == 0) {  // QuantizedEmbedding: rows dequantised to the storage dtype, 6 bits ("embed")
      LaunchCtx lc{stream, nullptr};
      void *sc = nullptr, *bi = nullptr;
      const size_t gb = (size_t)rows * (dim / 64) * dtype_size(e.dt);
      Q3_CUDA(cudaMalloc(&sc, gb)); Q3_CUDA(cudaMalloc(&bi, gb));
      launch_mlx_quantize(lc, d, e.dt, rows, dim, 6, nullptr, sc, bi, d);  // in place: a group is read completely before it is written
      Q3_CUDA(cudaStreamSynchronize(stream));
      cudaFree(sc); cudaFree(bi);
    }
    e.w = d;
    return e;
  }

  // The packed words (cbits-bit container), scales and biases of a linear in the arena -> L, used as they are (`quantization`), or
  // dequantised offline to fp16 (`quantization_config` only).
  void packed_result(Linear& L, int in, int cbits, int grp, int sdt, const uint32_t* qw, const void* sc, const void* bi) {
    if (weight_dtype < 0) weight_dtype = sdt;
    if (packed) {
      L.bits = cbits; L.group = grp; L.sdt = sdt; L.qw = qw; L.scales = sc; L.biases = bi;
    } else {
      // offline `dequantized(..., dtype: .float16)` (Qwen3Talker.swift:156-164) with the bit-exact kernel
      Q3_CHECK(offline_dequant, Q3TTS_ERR_BAD_CONFIG, "packed weights found but config.json has neither `quantization` nor `quantization_config`");
      __half* dense = (__half*)arena.alloc((size_t)L.out * in * 2);
      LaunchCtx lc{stream, nullptr};
      launch_dequantize(lc, qw, sc, bi, sdt, L.out, in, grp, cbits, Q3TTS_F16, dense);
      L.bits = 0; L.sdt = Q3TTS_F16; L.w = dense;
      weight_dtype = Q3TTS_F16;  // what the handle computes with after the load (q3tts_info.weight_dtype)
    }
  }

  // One or several reference leaves concatenated along `out` (q|k|v, gate|up).
  Linear linear(const std::vector<std::string>& prefixes, int in, const std::vector<int>& outs, bool with_bias) {
    Linear L;
    L.in = in;
    for (int o : outs) L.out += o;
    const STensor& w0 = get(prefixes[0] + ".weight");
    const bool is_packed = (w0.dtype == "U32" || w0.dtype == "I32") && has(prefixes[0] + ".scales");
    if (is_packed && mxfp4) {
      // .weight [out, in / 8] uint32 + .scales [out, in / 32] uint8, no .biases; the raw leaves go into temporaries and are converted
      // into the arena.  Every scale byte is checked here, so a leaf the container cannot hold fails q3tts_create.
      Q3_CHECK(in % 32 == 0, Q3TTS_ERR_BAD_WEIGHTS, "mxfp4 leaf '%s': in_features %d is not a multiple of 32", prefixes[0].c_str(), in);
      ckpt_bits = 4;
      const size_t row_words = (size_t)in / 8, row_groups = (size_t)in / 32;
      uint32_t* qw = (uint32_t*)arena.alloc((size_t)L.out * in);
      uint16_t* sc = (uint16_t*)arena.alloc((size_t)L.out * row_groups * 2);
      uint16_t* bi = (uint16_t*)arena.alloc((size_t)L.out * row_groups * 2);
      std::unique_ptr<void, cudaError_t (*)(void*)> raw_w(nullptr, cudaFree), raw_s(nullptr, cudaFree);
      void *pw = nullptr, *ps = nullptr;
      Q3_CUDA(cudaMalloc(&pw, (size_t)L.out * row_words * 4));
      raw_w.reset(pw);
      Q3_CUDA(cudaMalloc(&ps, (size_t)L.out * row_groups));
      raw_s.reset(ps);
      size_t r0 = 0;
      for (size_t i = 0; i < prefixes.size(); ++i) {
        const char* name = prefixes[i].c_str();
        const STensor& w = get(prefixes[i] + ".weight");
        const STensor& s = get(prefixes[i] + ".scales");
        Q3_CHECK(!has(prefixes[i] + ".biases"), Q3TTS_ERR_BAD_WEIGHTS, "mxfp4 leaf '%s' has a .biases tensor (an affine leaf?)", name);
        const size_t wbytes = (size_t)outs[i] * row_words * 4, sbytes = (size_t)outs[i] * row_groups;
        Q3_CHECK((w.dtype == "U32" || w.dtype == "I32") && w.shape.size() == 2 && w.shape[0] == outs[i] && (size_t)w.shape[1] == row_words &&
                     w.nbytes == wbytes,
                 Q3TTS_ERR_BAD_WEIGHTS, "mxfp4 weight '%s' must be uint32 [%d, %zu]", name, outs[i], row_words);
        Q3_CHECK(s.dtype == "U8" && s.shape.size() == 2 && s.shape[0] == outs[i] && (size_t)s.shape[1] == row_groups && s.nbytes == sbytes,
                 Q3TTS_ERR_BAD_WEIGHTS, "mxfp4 scales of '%s' must be uint8 [%d, %zu]", name, outs[i], row_groups);
        for (size_t k = 0; k < sbytes; ++k)
          Q3_CHECK(s.data[k] <= kMxfp4MaxScaleByte, Q3TTS_ERR_BAD_WEIGHTS,
                   "mxfp4 leaf '%s': scale byte %d at index %zu (2^%d) is beyond the 8-bit affine container (bytes 0..%d)", name, (int)s.data[k], k,
                   (int)s.data[k] - 127, kMxfp4MaxScaleByte);
        Q3_CUDA(cudaMemcpyAsync((uint32_t*)pw + r0 * row_words, w.data, wbytes, cudaMemcpyHostToDevice, stream));
        Q3_CUDA(cudaMemcpyAsync((uint8_t*)ps + r0 * row_groups, s.data, sbytes, cudaMemcpyHostToDevice, stream));
        r0 += outs[i];
      }
      LaunchCtx lc{stream, nullptr};
      launch_mxfp4_to_affine(lc, (const uint32_t*)pw, (const uint8_t*)ps, L.out, in, qw, sc, bi);
      Q3_CUDA(cudaStreamSynchronize(stream));  // the temporaries are freed when they leave scope
      packed_result(L, in, 8, 32, Q3TTS_BF16, qw, sc, bi);
    } else if (is_packed) {
      const int cbits = container_bits(bits);
      Q3_CHECK(cbits != 0, Q3TTS_ERR_BAD_CONFIG, "packed weights with bits=%d: MLX affine checkpoints of 2, 3, 4, 5, 6 or 8 bits are supported", bits);
      const bool widen = cbits != bits;  // 2/3/5/6-bit rows are re-laid into the 4/8-bit words every kernel reads
      if (widen) {
        Q3_CHECK(group == 32 || group == 64 || group == 128, Q3TTS_ERR_BAD_CONFIG, "%d-bit checkpoint with group_size %d: 32, 64 or 128 are supported",
                 bits, group);
        Q3_CHECK(in % group == 0 && in % 32 == 0, Q3TTS_ERR_BAD_CONFIG, "%d-bit checkpoint: in_features %d must be a multiple of 32 and of group_size %d",
                 bits, in, group);
      }
      Q3_CHECK(in % group == 0, Q3TTS_ERR_BAD_WEIGHTS, "in_features %d not a multiple of group_size %d", in, group);
      ckpt_bits = bits;
      const size_t row_words = (size_t)in * bits / 32, row_groups = (size_t)in / group;
      const int sdt = get(prefixes[0] + ".scales").q3_dtype();
      const size_t ssz = dtype_size(sdt);
      // the raw rows go straight into the arena, or into a temporary that is widened into it
      uint32_t* qw = (uint32_t*)arena.alloc((size_t)L.out * in * cbits / 8);
      uint32_t* raw = qw;
      std::unique_ptr<void, cudaError_t (*)(void*)> raw_tmp(nullptr, cudaFree);
      if (widen) {
        void* p = nullptr;
        Q3_CUDA(cudaMalloc(&p, (size_t)L.out * row_words * 4));
        raw_tmp.reset(p);
        raw = (uint32_t*)p;
      }
      char* sc = (char*)arena.alloc((size_t)L.out * row_groups * ssz);
      char* bi = (char*)arena.alloc((size_t)L.out * row_groups * ssz);
      size_t r0 = 0;
      for (size_t i = 0; i < prefixes.size(); ++i) {
        const STensor& w = get(prefixes[i] + ".weight");
        const STensor& s = get(prefixes[i] + ".scales");
        const STensor& b = get(prefixes[i] + ".biases");
        Q3_CHECK(w.shape.size() == 2 && w.shape[0] == outs[i] && (size_t)w.shape[1] == row_words, Q3TTS_ERR_BAD_WEIGHTS,
                 "packed weight '%s' has shape [%lld,%lld], expected [%d,%zu]", prefixes[i].c_str(), (long long)w.shape[0],
                 (long long)(w.shape.size() > 1 ? w.shape[1] : 0), outs[i], row_words);
        Q3_CHECK(s.q3_dtype() == sdt && b.q3_dtype() == sdt && (size_t)s.numel() == outs[i] * row_groups &&
                     (size_t)b.numel() == outs[i] * row_groups,
                 Q3TTS_ERR_BAD_WEIGHTS, "scales/biases of '%s' have the wrong shape or dtype", prefixes[i].c_str());
        // copy the byte counts the destination was sized for (SafeTensors already proved nbytes == numel * element size)
        const size_t wbytes = (size_t)outs[i] * row_words * 4, sbytes = (size_t)outs[i] * row_groups * ssz;
        Q3_CHECK((w.dtype == "U32" || w.dtype == "I32") && w.nbytes == wbytes && s.nbytes == sbytes && b.nbytes == sbytes, Q3TTS_ERR_BAD_WEIGHTS,
                 "packed leaf '%s' has the wrong dtype or byte size", prefixes[i].c_str());
        Q3_CUDA(cudaMemcpyAsync(raw + r0 * row_words, w.data, wbytes, cudaMemcpyHostToDevice, stream));
        Q3_CUDA(cudaMemcpyAsync(sc + r0 * row_groups * ssz, s.data, sbytes, cudaMemcpyHostToDevice, stream));
        Q3_CUDA(cudaMemcpyAsync(bi + r0 * row_groups * ssz, b.data, sbytes, cudaMemcpyHostToDevice, stream));
        r0 += outs[i];
      }
      if (widen) {
        LaunchCtx lc{stream, nullptr};
        launch_widen_bits(lc, raw, L.out, in, bits, qw);
        Q3_CUDA(cudaStreamSynchronize(stream));  // raw_tmp is freed when it leaves scope
      }
      packed_result(L, in, cbits, group, sdt, qw, sc, bi);
    } else {
      const int sdt = w0.q3_dtype();
      const size_t esz = dtype_size(sdt);
      char* w = (char*)arena.alloc((size_t)L.out * in * esz);
      size_t r0 = 0;
      for (size_t i = 0; i < prefixes.size(); ++i) {
        const STensor& s = get(prefixes[i] + ".weight");
        Q3_CHECK(s.q3_dtype() == sdt && s.shape.size() == 2 && s.shape[0] == outs[i] && s.shape[1] == in, Q3TTS_ERR_BAD_WEIGHTS,
                 "dense weight '%s' has the wrong shape or dtype", prefixes[i].c_str());
        Q3_CHECK(s.nbytes == (size_t)outs[i] * in * esz, Q3TTS_ERR_BAD_WEIGHTS, "dense weight '%s' has the wrong byte size", prefixes[i].c_str());
        Q3_CUDA(cudaMemcpyAsync(w + r0 * in * esz, s.data, (size_t)outs[i] * in * esz, cudaMemcpyHostToDevice, stream));
        r0 += outs[i];
      }
      if (weight_dtype < 0) weight_dtype = sdt;
      L.bits = 0; L.sdt = sdt; L.w = w;
    }
    if (runtime_quant && L.bits == 0 && in % 64 == 0) {  // the dense copy stays in the arena (load-time cost only; the kernels read the codes)
      const int qbits = six_bit(prefixes[0]) ? 6 : 4;
      const size_t gb = (size_t)L.out * (in / 64) * dtype_size(L.sdt);
      uint32_t* qw = (uint32_t*)arena.alloc((size_t)L.out * in);
      void* sc = arena.alloc(gb);
      void* bi = arena.alloc(gb);
      LaunchCtx lc{stream, nullptr};
      launch_mlx_quantize(lc, L.w, L.sdt, L.out, in, qbits, qw, sc, bi, nullptr);
      L.bits = 8; L.group = 64; L.qw = qw; L.scales = sc; L.biases = bi; L.w = nullptr;
    }
    if (with_bias) {
      std::vector<float> hb;
      for (size_t i = 0; i < prefixes.size(); ++i) {
        std::vector<float> p = to_f32_host(get(prefixes[i] + ".bias"));
        Q3_CHECK((int)p.size() == outs[i], Q3TTS_ERR_BAD_WEIGHTS, "bias of '%s' has the wrong size", prefixes[i].c_str());
        hb.insert(hb.end(), p.begin(), p.end());
      }
      void* d = arena.alloc(hb.size() * 4);
      Q3_CUDA(cudaMemcpyAsync(d, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice, stream));
      Q3_CUDA(cudaStreamSynchronize(stream));
      L.bias = (const float*)d;
    }
    return L;
  }

  void stack(const std::string& prefix, StackWeights& s) {
    s.layer.resize(s.layers);
    const int qd = s.heads * s.head_dim, kd = s.kv_heads * s.head_dim;
    for (int i = 0; i < s.layers; ++i) {
      const std::string p = prefix + "layers." + std::to_string(i);
      LayerWeights& l = s.layer[i];
      l.qkv = linear({p + ".self_attn.q_proj", p + ".self_attn.k_proj", p + ".self_attn.v_proj"}, s.hidden, {qd, kd, kd}, false);
      l.o = linear({p + ".self_attn.o_proj"}, qd, {s.hidden}, false);
      l.gate_up = linear({p + ".mlp.gate_proj", p + ".mlp.up_proj"}, s.hidden, {s.inter, s.inter}, false);
      l.down = linear({p + ".mlp.down_proj"}, s.inter, {s.hidden}, false);
      l.in_norm = upload_f32(p + ".input_layernorm.weight", s.hidden);
      l.post_norm = upload_f32(p + ".post_attention_layernorm.weight", s.hidden);
      l.q_norm = upload_f32(p + ".self_attn.q_norm.weight", s.head_dim);
      l.k_norm = upload_f32(p + ".self_attn.k_norm.weight", s.head_dim);
    }
    s.final_norm = upload_f32(prefix + "norm.weight", s.hidden);
  }
};

size_t stack_bytes(const StackWeights& s) {
  size_t b = 0;
  for (auto& l : s.layer) b += l.qkv.weight_bytes() + l.o.weight_bytes() + l.gate_up.weight_bytes() + l.down.weight_bytes();
  return b;
}

}  // namespace

void load_talker_weights(const std::string& model_dir, const TalkerConfig& cfg, DeviceArena& arena, cudaStream_t stream,
                         TalkerWeights& out, int& weight_dtype, int& eff_bits, int& eff_group, bool runtime_quantization) {
  SafeTensors st(model_dir + "/model.safetensors");
  // key remap (Qwen3Talker.swift:117-137): drop audio_decoder.*, strip "talker.", "code_predictor.model." ->
  // "code_predictor.", strip "model."
  std::map<std::string, STensor> t;
  for (auto& kv : st.tensors()) {
    std::string k = kv.first;
    if (k.rfind("audio_decoder.", 0) == 0) continue;
    if (k.rfind("talker.", 0) == 0) k = k.substr(7);
    if (k.rfind("code_predictor.model.", 0) == 0) k = "code_predictor." + k.substr(21);
    if (k.rfind("model.", 0) == 0) k = k.substr(6);
    t[k] = kv.second;
  }
  // quantizationSettings prefers quantization_config over quantization (Qwen3Config.swift:275-280);
  // pre-quantised use of the packed leaves requires `quantization` (Qwen3Talker.swift:139)
  const bool packed = cfg.has_quantization;
  int bits = 0, group = 64, mode = QMODE_AFFINE;
  if (cfg.has_quantization_config && cfg.qc_bits) { bits = cfg.qc_bits; group = cfg.qc_group; mode = cfg.qc_mode; }
  else if (cfg.has_quantization && cfg.q_bits) { bits = cfg.q_bits; group = cfg.q_group; mode = cfg.q_mode; }
  else if (!packed) { bits = 8; group = 64; }  // defaults of the offline path (:142-143)
  Loader L{t, arena, stream, packed, !packed, bits, group, mode == QMODE_MXFP4};
  L.runtime_quant = runtime_quantization && !cfg.has_quantization;  // `modelConfig.quantization == nil && applyRuntimeQuantization` (:184)

  out.talker.hidden = cfg.hidden_size; out.talker.layers = cfg.num_hidden_layers; out.talker.heads = cfg.num_attention_heads;
  out.talker.kv_heads = cfg.num_key_value_heads; out.talker.head_dim = cfg.head_dim; out.talker.inter = cfg.intermediate_size;
  out.talker.eps = cfg.rms_norm_eps; out.talker.theta = cfg.rope_theta;
  out.cp.hidden = cfg.cp.hidden_size; out.cp.layers = cfg.cp.num_hidden_layers; out.cp.heads = cfg.cp.num_attention_heads;
  out.cp.kv_heads = cfg.cp.num_key_value_heads; out.cp.head_dim = cfg.cp.head_dim; out.cp.inter = cfg.cp.intermediate_size;
  out.cp.eps = cfg.cp.rms_norm_eps; out.cp.theta = cfg.cp.rope_theta;

  out.text_embedding = L.embedding("text_embedding.weight", cfg.text_vocab_size, cfg.text_hidden_size);
  out.codec_embedding = L.embedding("codec_embedding.weight", cfg.vocab_size, cfg.hidden_size);
  out.fc1 = L.linear({"text_projection.linear_fc1"}, cfg.text_hidden_size, {cfg.text_hidden_size}, true);
  out.fc2 = L.linear({"text_projection.linear_fc2"}, cfg.text_hidden_size, {cfg.hidden_size}, true);
  L.stack("", out.talker);
  out.codec_head = L.linear({"codec_head"}, cfg.hidden_size, {cfg.vocab_size}, false);
  const int G = cfg.cp.num_code_groups;
  for (int i = 0; i < G - 1; ++i)
    out.cp_codec_embedding.push_back(L.embedding("code_predictor.codec_embedding." + std::to_string(i) + ".weight", cfg.cp.vocab_size, cfg.hidden_size));
  L.stack("code_predictor.", out.cp);
  for (int i = 0; i < G - 1; ++i)
    out.lm_head.push_back(L.linear({"code_predictor.lm_head." + std::to_string(i)}, cfg.cp.hidden_size, {cfg.cp.vocab_size}, false));
  out.has_mtp = cfg.cp.hidden_size != cfg.hidden_size;  // Qwen3CodePredictor.swift:171-175
  if (out.has_mtp)
    out.small_to_mtp = L.linear({"code_predictor.small_to_mtp_projection"}, cfg.hidden_size, {cfg.cp.hidden_size}, true);
  Q3_CUDA(cudaStreamSynchronize(stream));

  out.talker_step_bytes = stack_bytes(out.talker) + out.codec_head.weight_bytes();
  out.cp_pass_bytes = stack_bytes(out.cp) + out.lm_head[0].weight_bytes() + (out.has_mtp ? out.small_to_mtp.weight_bytes() : 0);
  out.checkpoint_bits = L.ckpt_bits;
  out.checkpoint_mode = L.ckpt_bits && L.mxfp4 ? QMODE_MXFP4 : QMODE_AFFINE;
  weight_dtype = L.weight_dtype < 0 ? Q3TTS_BF16 : L.weight_dtype;
  eff_bits = out.talker.layer[0].qkv.bits;
  eff_group = group;
}

}  // namespace q3
