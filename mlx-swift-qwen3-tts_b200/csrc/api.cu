// extern "C" entry points of libqwen3tts_b200.so (declared in include/qwen3tts_b200.h).
#include <algorithm>
#include <atomic>
#include <deque>
#include <chrono>
#include <cmath>
#include <map>
#include <thread>

#include "audio_encoder.h"
#include "speaker_encoder.h"
#include "codec.h"
#include "codec_kernels.h"
#include "codec_unit.h"
#include "engine.h"
#include "gemm_tc.h"
#include "sampler.cuh"

using namespace q3;

struct q3tts_handle : q3::Handle {};

namespace q3 {
void init_talker_kernels();
Handle::~Handle() {
  for (Handle* l : lanes) {  // clones made for q3tts_options.lanes (allocated as q3tts_handle)
    cudaStreamSynchronize(l->stream);
    delete static_cast<q3tts_handle*>(l);
  }
  lanes.clear();
  talker.reset();
  codec.reset();
  audio_encoder.reset();
  speaker_encoder.reset();
  if (ev_start) cudaEventDestroy(ev_start);
  if (ev_stop) cudaEventDestroy(ev_stop);
  if (h_pcm) cudaFreeHost(h_pcm);
  if (h_codes) cudaFreeHost(h_codes);
  if (d_codes) cudaFree(d_codes);
  if (d_pcm) cudaFree(d_pcm);
  if (own_stream && stream) cudaStreamDestroy(stream);
}
}  // namespace q3


namespace {

thread_local std::string g_create_error;

template <typename F>
q3tts_status guarded(q3tts_handle* h, F&& f) {
  if (!h) return Q3TTS_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(h->mu);
  if (h->poisoned) return Q3TTS_ERR_CUDA;  // last_error keeps the fault that poisoned the handle
  try {
    Q3_CUDA(cudaSetDevice(h->opt.device));
    f();
    return Q3TTS_OK;
  } catch (const Error& e) {
    h->last_error = e.what();
    cudaGetLastError();
    // A fault inside a kernel (the bounded mbarrier wait of tc_ptx.cuh trapping, an illegal address) is STICKY: the context is gone for the
    // whole process.  Say so once, deterministically, instead of letting every later call fail with whatever the runtime reports first.
    if (e.status == Q3TTS_ERR_CUDA && cudaDeviceSynchronize() != cudaSuccess) {
      h->poisoned = true;
      h->last_error += " -- the CUDA context is unusable after this fault: the handle is poisoned, destroy it and restart the process";
    }
    cudaGetLastError();
    return e.status;
  } catch (const std::exception& e) {
    h->last_error = e.what();
    return Q3TTS_ERR_CUDA;
  }
}

void require_device(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    fail(Q3TTS_ERR_NO_DEVICE, "no CUDA device visible (%s); libqwen3tts_b200 has no CPU path", e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
  }
  Q3_CHECK(device >= 0 && device < n, Q3TTS_ERR_NO_DEVICE, "CUDA device %d not present (%d visible)", device, n);
  cudaDeviceProp p;
  Q3_CUDA(cudaGetDeviceProperties(&p, device));
  Q3_CHECK(p.major == 10, Q3TTS_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, p.major, p.minor);
  Q3_CUDA(cudaSetDevice(device));
}

struct CallTimer {
  q3tts_handle* h;
  int64_t launches0;
  int64_t replays0 = 0, mega0 = 0;
  explicit CallTimer(q3tts_handle* hh) : h(hh) {
    h->timing = q3tts_timing{};
    launches0 = h->counter.n;
    if (h->talker) {
      replays0 = h->talker->graph_replays; mega0 = h->talker->mega_launches;
      h->talker->last_prefill_ms = 0; h->talker->last_prefill_rows = 0;
    }
    cudaEventRecord(h->ev_start, h->stream);
  }
  void finish() {
    cudaEventRecord(h->ev_stop, h->stream);
    cudaEventSynchronize(h->ev_stop);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev_start, h->ev_stop);
    h->timing.device_ms = ms;
    h->timing.kernel_launches = h->counter.n - launches0;
    if (h->talker) {
      h->timing.graph_replays = h->talker->graph_replays - replays0;
      h->timing.persistent_launches = h->talker->mega_launches - mega0;
      h->timing.prefill_ms = h->talker->last_prefill_ms;
      h->timing.prefill_rows = h->talker->last_prefill_rows;
      h->timing.weight_bytes_per_frame = (int64_t)h->talker->weight_bytes_per_frame();
    }
  }
};

void require_no_open_stream(q3tts_handle* h) {
  Q3_CHECK(h->open_stream == nullptr, Q3TTS_ERR_INVALID_ARG,
           "a stream is open on this handle (it owns talker slot 0): finish or free it before another talker call");
}

// the voice rules of every request of a call, before any device work (the engine checks them again at admission)
void check_voices(q3tts_handle* h, const q3tts_request* reqs, int n) {
  for (int i = 0; i < n; ++i) h->talker->check_voice_request(reqs[i]);
}

bool frame_valid(const int32_t* f) { return f[0] >= 0 && f[0] < 2048; }  // Model/Qwen3Talker.swift:571-576

// ---- talker drivers ------------------------------------------------------------------------------------------
// Runs one admitted utterance in slot 0 to completion; returns raw frames.
struct TalkerSpan {  // accumulates q3tts_timing.talker_ms over the talker part of a call
  q3tts_handle* h;
  cudaEvent_t a = nullptr, b = nullptr;
  explicit TalkerSpan(q3tts_handle* hh) : h(hh) {
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, h->stream);
  }
  ~TalkerSpan() {
    cudaEventRecord(b, h->stream);
    cudaEventSynchronize(b);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    h->timing.talker_ms += ms;
    cudaEventDestroy(a);
    cudaEventDestroy(b);
  }
};

void run_single(q3tts_handle* h, const q3tts_request& req, std::vector<int32_t>& raw, int& n_raw) {
  TalkerEngine& t = *h->talker;
  TalkerSpan span(h);
  n_raw = 0;
  Admission a = t.admit(0, req);
  if (a.too_short) return;
  std::vector<SlotState> st;
  const int limit = (req.forced_codes && req.n_forced_frames > 0) ? req.n_forced_frames : std::min(std::max(req.max_tokens, 0), t.max_frames());
  int done_steps = 0;
  while (true) {
    const int chunk = std::min(8, std::max(1, limit - done_steps));
    t.run_frames(1, chunk);
    t.fetch_states(1, st);
    done_steps = st[0].step;
    if (st[0].finished || st[0].step >= limit) break;
  }
  n_raw = st[0].n_frames;
  h->timing.frames += n_raw;
  raw.resize((size_t)std::max(n_raw, 1) * 16);
  t.fetch_frames(0, 0, n_raw, raw.data());
  if (req.code0_logits_out || req.cp_logits_out) t.fetch_logits(std::min(st[0].step + (st[0].finished ? 1 : 0), req.logits_capacity_frames), req.code0_logits_out, req.cp_logits_out);
  t.release(0);
}

int filter_frames(const q3tts_request& req, const std::vector<int32_t>& raw, int n_raw, int32_t* out, int capacity) {
  int n = 0;
  for (int i = 0; i < n_raw && n < capacity; ++i) {
    const int32_t* f = raw.data() + (size_t)i * 16;
    if (req.keep_invalid_frames || frame_valid(f)) {
      if (out) memcpy(out + (size_t)n * 16, f, 64);
      ++n;
    }
  }
  return n;
}

// Continuous batching of independent utterances over the handle's slots; raw[i] receives utterance i's raw frames.
void run_batch(q3tts_handle* h, const q3tts_request* reqs, int n, std::vector<std::vector<int32_t>>& raw, std::vector<int>& n_raw) {
  TalkerEngine& t = *h->talker;
  TalkerSpan span(h);
  const int B = t.max_batch();
  raw.assign(n, {});
  n_raw.assign(n, 0);
  std::vector<int> slot_req(B, -1), slot_limit(B, 0), slot_step(B, 0);
  int next = 0, active = 0, logit_req = -1;
  std::vector<SlotState> st;
  while (next < n || active > 0) {
    // admit as many pending utterances as there are free slots, in ONE concatenated prefill pass
    std::vector<TalkerEngine::AdmitItem> items;
    std::vector<int> item_req;
    int rows = 0;
    for (int s = 0; s < B && next < n; ++s) {
      if (slot_req[s] >= 0) continue;
      while (next < n) {
        const q3tts_request& rq = reqs[next];
        if (rq.code0_logits_out || rq.cp_logits_out) {
          Q3_CHECK(logit_req < 0 || logit_req == next, Q3TTS_ERR_INVALID_ARG, "at most one request of a batch may ask for logit dumps");
          logit_req = next;
        }
        if (rq.n_text_ids < 9) { ++next; continue; }  // too short: zero frames, like the reference's [] (Model/Qwen3Talker.swift:348-352)
        const int est = rq.n_instruct_ids + rq.n_ref_text_ids + std::max(rq.ref_frames, 0) + 10;
        if (!items.empty() && rows + est > t.max_prefill_rows()) break;
        rows += est;
        items.push_back({s, &rq});
        item_req.push_back(next);
        slot_limit[s] = (rq.forced_codes && rq.n_forced_frames > 0) ? rq.n_forced_frames : std::min(std::max(rq.max_tokens, 0), t.max_frames());
        slot_step[s] = 0;
        slot_req[s] = next++;
        ++active;
        break;
      }
      if (!items.empty() && rows >= t.max_prefill_rows()) break;
    }
    if (!items.empty()) {
      std::vector<Admission> adm;
      t.admit_batch(items, adm);
    }
    if (active == 0) break;
    int hi = 0;
    for (int s = 0; s < B; ++s)
      if (slot_req[s] >= 0) hi = s + 1;
    // frames still owed by the slowest active slot bound the chunk (no frame steps past max_tokens)
    int need = 1;
    for (int s = 0; s < hi; ++s)
      if (slot_req[s] >= 0) need = std::max(need, slot_limit[s] - slot_step[s]);
    // slots beyond `hi` are inactive (their sampler / finalize / advance are no-ops): running a few more rows costs nothing on the
    // tensor-core step, while every distinct slot count is its own CUDA graph (capture + instantiate: tens of ms) -- utterances
    // finishing one by one must not trigger a capture each
    const int run_slots = t.step_slots(hi);
    t.run_frames(run_slots, std::min(8, need));
    t.fetch_states(hi, st);
    for (int s = 0; s < hi; ++s) slot_step[s] = st[s].step;
    for (int s = 0; s < hi; ++s) {
      if (slot_req[s] < 0 || !st[s].finished) continue;
      const int r = slot_req[s];
      n_raw[r] = st[s].n_frames;
      h->timing.frames += n_raw[r];
      raw[r].resize((size_t)std::max(n_raw[r], 1) * 16);
      t.fetch_frames(s, 0, n_raw[r], raw[r].data());
      if (r == logit_req && t.dump_slot() == s)  // before the slot can be re-admitted
        t.fetch_logits(std::min(st[s].step + 1, reqs[r].logits_capacity_frames), reqs[r].code0_logits_out, reqs[r].cp_logits_out);
      t.release(s);
      slot_req[s] = -1;
      --active;
    }
  }
}

// ---- codec drivers ---------------------------------------------------------------------------------------------
struct DecodeJob {
  const int32_t* frames;  // host [T][16]
  int T;
  float* out;         // host destination
  int64_t drop;       // leading samples to skip (left context)
  int64_t max_out;    // samples to deliver at most
};

void ensure_pinned(q3tts_handle* h, size_t pcm_floats, size_t code_ints) {
  // grow in coarse steps (cudaMallocHost / cudaFree of tens of MB stall the call that first needs them)
  pcm_floats = (pcm_floats + (size_t(1) << 20) - 1) >> 20 << 20;
  code_ints = (code_ints + 8191) / 8192 * 8192;
  if (pcm_floats > h->h_pcm_floats) {
    if (h->h_pcm) cudaFreeHost(h->h_pcm);
    h->h_pcm = nullptr;
    Q3_CUDA(cudaMallocHost(&h->h_pcm, pcm_floats * sizeof(float)));
    h->h_pcm_floats = pcm_floats;
  }
  if (code_ints > h->h_codes_ints) {
    if (h->h_codes) cudaFreeHost(h->h_codes);
    h->h_codes = nullptr;
    Q3_CUDA(cudaMallocHost(&h->h_codes, code_ints * sizeof(int32_t)));
    h->h_codes_ints = code_ints;
  }
  if (code_ints > h->d_codes_ints) {
    if (h->d_codes) { Q3_CUDA(cudaStreamSynchronize(h->stream)); cudaFree(h->d_codes); }
    h->d_codes = nullptr;
    Q3_CUDA(cudaMalloc(&h->d_codes, code_ints * sizeof(int32_t)));
    h->d_codes_ints = code_ints;
  }
  if (pcm_floats > h->d_pcm_floats) {
    if (h->d_pcm) { Q3_CUDA(cudaStreamSynchronize(h->stream)); cudaFree(h->d_pcm); }
    h->d_pcm = nullptr;
    Q3_CUDA(cudaMalloc(&h->d_pcm, pcm_floats * sizeof(float)));
    h->d_pcm_floats = pcm_floats;
  }
}

// Decodes jobs grouped by equal T, each group in passes of up to pass_frames frames (jobs stacked on the batch axis).
void run_decode_jobs(q3tts_handle* h, std::vector<DecodeJob>& jobs) {
  CodecDecoder& c = *h->codec;
  const int up = c.total_upsample();
  std::map<int, std::vector<size_t>> by_t;
  for (size_t i = 0; i < jobs.size(); ++i)
    if (jobs[i].T > 0) by_t[jobs[i].T].push_back(i);
  // Passes are double-buffered: while pass k runs on the device, the host copies pass k-1's PCM from pinned staging into the
  // caller's buffers (10-13 MB per window batch: 2-3 ms during which the GPU used to idle).
  struct Pass { int T, nb; size_t p0; const std::vector<size_t>* idx; };
  std::vector<Pass> passes;
  for (auto& kv : by_t) {
    const int T = kv.first;
    Q3_CHECK(T <= c.pass_frames(), Q3TTS_ERR_CAPACITY, "decode window of %d frames exceeds codec pass capacity %d (q3tts_options.codec_max_frames)", T, c.pass_frames());
    const int per_pass = std::max(1, c.pass_frames() / T);
    for (size_t p0 = 0; p0 < kv.second.size(); p0 += per_pass)
      passes.push_back({T, (int)std::min<size_t>(per_pass, kv.second.size() - p0), p0, &kv.second});
  }
  if (passes.empty()) return;
  // staging sized once for two full passes (pass_frames x 1920 floats = 18 MB pinned each at the default 2400 frames): growing on
  // demand put a cudaMallocHost / cudaFree pair (27-800 ms measured) into whichever call first saw a slightly larger window batch
  const size_t pcm_cap = (size_t)c.pass_frames() * up, code_cap = (size_t)c.pass_frames() * 16;
  ensure_pinned(h, 2 * pcm_cap, 2 * code_cap);
  struct Events {  // destroyed on every exit path (a failing pass throws)
    cudaEvent_t e0[2] = {nullptr, nullptr}, e1[2] = {nullptr, nullptr}, done[2] = {nullptr, nullptr};
    ~Events() {
      for (int i = 0; i < 2; ++i) {
        if (e0[i]) cudaEventDestroy(e0[i]);
        if (e1[i]) cudaEventDestroy(e1[i]);
        if (done[i]) cudaEventDestroy(done[i]);
      }
    }
  } ev;
  cudaEvent_t (&e0)[2] = ev.e0, (&e1)[2] = ev.e1, (&done)[2] = ev.done;
  for (int i = 0; i < 2; ++i) {
    Q3_CUDA(cudaEventCreate(&e0[i]));
    Q3_CUDA(cudaEventCreate(&e1[i]));
    Q3_CUDA(cudaEventCreate(&done[i]));
  }
  const bool trace = getenv("Q3TTS_HOST_TRACE") != nullptr;
  auto drain = [&](size_t k) {  // wait for pass k's PCM, account its device time, scatter it to the jobs' destinations
    const Pass& ps = passes[k];
    const int buf = (int)(k & 1);
    Q3_CUDA(cudaEventSynchronize(done[buf]));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0[buf], e1[buf]);
    h->timing.decode_ms += ms;
    h->timing.codec_flops += (int64_t)ps.nb * ps.T * c.flops_per_frame();
    if (trace) fprintf(stderr, "[q3tts host]   codec pass nb=%d T=%d: %.2f ms on the device\n", ps.nb, ps.T, ms);
    const float* src = h->h_pcm + (size_t)buf * pcm_cap;
    for (int b = 0; b < ps.nb; ++b) {
      DecodeJob& j = jobs[(*ps.idx)[ps.p0 + b]];
      const int64_t total = (int64_t)ps.T * up;
      const int64_t n = std::max<int64_t>(0, std::min<int64_t>(total - j.drop, j.max_out));
      if (n > 0) memcpy(j.out, src + (size_t)b * total + j.drop, (size_t)n * sizeof(float));
    }
  };
  for (size_t k = 0; k < passes.size(); ++k) {
    const Pass& ps = passes[k];
    const int buf = (int)(k & 1), T = ps.T, nb = ps.nb;
    const size_t code_ints = (size_t)nb * T * 16, pcm_floats = (size_t)nb * T * up;
    int32_t* hc = h->h_codes + (size_t)buf * code_cap;   // buffer `buf` was last used by pass k-2, drained during iteration k-1
    int32_t* d_codes = h->d_codes + (size_t)buf * code_cap;
    float* d_pcm = h->d_pcm + (size_t)buf * pcm_cap;
    for (int b = 0; b < nb; ++b) memcpy(hc + (size_t)b * T * 16, jobs[(*ps.idx)[ps.p0 + b]].frames, (size_t)T * 64);
    Q3_CUDA(cudaMemcpyAsync(d_codes, hc, code_ints * 4, cudaMemcpyHostToDevice, h->stream));
    h->timing.h2d_bytes += (int64_t)code_ints * 4;
    Q3_CUDA(cudaEventRecord(e0[buf], h->stream));
    c.decode_pass(d_codes, nb, T, d_pcm);
    Q3_CUDA(cudaEventRecord(e1[buf], h->stream));
    Q3_CUDA(cudaMemcpyAsync(h->h_pcm + (size_t)buf * pcm_cap, d_pcm, pcm_floats * 4, cudaMemcpyDeviceToHost, h->stream));
    Q3_CUDA(cudaEventRecord(done[buf], h->stream));
    h->timing.d2h_bytes += (int64_t)pcm_floats * 4;
    if (k >= 1) drain(k - 1);
  }
  drain(passes.size() - 1);
}

// NaN/Inf -> 0, clamp (Qwen3TTSPipeline.swift:565-570, 726-732) happen on the device in the codec's output kernel
// (clip(-1, 1) maps +-Inf to +-1 before the Swift scrub would see it; NaN -> 0 is fused into out_conv_kernel), so the PCM that
// reaches the host needs no second pass over every sample.

// Schedules the decode windows of one utterance's valid frames as `mode` prescribes; appends jobs writing into out.
int64_t plan_decode(int mode, const int32_t* frames, int n, float* out, int64_t capacity, int up, std::vector<DecodeJob>& jobs) {
  if (n <= 0) return 0;
  const int64_t total = std::min<int64_t>((int64_t)n * up, capacity);
  if (mode == Q3TTS_DECODE_WHOLE) {
    jobs.push_back({frames, n, out, 0, total});
    return total;
  }
  const int chunk = mode == Q3TTS_DECODE_FILE ? 16 : (mode == Q3TTS_DECODE_BATCHAPI ? 24 : 18), left = 8;
  for (int pos = 0; pos < n; pos += chunk) {
    const int end = std::min(pos + chunk, n);
    const int ctx = pos == 0 ? 0 : std::min(left, pos);  // codes[max(0,end-8)..<end] of the previous window (:734, 561)
    const int64_t o0 = (int64_t)pos * up;
    if (o0 >= total) break;
    jobs.push_back({frames + (size_t)(pos - ctx) * 16, end - pos + ctx, out + o0, (int64_t)ctx * up, std::min<int64_t>((int64_t)(end - pos) * up, total - o0)});
  }
  return total;
}

}  // namespace

// =================================================================================================== lifecycle
extern "C" {

int32_t q3tts_abi_version(void) { return Q3TTS_ABI_VERSION; }

void q3tts_default_options(q3tts_options* o) {
  if (!o) return;
  memset(o, 0, sizeof *o);
  o->struct_size = (int32_t)sizeof *o;
  o->device = 0;
  o->max_batch = 1;
  o->kv_capacity = 512;
  o->max_frames = 2400;
  o->use_cuda_graph = 1;
  o->load_codec = 1;
  o->load_talker = 1;
  o->codec_max_frames = 2400;
  o->codec_max_batch = 8;
}

void q3tts_default_request(q3tts_request* r) {
  if (!r) return;
  memset(r, 0, sizeof *r);
  r->struct_size = (int32_t)sizeof *r;
  r->speaker_id = -1;
  r->temperature = 0.9f;          // Model/Qwen3Talker.swift:335
  r->top_k = 0;                   // :277
  r->top_p = 1.0f;
  r->repetition_penalty = 1.05f;  // :279
  r->max_tokens = 1200;           // :336
}

q3tts_status q3tts_create(const char* model_dir, const q3tts_options* opts, q3tts_handle** out) {
  if (!out) return Q3TTS_ERR_INVALID_ARG;
  *out = nullptr;
  q3tts_handle* h = nullptr;
  try {
    Q3_CHECK(model_dir != nullptr, Q3TTS_ERR_INVALID_ARG, "model_dir is NULL");
    q3tts_options o;
    q3tts_default_options(&o);
    if (opts) {
      const size_t n = std::min<size_t>(sizeof o, opts->struct_size > 0 ? (size_t)opts->struct_size : sizeof o);
      memcpy(&o, opts, n);
    }
    require_device(o.device);
    h = new q3tts_handle();
    h->opt.device = o.device;
    h->opt.max_batch = o.max_batch > 0 ? o.max_batch : 1;
    h->opt.kv_capacity = o.kv_capacity > 0 ? std::max(o.kv_capacity, 208) : 512;
    h->opt.max_frames = o.max_frames > 0 ? o.max_frames : 2400;
    h->opt.use_cuda_graph = o.use_cuda_graph;
    h->opt.load_codec = o.load_codec;
    h->opt.load_talker = o.load_talker;
    h->opt.codec_max_frames = o.codec_max_frames > 0 ? o.codec_max_frames : 2400;
    h->opt.codec_max_batch = o.codec_max_batch > 0 ? o.codec_max_batch : 8;
    Q3_CHECK(o.packed_gemm >= 0 && o.packed_gemm <= 2, Q3TTS_ERR_INVALID_ARG, "options.packed_gemm must be 0, 1 or 2");
    h->opt.packed_gemm = o.packed_gemm;
    h->opt.runtime_quantization = o.runtime_quantization != 0;
    h->opt.lanes = std::max(1, std::min(o.lanes, 8));
    if (o.cuda_stream) {
      h->stream = (cudaStream_t)o.cuda_stream;
    } else {
      Q3_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
      h->own_stream = true;
    }
    h->opt.stream = h->stream;
    Q3_CUDA(cudaEventCreate(&h->ev_start));
    Q3_CUDA(cudaEventCreate(&h->ev_stop));
    const std::string dir(model_dir);
    h->model_dir = dir;
    if (h->opt.load_talker) {
      // config.json, then model.safetensors (Qwen3TTSPipeline.swift:127-141)
      Json root = parse_json_file(dir + "/config.json");
      h->cfg = parse_talker_config(root);
      h->talker.reset(new TalkerEngine(dir, h->cfg, h->opt, h->stream, &h->counter));
      h->has_talker = true;
      // speaker encoder, optional (Qwen3TTSPipeline.swift:155-169): present only in checkpoints that carry `speaker_encoder.*`
      if (SpeakerEncoderDev::present(dir)) {
        try {
          h->speaker_encoder.reset(new SpeakerEncoderDev(dir, h->stream, &h->counter));
        } catch (const Error& e) {
          g_create_error = std::string("speaker encoder not loaded: ") + e.what();
          cudaGetLastError();
        }
      }
    }
    if (h->opt.load_codec) {
      // speech_tokenizer/{config...} + model.safetensors (Qwen3TTSPipeline.swift:191-208)
      // one pass holds up to codec_max_frames frames (batch x window); the workspace itself is allocated on first use
      h->codec.reset(new CodecDecoder(dir + "/speech_tokenizer", h->stream, &h->counter, h->opt.codec_max_frames));
      // audio encoder for ICL, optional: a failing load leaves ICL unavailable, it does not fail the pipeline (Qwen3TTSPipeline.swift:210-218)
      if (AudioEncoder::present(dir + "/speech_tokenizer")) {
        try {
          h->audio_encoder.reset(new AudioEncoder(dir + "/speech_tokenizer", h->stream, &h->counter));
        } catch (const Error& e) {
          g_create_error = std::string("audio encoder not loaded: ") + e.what();
          cudaGetLastError();
        }
      }
    }
    Q3_CUDA(cudaStreamSynchronize(h->stream));
    *out = h;
    return Q3TTS_OK;
  } catch (const Error& e) {
    g_create_error = e.what();
    cudaGetLastError();
    delete h;
    return e.status;
  } catch (const std::exception& e) {
    g_create_error = e.what();
    delete h;
    return Q3TTS_ERR_CUDA;
  }
}

q3tts_status q3tts_clone(q3tts_handle* parent, q3tts_handle** out) {
  if (!out) return Q3TTS_ERR_INVALID_ARG;
  *out = nullptr;
  if (!parent) return Q3TTS_ERR_INVALID_ARG;
  q3tts_handle* h = nullptr;
  try {
    std::lock_guard<std::mutex> lk(parent->mu);
    Q3_CHECK(!parent->poisoned, Q3TTS_ERR_CUDA, "the parent handle is poisoned");
    Q3_CUDA(cudaSetDevice(parent->opt.device));
    h = new q3tts_handle();
    h->opt = parent->opt;
    h->opt.lanes = 1;  // a clone is one chain
    h->model_dir = parent->model_dir;
    Q3_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));  // always its own stream: the point of a clone is a second chain
    h->own_stream = true;
    h->opt.stream = h->stream;
    Q3_CUDA(cudaEventCreate(&h->ev_start));
    Q3_CUDA(cudaEventCreate(&h->ev_stop));
    if (parent->talker) {
      h->cfg = parent->cfg;
      h->talker.reset(new TalkerEngine(h->model_dir, h->cfg, h->opt, h->stream, &h->counter, parent->talker->shared()));
      h->has_talker = true;
    }
    if (parent->codec) {  // codec weights are small (0.6 GB with their fp16 copies): loaded again, with their own workspace
      h->codec.reset(new CodecDecoder(h->model_dir + "/speech_tokenizer", h->stream, &h->counter, h->opt.codec_max_frames));
    }
    Q3_CUDA(cudaStreamSynchronize(h->stream));
    *out = h;
    return Q3TTS_OK;
  } catch (const Error& e) {
    g_create_error = e.what();
    cudaGetLastError();
    delete h;
    return e.status;
  } catch (const std::exception& e) {
    g_create_error = e.what();
    delete h;
    return Q3TTS_ERR_CUDA;
  }
}

void q3tts_destroy(q3tts_handle* h) {
  if (!h) return;
  cudaSetDevice(h->opt.device);
  cudaStreamSynchronize(h->stream);
  delete h;
}

const char* q3tts_last_error(const q3tts_handle* h) { return h ? h->last_error.c_str() : g_create_error.c_str(); }

q3tts_status q3tts_get_info(const q3tts_handle* hc, q3tts_info* out) {
  if (!hc || !out) return Q3TTS_ERR_INVALID_ARG;
  memset(out, 0, sizeof *out);
  const TalkerConfig& c = hc->cfg;
  if (hc->talker) {
    out->hidden_size = c.hidden_size; out->num_layers = c.num_hidden_layers; out->num_heads = c.num_attention_heads;
    out->num_kv_heads = c.num_key_value_heads; out->head_dim = c.head_dim; out->intermediate_size = c.intermediate_size;
    out->vocab_size = c.vocab_size; out->text_vocab_size = c.text_vocab_size; out->text_hidden_size = c.text_hidden_size;
    out->cp_hidden_size = c.cp.hidden_size; out->cp_num_layers = c.cp.num_hidden_layers; out->cp_vocab_size = c.cp.vocab_size;
    out->num_code_groups = c.cp.num_code_groups;
    out->quant_bits = hc->talker->quant_bits(); out->quant_group_size = hc->talker->quant_group();
    out->checkpoint_quant_bits = hc->talker->checkpoint_quant_bits();
    out->checkpoint_quant_mode = hc->talker->checkpoint_quant_mode();
    out->weight_dtype = hc->talker->weight_dtype();
    out->num_speakers = (int32_t)c.spk_id.size();
    out->model_type = c.tts_model_type == "voice_design" ? 1 : (c.tts_model_type == "custom_voice" ? 2 : 0);
    out->codec_eos_id = c.codec_eos_token_id; out->codec_pad_id = c.codec_pad_id;
    out->max_batch = hc->talker->max_batch(); out->kv_capacity = hc->talker->kv_capacity(); out->max_frames = hc->talker->max_frames();
    out->device_bytes += (int64_t)hc->talker->device_bytes();
  }
  if (hc->codec) {
    out->has_codec = 1;
    out->codec_num_quantizers = hc->codec->config().num_quantizers;
    out->codec_total_upsample = hc->codec->total_upsample();
    out->device_bytes += (int64_t)hc->codec->device_bytes();
  }
  if (hc->speaker_encoder) {
    out->has_speaker_encoder = 1;
    out->speaker_embedding_dim = hc->speaker_encoder->embedding_dim();
    out->device_bytes += (int64_t)hc->speaker_encoder->device_bytes();
  }
  if (hc->audio_encoder) {
    out->has_audio_encoder = 1;
    out->audio_encoder_hidden = hc->audio_encoder->config().hidden_size;
    out->device_bytes += (int64_t)hc->audio_encoder->device_bytes();
  }
  return Q3TTS_OK;
}

q3tts_status q3tts_speaker_name(const q3tts_handle* h, int32_t index, char* name_out, int32_t capacity, int32_t* id_out) {
  if (!h || index < 0 || index >= (int32_t)h->cfg.spk_id.size()) return Q3TTS_ERR_INVALID_ARG;
  std::vector<std::pair<std::string, int>> s = h->cfg.spk_id;
  std::sort(s.begin(), s.end());  // availableSpeakers = keys.sorted() (Qwen3TTSPipeline.swift:77-79)
  if (name_out && capacity > 0) {
    strncpy(name_out, s[index].first.c_str(), capacity - 1);
    name_out[capacity - 1] = 0;
  }
  if (id_out) *id_out = s[index].second;
  return Q3TTS_OK;
}

int32_t q3tts_speaker_id(const q3tts_handle* h, const char* name) {
  if (!h || !name) return -1;
  for (auto& kv : h->cfg.spk_id)
    if (kv.first == name) return kv.second;
  return -1;
}

q3tts_status q3tts_clear_cache(q3tts_handle* h) {
  if (h) {  // the lanes of q3tts_options.lanes first (each under its own mutex)
    std::lock_guard<std::mutex> lk(h->lanes_mu);
    for (q3::Handle* l : h->lanes) q3tts_clear_cache(static_cast<q3tts_handle*>(l));
  }
  return guarded(h, [&] {
    Q3_CUDA(cudaStreamSynchronize(h->stream));
    if (h->talker) h->talker->drop_graphs();
  });
}

q3tts_status q3tts_get_timing(const q3tts_handle* h, q3tts_timing* out) {
  if (!h || !out) return Q3TTS_ERR_INVALID_ARG;
  *out = h->timing;
  return Q3TTS_OK;
}

// =================================================================================================== talker
q3tts_status q3tts_generate_codes(q3tts_handle* h, const q3tts_request* req, int32_t* codes_out, int32_t capacity_frames,
                                  int32_t* frames_out) {
  return guarded(h, [&] {
    Q3_CHECK(req && frames_out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(h->talker != nullptr, Q3TTS_ERR_MODEL_NOT_LOADED, "Model is not loaded");
    require_no_open_stream(h);
    check_voices(h, req, 1);
    *frames_out = 0;
    CallTimer tm(h);
    std::vector<int32_t> raw;
    int n_raw = 0;
    run_single(h, *req, raw, n_raw);
    *frames_out = filter_frames(*req, raw, n_raw, codes_out, capacity_frames);
    h->timing.d2h_bytes += (int64_t)n_raw * 64;
    h->timing.h2d_bytes += (int64_t)req->n_text_ids * 4;
    tm.finish();
  });
}

// ---- q3tts_options.lanes: one call, several launch chains ---------------------------------------------------------------
// A call with more requests than one handle has slots is split into contiguous shares, one per lane (this handle + clones that share its
// weights); every share runs the ordinary single-handle path -- continuous batching over the lane's slots -- on a worker thread that lives
// only inside the call.  Requests are independent (SURVEY.md 8e) and a handle's numeric path is fixed at creation, so every request gets
// the bits it gets from a single-lane call.  Requests that ask for logits dumps keep the call on one lane (one dump slot per handle).
static bool use_lanes(q3tts_handle* h, const q3tts_request* reqs, int32_t n) {
  if (!h || !reqs || h->opt.lanes <= 1 || n <= h->opt.max_batch || h->poisoned) return false;
  for (int i = 0; i < n; ++i)
    if (reqs[i].code0_logits_out || reqs[i].cp_logits_out) return false;
  return true;
}

}  // extern "C"
template <typename F>
static q3tts_status over_lanes(q3tts_handle* h, int32_t n, F&& run) {
  const int B = h->opt.max_batch;
  const int blocks = (n + B - 1) / B;
  const int L = std::min(h->opt.lanes, blocks);
  std::vector<q3::Handle*> lanes;
  {  // clones are created on the first call that needs them
    std::lock_guard<std::mutex> lk(h->lanes_mu);
    while ((int)h->lanes.size() < L - 1) {
      q3tts_handle* c = nullptr;
      const q3tts_status st = q3tts_clone(h, &c);
      if (st != Q3TTS_OK) {
        std::lock_guard<std::mutex> lk2(h->mu);
        h->last_error = "lane handle not created: " + g_create_error;
        return st;
      }
      h->lanes.push_back(c);
    }
    lanes.assign(h->lanes.begin(), h->lanes.begin() + (L - 1));  // a private copy: another call on this handle may grow the vector meanwhile
  }
  // contiguous shares in whole blocks of max_batch requests (the last lane takes the remainder)
  std::vector<int> off(L + 1, 0);
  for (int l = 0; l < L; ++l) off[l + 1] = std::min<int>(n, off[l] + (blocks / L + (l < blocks % L ? 1 : 0)) * B);
  off[L] = n;
  std::vector<q3tts_status> st(L, Q3TTS_OK);
  std::vector<std::thread> workers;
  for (int l = 1; l < L; ++l)
    workers.emplace_back([&, l] { st[l] = run(static_cast<q3tts_handle*>(lanes[l - 1]), off[l], off[l + 1] - off[l]); });
  st[0] = run(h, off[0], off[1] - off[0]);
  for (auto& w : workers) w.join();
  // the call's timing: the lanes ran side by side -- times are the slowest lane's, counters add up
  std::lock_guard<std::mutex> lk(h->mu);
  q3tts_status result = st[0];
  for (int l = 1; l < L; ++l) {
    q3::Handle* lane = lanes[l - 1];
    std::lock_guard<std::mutex> lk2(lane->mu);
    const q3tts_timing& t = lane->timing;
    q3tts_timing& a = h->timing;
    a.device_ms = std::max(a.device_ms, t.device_ms); a.prefill_ms = std::max(a.prefill_ms, t.prefill_ms);
    a.decode_ms = std::max(a.decode_ms, t.decode_ms); a.talker_ms = std::max(a.talker_ms, t.talker_ms);
    a.kernel_launches += t.kernel_launches; a.graph_replays += t.graph_replays; a.frames += t.frames;
    a.h2d_bytes += t.h2d_bytes; a.d2h_bytes += t.d2h_bytes; a.codec_flops += t.codec_flops; a.persistent_launches += t.persistent_launches;
    a.prefill_rows += t.prefill_rows;
    if (result == Q3TTS_OK && st[l] != Q3TTS_OK) {
      result = st[l];
      h->last_error = "lane " + std::to_string(l) + ": " + lane->last_error;
      if (lane->poisoned) h->poisoned = true;  // one CUDA context: a kernel fault on any lane ends them all
    }
  }
  return result;
}
extern "C" {

static q3tts_status generate_codes_batch_one(q3tts_handle* h, const q3tts_request* reqs, int32_t n, int32_t* const* codes_out,
                                             int32_t capacity_frames, int32_t* frames_out) {
  return guarded(h, [&] {
    Q3_CHECK(reqs && frames_out && n >= 0, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(h->talker != nullptr, Q3TTS_ERR_MODEL_NOT_LOADED, "Model is not loaded");
    require_no_open_stream(h);
    check_voices(h, reqs, n);
    CallTimer tm(h);
    std::vector<std::vector<int32_t>> raw;
    std::vector<int> n_raw;
    run_batch(h, reqs, n, raw, n_raw);
    for (int i = 0; i < n; ++i) {
      frames_out[i] = filter_frames(reqs[i], raw[i], n_raw[i], codes_out ? codes_out[i] : nullptr, capacity_frames);
      h->timing.d2h_bytes += (int64_t)n_raw[i] * 64;
      h->timing.h2d_bytes += (int64_t)reqs[i].n_text_ids * 4;
    }
    tm.finish();
  });
}

q3tts_status q3tts_generate_codes_batch(q3tts_handle* h, const q3tts_request* reqs, int32_t n, int32_t* const* codes_out,
                                        int32_t capacity_frames, int32_t* frames_out) {
  if (!use_lanes(h, reqs, n) || !frames_out) return generate_codes_batch_one(h, reqs, n, codes_out, capacity_frames, frames_out);
  const q3tts_status st = guarded(h, [&] { check_voices(h, reqs, n); });  // every lane's share, before any lane starts
  if (st != Q3TTS_OK) return st;
  return over_lanes(h, n, [&](q3tts_handle* lane, int off, int cnt) {
    return generate_codes_batch_one(lane, reqs + off, cnt, codes_out ? codes_out + off : nullptr, capacity_frames, frames_out + off);
  });
}

}  // extern "C"

// ---- streaming ---------------------------------------------------------------------------------------------------
struct q3tts_stream {
  q3tts_handle* h = nullptr;
  int chunk_size = 12;
  int limit = 0;
  int emitted = 0;     // raw frames already delivered
  bool talker_done = false, too_short = false;
  std::atomic<bool> cancelled{false};  // q3tts_stream_cancel may be called from another thread than the one pulling chunks
  // consumer state of _generateStreamImpl (Qwen3TTSPipeline.swift:520-563)
  std::deque<std::vector<int32_t>> code_buffer;  // valid frames
  std::vector<int32_t> left_context;             // up to 8 frames
  bool first_decode = true, final_sent = false;
  int total_processed = 0;
  bool released = false;
};

namespace {
// Produce the next chunk of raw frames (up to chunk_size); sets talker_done when the loop ended.
int stream_pull(q3tts_stream* s, int32_t* out) {
  TalkerEngine& t = *s->h->talker;
  if (s->talker_done || s->too_short) { s->talker_done = true; return 0; }
  std::vector<SlotState> st;
  t.fetch_states(1, st);
  while (!s->cancelled && !st[0].finished && st[0].n_frames - s->emitted < s->chunk_size) {
    const int want = s->chunk_size - (st[0].n_frames - s->emitted);
    t.run_frames(1, std::max(1, std::min(want, s->limit - st[0].step)));
    t.fetch_states(1, st);
  }
  const int avail = st[0].n_frames - s->emitted;
  const int n = std::min(avail, s->chunk_size);
  if (n > 0) t.fetch_frames(0, s->emitted, n, out);
  s->emitted += n;
  s->h->timing.frames += n;
  if ((st[0].finished || s->cancelled) && s->emitted >= st[0].n_frames) {
    s->talker_done = true;
    if (!s->released) { t.release(0); s->released = true; }
  }
  return n;
}
}  // namespace

extern "C" {

q3tts_status q3tts_stream_begin(q3tts_handle* h, const q3tts_request* req, int32_t chunk_size, q3tts_stream** out) {
  if (out) *out = nullptr;
  return guarded(h, [&] {
    Q3_CHECK(req && out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(h->talker != nullptr, Q3TTS_ERR_MODEL_NOT_LOADED, "Model is not loaded");
    require_no_open_stream(h);
    check_voices(h, req, 1);
    h->timing = q3tts_timing{};
    std::unique_ptr<q3tts_stream> s(new q3tts_stream());
    s->h = h;
    s->chunk_size = chunk_size > 0 ? chunk_size : 12;  // defaultStreamingChunkSize (Qwen3TTSPipeline.swift:43)
    q3tts_request r = *req;
    r.stream_variant = 1;
    h->talker->last_prefill_ms = 0;
    h->talker->last_prefill_rows = 0;
    Admission a = h->talker->admit(0, r);
    h->timing.prefill_ms = h->talker->last_prefill_ms;
    h->timing.prefill_rows = h->talker->last_prefill_rows;
    s->too_short = a.too_short;
    s->limit = std::min(std::max(r.max_tokens, 0), h->talker->max_frames());
    h->open_stream = s.get();
    *out = s.release();
  });
}

q3tts_status q3tts_stream_next(q3tts_stream* s, int32_t* codes_out, int32_t* frames_out, int32_t* done_out) {
  if (!s || !codes_out || !frames_out || !done_out) return Q3TTS_ERR_INVALID_ARG;
  return guarded(s->h, [&] {
    *frames_out = stream_pull(s, codes_out);
    *done_out = s->talker_done ? 1 : 0;
  });
}

q3tts_status q3tts_stream_next_audio(q3tts_stream* s, float* pcm_out, int32_t capacity_samples, int32_t* samples_out,
                                     int32_t* token_start_out, int32_t* token_end_out, int32_t* is_final_out, int32_t* done_out) {
  if (!s || !pcm_out || !samples_out || !done_out) return Q3TTS_ERR_INVALID_ARG;
  return guarded(s->h, [&] {
    q3tts_handle* h = s->h;
    Q3_CHECK(h->codec != nullptr, Q3TTS_ERR_DECODER_LOAD_FAILED, "Failed to load MLX audio decoder");
    const int DECODE_CHUNK = 18, LEFT = 8, up = h->codec->total_upsample();
    // checked BEFORE any stream state changes: a too-small buffer must not consume frames
    Q3_CHECK((int64_t)capacity_samples >= (int64_t)DECODE_CHUNK * up, Q3TTS_ERR_CAPACITY, "pcm_out holds %d samples, a chunk needs %d", capacity_samples, DECODE_CHUNK * up);
    *samples_out = 0;
    *done_out = 0;
    int tok0 = s->total_processed, tok1 = s->total_processed, is_final = 0;
    auto decode_batch = [&](int count) {
      std::vector<int32_t> win;
      const int ctx = s->first_decode ? 0 : (int)s->left_context.size() / 16;
      if (!s->first_decode) win = s->left_context;
      s->first_decode = false;
      std::vector<int32_t> batch;
      for (int i = 0; i < count; ++i) {
        batch.insert(batch.end(), s->code_buffer.front().begin(), s->code_buffer.front().end());
        s->code_buffer.pop_front();
      }
      win.insert(win.end(), batch.begin(), batch.end());
      const int T = (int)win.size() / 16;
      std::vector<DecodeJob> jobs{{win.data(), T, pcm_out, (int64_t)ctx * up, (int64_t)count * up}};
      run_decode_jobs(h, jobs);
      const int keep = std::min(LEFT, count);  // leftContext = codes.suffix(8) (:561)
      s->left_context.assign(batch.end() - (size_t)keep * 16, batch.end());
      *samples_out = count * up;
      tok0 = s->total_processed;
      s->total_processed += count;
      tok1 = s->total_processed;
    };
    std::vector<int32_t> chunk((size_t)s->chunk_size * 16);
    while (true) {
      if ((int)s->code_buffer.size() >= DECODE_CHUNK) { decode_batch(DECODE_CHUNK); break; }
      if (!s->talker_done) {
        const int n = stream_pull(s, chunk.data());
        for (int i = 0; i < n; ++i)
          if (frame_valid(chunk.data() + (size_t)i * 16))  // :576-579
            s->code_buffer.emplace_back(chunk.begin() + (size_t)i * 16, chunk.begin() + (size_t)(i + 1) * 16);
        continue;
      }
      if (!s->code_buffer.empty()) { decode_batch((int)s->code_buffer.size()); is_final = 1; break; }  // flush (:598-605)
      // trailing empty isFinal chunk, always (:607)
      s->final_sent = true;
      is_final = 1;
      *done_out = 1;
      break;
    }
    if (token_start_out) *token_start_out = tok0;
    if (token_end_out) *token_end_out = tok1;
    if (is_final_out) *is_final_out = is_final;
  });
}

q3tts_status q3tts_stream_cancel(q3tts_stream* s) {
  if (!s) return Q3TTS_ERR_INVALID_ARG;
  s->cancelled.store(true);
  return Q3TTS_OK;
}

void q3tts_stream_free(q3tts_stream* s) {
  if (!s) return;
  if (s->h) {
    guarded(s->h, [&] {
      if (s->h->talker && !s->released) s->h->talker->release(0);
      if (s->h->open_stream == s) s->h->open_stream = nullptr;
    });
  }
  delete s;
}

// =================================================================================================== registered voices
q3tts_status q3tts_voice_create(q3tts_handle* h, const q3tts_request* voice, q3tts_voice** out) {
  if (out) *out = nullptr;
  if (!h || !voice || !out) return Q3TTS_ERR_INVALID_ARG;
  return guarded(h, [&] {
    Q3_CHECK(h->talker != nullptr, Q3TTS_ERR_MODEL_NOT_LOADED, "Model is not loaded");
    require_no_open_stream(h);  // the stream owns slot 0, the scratch slot of the prefix prefill
    std::unique_ptr<q3tts_voice> v(new q3tts_voice());
    v->device = h->opt.device;
    h->talker->create_voice(*voice, *v);
    *out = v.release();
  });
}

q3tts_status q3tts_voice_info(const q3tts_voice* v, int32_t* prefix_positions_out, int64_t* device_bytes_out) {
  if (!v) return Q3TTS_ERR_INVALID_ARG;
  if (prefix_positions_out) *prefix_positions_out = v->prefix_len;
  if (device_bytes_out) *device_bytes_out = (int64_t)v->bytes;
  return Q3TTS_OK;
}

void q3tts_voice_free(q3tts_voice* v) { delete v; }

// =================================================================================================== codec
q3tts_status q3tts_decode(q3tts_handle* h, const int32_t* codes, int32_t batch, int32_t frames, float* pcm_out) {
  return guarded(h, [&] {
    Q3_CHECK(h->codec != nullptr, Q3TTS_ERR_DECODER_LOAD_FAILED, "Failed to load MLX audio decoder");
    Q3_CHECK(codes && pcm_out && batch >= 0 && frames >= 0, Q3TTS_ERR_INVALID_ARG, "bad arguments");
    CallTimer tm(h);
    const int up = h->codec->total_upsample(), Q = h->codec->config().num_quantizers;
    Q3_CHECK(Q == 16, Q3TTS_ERR_BAD_CONFIG, "codec with %d quantizers: the ABI carries 16 codes per frame", Q);
    std::vector<DecodeJob> jobs;
    for (int b = 0; b < batch; ++b)
      jobs.push_back({codes + (size_t)b * frames * 16, frames, pcm_out + (size_t)b * frames * up, 0, (int64_t)frames * up});
    run_decode_jobs(h, jobs);
    tm.finish();
  });
}

q3tts_status q3tts_decode_chunked(q3tts_handle* h, const int32_t* codes, int32_t batch, int32_t frames, int32_t chunk_size,
                                  int32_t left_context, float* pcm_out) {
  return guarded(h, [&] {
    Q3_CHECK(h->codec != nullptr, Q3TTS_ERR_DECODER_LOAD_FAILED, "Failed to load MLX audio decoder");
    Q3_CHECK(codes && pcm_out && batch >= 0 && frames >= 0 && chunk_size > 0 && left_context >= 0, Q3TTS_ERR_INVALID_ARG, "bad arguments");
    CallTimer tm(h);
    const int up = h->codec->total_upsample();
    // chunkedDecode (Vocoder/SpeechTokenizer.swift:954-987): left-pad with code 0 x left_context, right-pad to a multiple of
    // chunk_size, windows of chunk_size + left_context stacked on the batch axis, drop the context samples, trim to T*up.
    const int n_chunks = (frames + chunk_size - 1) / chunk_size;
    const int Lw = chunk_size + left_context;
    std::vector<int32_t> win((size_t)batch * n_chunks * Lw * 16, 0);
    std::vector<DecodeJob> jobs;
    for (int b = 0; b < batch; ++b)
      for (int ci = 0; ci < n_chunks; ++ci) {
        int32_t* w = win.data() + ((size_t)b * n_chunks + ci) * Lw * 16;
        for (int p = 0; p < Lw; ++p) {
          const int src = ci * chunk_size + p - left_context;
          if (src >= 0 && src < frames) memcpy(w + (size_t)p * 16, codes + ((size_t)b * frames + src) * 16, 64);
        }
        const int64_t o0 = (int64_t)ci * chunk_size * up;
        jobs.push_back({w, Lw, pcm_out + (size_t)b * frames * up + o0, (int64_t)left_context * up,
                        std::min<int64_t>((int64_t)chunk_size * up, (int64_t)frames * up - o0)});
      }
    run_decode_jobs(h, jobs);
    tm.finish();
  });
}

// =================================================================================================== ICL reference-audio encoder
q3tts_status q3tts_encode_reference_audio(q3tts_handle* h, const float* samples, int64_t n_samples, int32_t* codes_out, int32_t capacity_frames,
                                          int32_t* frames_out, int32_t* quantizers_out, float* latent_out) {
  return guarded(h, [&] {
    Q3_CHECK(frames_out != nullptr, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    *frames_out = 0;
    if (quantizers_out) *quantizers_out = 0;
    if (!h->audio_encoder) return;  // encodeReferenceAudio returns nil without an encoder (Qwen3TTSPipeline.swift:925)
    Q3_CHECK(samples != nullptr && n_samples > 0 && codes_out != nullptr, Q3TTS_ERR_INVALID_ARG, "bad arguments");
    CallTimer tm(h);
    const int f = h->audio_encoder->encode(samples, n_samples, codes_out, capacity_frames, latent_out);
    *frames_out = f;
    if (quantizers_out) *quantizers_out = h->audio_encoder->quantizers_out();
    h->timing.h2d_bytes += n_samples * 4;
    h->timing.d2h_bytes += (int64_t)f * h->audio_encoder->quantizers_out() * 4;
    tm.finish();
  });
}

q3tts_status q3tts_extract_speaker_embedding(q3tts_handle* h, const float* samples, int64_t n_samples, float* embedding_out, int32_t capacity,
                                             int32_t* dim_out, float* mels_out) {
  return guarded(h, [&] {
    Q3_CHECK(dim_out != nullptr, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    *dim_out = 0;
    if (!h->speaker_encoder) return;  // extractSpeakerEmbedding returns nil without the weights (Qwen3TTSPipeline.swift:907-909)
    Q3_CHECK(samples != nullptr && n_samples > 0 && embedding_out != nullptr, Q3TTS_ERR_INVALID_ARG, "bad arguments");
    Q3_CHECK(capacity >= h->speaker_encoder->embedding_dim(), Q3TTS_ERR_CAPACITY, "embedding buffer holds %d floats, the speaker embedding has %d", capacity,
             h->speaker_encoder->embedding_dim());
    CallTimer tm(h);
    h->speaker_encoder->extract(samples, n_samples, embedding_out, mels_out);
    *dim_out = h->speaker_encoder->embedding_dim();
    h->timing.h2d_bytes += n_samples * 4;
    h->timing.d2h_bytes += (int64_t)*dim_out * 4;
    tm.finish();
  });
}

// =================================================================================================== fused text -> PCM
q3tts_status q3tts_generate_pcm(q3tts_handle* h, const q3tts_request* req, int32_t mode, float* pcm_out, int64_t capacity_samples,
                                int64_t* samples_out, int32_t* frames_out) {
  return guarded(h, [&] {
    Q3_CHECK(req && pcm_out && samples_out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(h->talker != nullptr, Q3TTS_ERR_MODEL_NOT_LOADED, "Model is not loaded");
    require_no_open_stream(h);
    Q3_CHECK(h->codec != nullptr, Q3TTS_ERR_DECODER_LOAD_FAILED, "Failed to load MLX audio decoder");
    check_voices(h, req, 1);
    *samples_out = 0;
    if (frames_out) *frames_out = 0;
    CallTimer tm(h);
    std::vector<int32_t> raw;
    int n_raw = 0;
    run_single(h, *req, raw, n_raw);
    std::vector<int32_t> valid((size_t)std::max(n_raw, 1) * 16);
    q3tts_request r = *req;
    r.keep_invalid_frames = 0;
    const int n = filter_frames(r, raw, n_raw, valid.data(), n_raw);
    std::vector<DecodeJob> jobs;
    const int64_t total = plan_decode(mode, valid.data(), n, pcm_out, capacity_samples, h->codec->total_upsample(), jobs);
    run_decode_jobs(h, jobs);
    *samples_out = total;
    if (frames_out) *frames_out = n;
    h->timing.h2d_bytes += (int64_t)req->n_text_ids * 4;
    tm.finish();
  });
}

static q3tts_status generate_pcm_batch_one(q3tts_handle* h, const q3tts_request* reqs, int32_t n, int32_t mode, float* const* pcm_out,
                                           int64_t capacity_samples, int64_t* samples_out, int32_t* frames_out) {
  return guarded(h, [&] {
    Q3_CHECK(reqs && pcm_out && samples_out && n >= 0, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(h->talker != nullptr, Q3TTS_ERR_MODEL_NOT_LOADED, "Model is not loaded");
    require_no_open_stream(h);
    Q3_CHECK(h->codec != nullptr, Q3TTS_ERR_DECODER_LOAD_FAILED, "Failed to load MLX audio decoder");
    check_voices(h, reqs, n);
    CallTimer tm(h);
    static const bool host_trace = getenv("Q3TTS_HOST_TRACE") != nullptr;  // wall-clock phases of this call on stderr
    const auto w0 = std::chrono::steady_clock::now();
    std::vector<std::vector<int32_t>> raw;
    std::vector<int> n_raw;
    run_batch(h, reqs, n, raw, n_raw);
    const auto w1 = std::chrono::steady_clock::now();
    std::vector<std::vector<int32_t>> valid(n);
    std::vector<DecodeJob> jobs;
    std::vector<int64_t> totals(n, 0);
    for (int i = 0; i < n; ++i) {
      valid[i].resize((size_t)std::max(n_raw[i], 1) * 16);
      q3tts_request r = reqs[i];
      r.keep_invalid_frames = 0;
      const int nv = filter_frames(r, raw[i], n_raw[i], valid[i].data(), n_raw[i]);
      if (frames_out) frames_out[i] = nv;
      totals[i] = plan_decode(mode, valid[i].data(), nv, pcm_out[i], capacity_samples, h->codec->total_upsample(), jobs);
      h->timing.h2d_bytes += (int64_t)reqs[i].n_text_ids * 4;
    }
    const auto w2 = std::chrono::steady_clock::now();
    run_decode_jobs(h, jobs);
    const auto w3 = std::chrono::steady_clock::now();
    for (int i = 0; i < n; ++i) samples_out[i] = totals[i];
    tm.finish();
    if (host_trace) {
      auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
      fprintf(stderr, "[q3tts host] generate_pcm_batch n=%d: talker loop %.1f ms (device %.1f), plan %.1f ms, decode jobs %.1f ms (device %.1f)\n", n,
              ms(w0, w1), h->timing.talker_ms, ms(w1, w2), ms(w2, w3), h->timing.decode_ms);
    }
  });
}

q3tts_status q3tts_generate_pcm_batch(q3tts_handle* h, const q3tts_request* reqs, int32_t n, int32_t mode, float* const* pcm_out,
                                      int64_t capacity_samples, int64_t* samples_out, int32_t* frames_out) {
  if (!use_lanes(h, reqs, n) || !pcm_out || !samples_out) return generate_pcm_batch_one(h, reqs, n, mode, pcm_out, capacity_samples, samples_out, frames_out);
  const q3tts_status st = guarded(h, [&] { check_voices(h, reqs, n); });
  if (st != Q3TTS_OK) return st;
  return over_lanes(h, n, [&](q3tts_handle* lane, int off, int cnt) {
    return generate_pcm_batch_one(lane, reqs + off, cnt, mode, pcm_out + off, capacity_samples, samples_out + off, frames_out ? frames_out + off : nullptr);
  });
}

// =================================================================================================== parity probes
namespace {

// The widths and groups the packed probes take, checked on the host before any device is touched.  The container's words must not
// straddle a group (group % codes-per-word); 2 / 3 / 5 / 6-bit rows must be whole words (in % 32) and use MLX's groups.
void check_packed_args(int out_f, int in_f, int group, int bits) {
  const int cbits = container_bits(bits);
  Q3_CHECK(cbits != 0, Q3TTS_ERR_INVALID_ARG, "bits %d: 2, 3, 4, 5, 6 or 8 are supported", bits);
  Q3_CHECK(out_f > 0 && in_f > 0 && group > 0 && in_f % group == 0 && group % (32 / cbits) == 0, Q3TTS_ERR_INVALID_ARG,
           "unsupported bits/group/shape (%d/%d, %d x %d)", bits, group, out_f, in_f);
  if (cbits != bits)
    Q3_CHECK((group == 32 || group == 64 || group == 128) && in_f % 32 == 0, Q3TTS_ERR_INVALID_ARG,
             "%d-bit rows need group_size 32, 64 or 128 and in_features %% 32 == 0 (group %d, in %d)", bits, group, in_f);
}

// `packed` ([out_f][in_f * bits / 32] uint32 on the host) on the device in the container_bits(bits) word layout the kernels read.
const uint32_t* upload_packed(const uint32_t* packed, int out_f, int in_f, int bits, std::vector<void*>& allocs) {
  auto dev = [&](size_t bytes) -> void* {
    void* d = nullptr;
    Q3_CUDA(cudaMalloc(&d, bytes));
    allocs.push_back(d);
    return d;
  };
  const int cbits = container_bits(bits);
  void* raw = dev((size_t)out_f * in_f * bits / 8);
  Q3_CUDA(cudaMemcpy(raw, packed, (size_t)out_f * in_f * bits / 8, cudaMemcpyHostToDevice));
  if (cbits == bits) return (const uint32_t*)raw;
  uint32_t* wide = (uint32_t*)dev((size_t)out_f * in_f * cbits / 8);
  LaunchCtx c{nullptr, nullptr};
  launch_widen_bits(c, (const uint32_t*)raw, out_f, in_f, bits, wide);
  return wide;
}

}  // namespace

q3tts_status q3tts_dequantize(int32_t device, const uint32_t* packed, const void* scales, const void* biases, int32_t scale_dtype,
                              int32_t out_f, int32_t in_f, int32_t group, int32_t bits, int32_t out_dtype, void* out) {
  std::vector<void*> allocs;
  try {
    Q3_CHECK(packed && scales && biases && out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    check_packed_args(out_f, in_f, group, bits);
    require_device(device);
    const size_t sbytes = (size_t)out_f * (in_f / group) * dtype_size(scale_dtype);
    const size_t obytes = (size_t)out_f * in_f * dtype_size(out_dtype);
    const uint32_t* dw = upload_packed(packed, out_f, in_f, bits, allocs);
    void *ds = nullptr, *db = nullptr, *dout = nullptr;
    Q3_CUDA(cudaMalloc(&ds, sbytes)); allocs.push_back(ds);
    Q3_CUDA(cudaMalloc(&db, sbytes)); allocs.push_back(db);
    Q3_CUDA(cudaMalloc(&dout, obytes)); allocs.push_back(dout);
    Q3_CUDA(cudaMemcpy(ds, scales, sbytes, cudaMemcpyHostToDevice));
    Q3_CUDA(cudaMemcpy(db, biases, sbytes, cudaMemcpyHostToDevice));
    LaunchCtx c{nullptr, nullptr};
    launch_dequantize(c, dw, ds, db, scale_dtype, out_f, in_f, group, container_bits(bits), out_dtype, dout);
    Q3_CUDA(cudaDeviceSynchronize());
    Q3_CUDA(cudaMemcpy(out, dout, obytes, cudaMemcpyDeviceToHost));
    for (void* d : allocs) cudaFree(d);
    return Q3TTS_OK;
  } catch (const Error& e) {
    for (void* d : allocs) cudaFree(d);
    g_create_error = e.what();
    cudaGetLastError();
    return e.status;
  }
}

q3tts_status q3tts_mlx_quantize(int32_t device, const void* w, int32_t w_dtype, int32_t out_f, int32_t in_f, int32_t bits, uint32_t* codes8_out,
                                void* scales_out, void* biases_out) {
  try {
    Q3_CHECK(w && codes8_out && scales_out && biases_out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK((bits == 4 || bits == 6 || bits == 8) && in_f > 0 && in_f % 64 == 0 && out_f > 0, Q3TTS_ERR_INVALID_ARG, "unsupported bits / shape (%d, %d x %d)", bits,
             out_f, in_f);
    require_device(device);
    const size_t wbytes = (size_t)out_f * in_f * dtype_size(w_dtype), gbytes = (size_t)out_f * (in_f / 64) * dtype_size(w_dtype), cbytes = (size_t)out_f * in_f;
    void *dw = nullptr, *ds = nullptr, *db = nullptr, *dc = nullptr;
    Q3_CUDA(cudaMalloc(&dw, wbytes)); Q3_CUDA(cudaMalloc(&ds, gbytes)); Q3_CUDA(cudaMalloc(&db, gbytes)); Q3_CUDA(cudaMalloc(&dc, cbytes));
    Q3_CUDA(cudaMemcpy(dw, w, wbytes, cudaMemcpyHostToDevice));
    LaunchCtx c{nullptr, nullptr};
    launch_mlx_quantize(c, dw, w_dtype, out_f, in_f, bits, (uint32_t*)dc, ds, db, nullptr);
    Q3_CUDA(cudaDeviceSynchronize());
    Q3_CUDA(cudaMemcpy(codes8_out, dc, cbytes, cudaMemcpyDeviceToHost));
    Q3_CUDA(cudaMemcpy(scales_out, ds, gbytes, cudaMemcpyDeviceToHost));
    Q3_CUDA(cudaMemcpy(biases_out, db, gbytes, cudaMemcpyDeviceToHost));
    cudaFree(dw); cudaFree(ds); cudaFree(db); cudaFree(dc);
    return Q3TTS_OK;
  } catch (const Error& e) {
    g_create_error = e.what();
    cudaGetLastError();
    return e.status;
  }
}

q3tts_status q3tts_mxfp4_to_affine(int32_t device, const uint32_t* packed, const uint8_t* scales, int32_t out_f, int32_t in_f, uint32_t* codes8_out,
                                   void* scales_out, void* biases_out) {
  std::vector<void*> allocs;
  try {
    Q3_CHECK(packed && scales && codes8_out && scales_out && biases_out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(out_f > 0 && in_f > 0 && in_f % 32 == 0, Q3TTS_ERR_INVALID_ARG, "unsupported shape %d x %d (in_features a multiple of 32)", out_f, in_f);
    const size_t wbytes = (size_t)out_f * in_f / 2, groups = (size_t)out_f * (in_f / 32), cbytes = (size_t)out_f * in_f;
    for (size_t k = 0; k < groups; ++k)
      Q3_CHECK(scales[k] <= kMxfp4MaxScaleByte, Q3TTS_ERR_INVALID_ARG, "scale byte %d at index %zu: bytes 0..%d fit the container", (int)scales[k], k,
               kMxfp4MaxScaleByte);
    require_device(device);
    auto dev = [&](const void* src, size_t bytes) -> void* {
      void* d = nullptr;
      Q3_CUDA(cudaMalloc(&d, bytes));
      allocs.push_back(d);
      if (src) Q3_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
      return d;
    };
    const uint32_t* dw = (const uint32_t*)dev(packed, wbytes);
    const uint8_t* ds = (const uint8_t*)dev(scales, groups);
    uint32_t* dc = (uint32_t*)dev(nullptr, cbytes);
    uint16_t* dsc = (uint16_t*)dev(nullptr, groups * 2);
    uint16_t* dbi = (uint16_t*)dev(nullptr, groups * 2);
    LaunchCtx c{nullptr, nullptr};
    launch_mxfp4_to_affine(c, dw, ds, out_f, in_f, dc, dsc, dbi);
    Q3_CUDA(cudaDeviceSynchronize());
    Q3_CUDA(cudaMemcpy(codes8_out, dc, cbytes, cudaMemcpyDeviceToHost));
    Q3_CUDA(cudaMemcpy(scales_out, dsc, groups * 2, cudaMemcpyDeviceToHost));
    Q3_CUDA(cudaMemcpy(biases_out, dbi, groups * 2, cudaMemcpyDeviceToHost));
    for (void* d : allocs) cudaFree(d);
    return Q3TTS_OK;
  } catch (const Error& e) {
    for (void* d : allocs) cudaFree(d);
    g_create_error = e.what();
    cudaGetLastError();
    return e.status;
  }
}

q3tts_status q3tts_quantized_matmul(int32_t device, const float* x, int32_t m, const uint32_t* packed, const void* scales,
                                    const void* biases, int32_t scale_dtype, int32_t out_f, int32_t in_f, int32_t group,
                                    int32_t bits, float* y) {
  std::vector<void*> allocs;
  try {
    Q3_CHECK(x && packed && y && m > 0, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    if (bits) {
      Q3_CHECK(scales && biases, Q3TTS_ERR_INVALID_ARG, "NULL scales/biases");
      check_packed_args(out_f, in_f, group, bits);
    }
    require_device(device);
    q3::init_talker_kernels();
    Linear L;
    L.out = out_f; L.in = in_f; L.bits = container_bits(bits); L.group = group; L.sdt = scale_dtype;
    auto dev = [&](const void* src, size_t bytes) -> void* {
      void* d = nullptr;
      Q3_CUDA(cudaMalloc(&d, bytes));
      allocs.push_back(d);
      if (src) Q3_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
      return d;
    };
    if (bits) {
      const size_t sbytes = (size_t)out_f * (in_f / group) * dtype_size(scale_dtype);
      L.qw = upload_packed(packed, out_f, in_f, bits, allocs); L.scales = dev(scales, sbytes); L.biases = dev(biases, sbytes);
    } else {
      L.w = dev(packed, (size_t)out_f * in_f * dtype_size(scale_dtype));
    }
    float* dx = (float*)dev(x, (size_t)m * in_f * 4);
    float* dy = (float*)dev(nullptr, (size_t)m * out_f * 4);
    LaunchCtx c{nullptr, nullptr};
    launch_linear(c, L, dx, in_f, m, dy, out_f, nullptr, 0.f, EPI_STORE);
    Q3_CUDA(cudaDeviceSynchronize());
    Q3_CUDA(cudaMemcpy(y, dy, (size_t)m * out_f * 4, cudaMemcpyDeviceToHost));
    for (void* d : allocs) cudaFree(d);
    return Q3TTS_OK;
  } catch (const Error& e) {
    for (void* d : allocs) cudaFree(d);
    g_create_error = e.what();
    cudaGetLastError();
    return e.status;
  }
}

q3tts_status q3tts_quantized_matmul_tc(int32_t device, const float* x, int32_t m, const uint32_t* packed, const void* scales, const void* biases,
                                       int32_t scale_dtype, int32_t out_f, int32_t in_f, int32_t group, int32_t bits, const float* fold,
                                       int32_t swiglu_halves, const float* residual, float* y) {
  std::vector<void*> allocs;
  try {
    Q3_CHECK(x && packed && scales && biases && y && m > 0 && m <= 128, Q3TTS_ERR_INVALID_ARG, "bad arguments (1 <= m <= 128)");
    check_packed_args(out_f, in_f, group, bits);
    require_device(device);
    init_tc_gemm();
    const int n_out = swiglu_halves ? out_f / 2 : out_f;
    const size_t sbytes = (size_t)out_f * (in_f / group) * dtype_size(scale_dtype);
    auto dev = [&](const void* src, size_t bytes) -> void* {
      void* d = nullptr;
      Q3_CUDA(cudaMalloc(&d, std::max<size_t>(bytes, 16)));
      allocs.push_back(d);
      if (src) Q3_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
      return d;
    };
    const void* dw = upload_packed(packed, out_f, in_f, bits, allocs);
    void *ds = dev(scales, sbytes), *db = dev(biases, sbytes);
    float* dx = (float*)dev(x, (size_t)m * in_f * 4);
    float* dfold = fold ? (float*)dev(fold, (size_t)in_f * 4) : nullptr;
    float* dy = (float*)dev(residual, (size_t)m * n_out * 4);
    if (!residual) Q3_CUDA(cudaMemset(dy, 0, (size_t)m * n_out * 4));
    __half* dx16 = (__half*)dev(nullptr, (size_t)m * in_f * 2);
    LaunchCtx c{nullptr, nullptr};
    Q3_CHECK(((size_t)m * in_f) % 4 == 0, Q3TTS_ERR_INVALID_ARG, "m * in_features must be divisible by 4");
    launch_f32_to_f16(c, dx, (size_t)m * in_f, dx16);
    Q3_CUDA(cudaDeviceSynchronize());
    TcGemm g;
    g.a = dx16; g.Bt = 1; g.T = m; g.cin = in_f; g.N = out_f; g.swiglu = swiglu_halves ? 1 : 0;
    g.q_w = (const uint32_t*)dw; g.q_scales = ds; g.q_biases = db; g.q_fold = dfold; g.q_bits = container_bits(bits); g.q_group = group;
    g.q_sdt = scale_dtype;
    g.q_halves = swiglu_halves ? 1 : 0;
    g.out32 = dy; g.ld32 = n_out;
    if (residual) { g.res = dy; g.ld_res = n_out; }
    Q3_CHECK(tc_skinny_q_supported(g), Q3TTS_ERR_INVALID_ARG, "shape not supported by the dequant-fused tensor-core GEMM");
    launch_tc_skinny_q(c, g);
    Q3_CUDA(cudaDeviceSynchronize());
    Q3_CUDA(cudaMemcpy(y, dy, (size_t)m * n_out * 4, cudaMemcpyDeviceToHost));
    for (void* d : allocs) cudaFree(d);
    return Q3TTS_OK;
  } catch (const Error& e) {
    for (void* d : allocs) cudaFree(d);
    g_create_error = e.what();
    cudaGetLastError();
    return e.status;
  }
}

q3tts_status q3tts_safetensors_check(const char* path, int32_t* n_tensors_out, int64_t* data_bytes_out) {
  try {
    Q3_CHECK(path != nullptr, Q3TTS_ERR_INVALID_ARG, "path is NULL");
    SafeTensors st(path);
    int64_t bytes = 0;
    for (auto& kv : st.tensors()) bytes += (int64_t)kv.second.nbytes;
    if (n_tensors_out) *n_tensors_out = (int32_t)st.tensors().size();
    if (data_bytes_out) *data_bytes_out = bytes;
    return Q3TTS_OK;
  } catch (const Error& e) {
    g_create_error = e.what();
    return e.status;
  } catch (const std::exception& e) {
    g_create_error = e.what();
    return Q3TTS_ERR_BAD_WEIGHTS;
  }
}

q3tts_status q3tts_conv_probe(int32_t device, const float* x, int32_t B, int32_t T, int32_t cin, const float* w, const float* bias, int32_t N,
                              int32_t ntap, int32_t dil, int32_t act, int32_t swiglu, const float* res, const float* scale,
                              const float* snake_ea, const float* snake_ieb, int32_t snake_ch, int32_t use_tc, float* y32, float* y16) {
  std::vector<void*> allocs;
  try {
    Q3_CHECK(x && w && B > 0 && T > 0 && cin > 0 && N > 0 && ntap > 0 && dil > 0, Q3TTS_ERR_INVALID_ARG, "bad arguments");
    require_device(device);
    const size_t M = (size_t)B * T, nx = M * cin, nw = (size_t)ntap * N * cin, n_out = swiglu ? N / 2 : N, ny = M * n_out;
    auto dev = [&](const void* src, size_t bytes) -> void* {
      void* d = nullptr;
      Q3_CUDA(cudaMalloc(&d, std::max<size_t>(bytes, 16)));
      allocs.push_back(d);
      if (src) Q3_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
      return d;
    };
    float* dx = (float*)dev(x, nx * 4);
    float* dw = (float*)dev(w, nw * 4);
    float* dbias = bias ? (float*)dev(bias, (size_t)N * 4) : nullptr;
    float* dres = res ? (float*)dev(res, ny * 4) : nullptr;
    float* dscale = scale ? (float*)dev(scale, n_out * 4) : nullptr;
    float* dea = snake_ea ? (float*)dev(snake_ea, (size_t)snake_ch * 4) : nullptr;
    float* dieb = snake_ieb ? (float*)dev(snake_ieb, (size_t)snake_ch * 4) : nullptr;
    float* dy32 = (float*)dev(nullptr, ny * 4);
    __half* dy16 = (__half*)dev(nullptr, ny * 2);
    Q3_CUDA(cudaMemset(dy32, 0, ny * 4));
    Q3_CUDA(cudaMemset(dy16, 0, ny * 2));
    LaunchCtx c{nullptr, nullptr};
    if (use_tc) {
      init_tc_gemm();
      __half* dx16 = (__half*)dev(nullptr, nx * 2);
      __half* dw16 = (__half*)dev(nullptr, nw * 2);
      Q3_CHECK(nx % 4 == 0 && nw % 4 == 0, Q3TTS_ERR_INVALID_ARG, "probe needs element counts divisible by 4");
      launch_f32_to_f16(c, dx, nx, dx16);
      launch_f32_to_f16(c, dw, nw, dw16);
      // the GEMM kernels request WEIGHT tiles before their programmatic dependency resolves (weights are static in the engine):
      // here the weights come from the launch just above, so it must have retired first
      Q3_CUDA(cudaDeviceSynchronize());
      TcGemm g;
      g.a = dx16; g.w = dw16; g.Bt = B; g.T = T; g.cin = cin; g.N = N; g.ntap = ntap; g.dil = dil;
      g.bias = dbias; g.res = dres; g.ld_res = (int)n_out; g.scale = dscale; g.act = act; g.swiglu = swiglu;
      g.out32 = dy32; g.ld32 = (int)n_out; g.out16 = dy16; g.ld16 = (int)n_out;
      g.snake_ea = dea; g.snake_ieb = dieb; g.snake_ch = snake_ch;
      Q3_CHECK(tc_gemm_supported(g), Q3TTS_ERR_INVALID_ARG, "shape not supported by the tcgen05 path (cin %% 8, N %% 32)");
      launch_tc_gemm(c, g);
    } else {
      Q3_CHECK(!swiglu && !snake_ea, Q3TTS_ERR_INVALID_ARG, "SIMT probe supports bias/act(gelu)/res/scale only");
      ConvW cw;
      cw.w = dw; cw.bias = dbias; cw.ntap = ntap; cw.dil = dil; cw.cin = cin; cw.n = N;
      launch_conv_gemm(c, dx, cw, dy32, dres, dscale, (int)M, T, res ? CE_RES_SCALE : (act == 1 ? CE_GELU : CE_STORE));
    }
    Q3_CUDA(cudaDeviceSynchronize());
    if (y32) Q3_CUDA(cudaMemcpy(y32, dy32, ny * 4, cudaMemcpyDeviceToHost));
    if (y16) {
      std::vector<uint16_t> h(ny);
      Q3_CUDA(cudaMemcpy(h.data(), dy16, ny * 2, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < ny; ++i) y16[i] = f16_to_f32(h[i]);
    }
    for (void* d : allocs) cudaFree(d);
    return Q3TTS_OK;
  } catch (const Error& e) {
    for (void* d : allocs) cudaFree(d);
    g_create_error = e.what();
    cudaGetLastError();
    return e.status;
  }
}

q3tts_status q3tts_attention_probe(int32_t device, int32_t kernel, int32_t kv_f16, int32_t out_f16, const float* qkv, int32_t m,
                                   int32_t heads, int32_t kv_heads, const float* q_norm, const float* k_norm, float eps,
                                   const float* inv_freq, const int32_t* row_slot, const int32_t* row_pos, const int32_t* win_start,
                                   int32_t n_slots, int32_t capacity, float* k_ring, float* v_ring, float* out) {
  std::vector<void*> allocs;
  try {
    // every index a kernel derives from these arguments is checked here, so no input can make a launch read or write outside
    // its buffers
    Q3_CHECK(qkv && q_norm && k_norm && inv_freq && row_slot && row_pos && k_ring && v_ring && out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(kernel >= 0 && kernel <= 2, Q3TTS_ERR_INVALID_ARG, "kernel must be 0, 1 or 2");
    Q3_CHECK(m > 0 && n_slots > 0 && capacity > 0 && kv_heads > 0 && heads > 0 && heads % kv_heads == 0, Q3TTS_ERR_INVALID_ARG,
             "bad sizes (m %d, n_slots %d, capacity %d, heads %d, kv_heads %d)", m, n_slots, capacity, heads, kv_heads);
    const int G = heads / kv_heads;
    Q3_CHECK(G == 1 || G == 2 || G == 4, Q3TTS_ERR_INVALID_ARG, "GQA group %d not in {1, 2, 4}", G);
    const size_t ring_elems = (size_t)n_slots * kv_heads * capacity * 128;
    Q3_CHECK(ring_elems < ((size_t)1 << 31) && (size_t)m * (heads + 2 * kv_heads) * 128 < ((size_t)1 << 31), Q3TTS_ERR_INVALID_ARG, "buffers too large");
    std::vector<int> rows_of_slot(n_slots, 0);
    for (int r = 0; r < m; ++r) {
      const int s = row_slot[r], p = row_pos[r];
      Q3_CHECK(s >= 0 && s < n_slots, Q3TTS_ERR_INVALID_ARG, "row %d: slot %d out of range", r, s);
      const int w = win_start ? win_start[s] : 0;
      Q3_CHECK(w >= 0 && w <= p && p - w + 1 <= capacity, Q3TTS_ERR_INVALID_ARG, "row %d: window [%d, %d] does not fit a ring of %d", r, w, p, capacity);
      ++rows_of_slot[s];
    }
    if (kernel == 0)
      for (int s = 0; s < n_slots; ++s) Q3_CHECK(rows_of_slot[s] <= 1, Q3TTS_ERR_INVALID_ARG, "kernel 0 takes at most one row per slot");
    if (kernel == 1)  // rows of one slot append at distinct ring indices (their windows fit the ring, so distinct positions suffice)
      for (int a = 0; a < m; ++a)
        for (int b = a + 1; b < m; ++b)
          Q3_CHECK(row_slot[a] != row_slot[b] || row_pos[a] != row_pos[b], Q3TTS_ERR_INVALID_ARG, "rows %d and %d share slot and position", a, b);
    if (kernel == 2) {
      Q3_CHECK(m == 2 * n_slots && !kv_f16 && out_f16 && capacity >= 2, Q3TTS_ERR_INVALID_ARG,
               "kernel 2 takes rows (2s, 2s+1) of every slot, an fp32 cache of >= 2 positions and fp16 output");
      for (int r = 0; r < m; ++r)
        Q3_CHECK(row_slot[r] == r / 2 && row_pos[r] == r % 2 && (!win_start || win_start[r / 2] == 0), Q3TTS_ERR_INVALID_ARG,
                 "kernel 2: row %d must be slot %d at position %d", r, r / 2, r % 2);
    }
    require_device(device);
    init_talker_kernels();
    auto dev = [&](const void* src, size_t bytes) -> void* {
      void* d = nullptr;
      Q3_CUDA(cudaMalloc(&d, std::max<size_t>(bytes, 16)));
      allocs.push_back(d);
      if (src) Q3_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
      return d;
    };
    const int ld = (heads + 2 * kv_heads) * 128, ldo = heads * 128;
    float* dqkv = (float*)dev(qkv, (size_t)m * ld * 4);
    const float* dqn = (const float*)dev(q_norm, 128 * 4);
    const float* dkn = (const float*)dev(k_norm, 128 * 4);
    const float* dfreq = (const float*)dev(inv_freq, 64 * 4);
    const int* dslot = (const int*)dev(row_slot, (size_t)m * 4);
    const int* dpos = (const int*)dev(row_pos, (size_t)m * 4);
    const int* dwin = win_start ? (const int*)dev(win_start, (size_t)n_slots * 4) : nullptr;
    KVLayout kv;
    kv.slot_stride = (size_t)kv_heads * capacity * 128;
    kv.capacity = capacity;
    kv.f16 = kv_f16 ? 1 : 0;
    std::vector<__half> h16;
    if (kv.f16) {
      h16.resize(ring_elems);
      for (size_t i = 0; i < ring_elems; ++i) h16[i] = __float2half_rn(k_ring[i]);
      kv.k = dev(h16.data(), ring_elems * 2);
      for (size_t i = 0; i < ring_elems; ++i) h16[i] = __float2half_rn(v_ring[i]);
      kv.v = dev(h16.data(), ring_elems * 2);
    } else {
      kv.k = dev(k_ring, ring_elems * 4);
      kv.v = dev(v_ring, ring_elems * 4);
    }
    void* dout = dev(nullptr, (size_t)m * ldo * (out_f16 ? 2 : 4));
    Q3_CUDA(cudaMemset(dout, 0, (size_t)m * ldo * (out_f16 ? 2 : 4)));
    LaunchCtx c{nullptr, nullptr};
    if (kernel == 0) {
      if (out_f16) launch_rope_attention_f16(c, dqkv, ld, m, heads, kv_heads, dqn, dkn, eps, dfreq, dslot, dpos, dwin, kv, (__half*)dout, ldo);
      else launch_rope_attention(c, dqkv, ld, m, heads, kv_heads, dqn, dkn, eps, dfreq, dslot, dpos, dwin, kv, (float*)dout, ldo);
    } else if (kernel == 1) {
      launch_qk_norm_rope_append(c, dqkv, ld, m, heads, kv_heads, 128, dqn, dkn, eps, dfreq, dslot, dpos, kv);
      if (out_f16) launch_attention_f16(c, dqkv, ld, m, heads, kv_heads, 128, dslot, dpos, dwin, kv, (__half*)dout, ldo);
      else launch_attention(c, dqkv, ld, m, heads, kv_heads, 128, dslot, dpos, dwin, kv, (float*)dout, ldo);
    } else {
      launch_cp_pass0_attention_f16(c, dqkv, ld, n_slots, heads, kv_heads, dqn, dkn, eps, dfreq, kv, (__half*)dout, ldo);
    }
    Q3_CUDA(cudaGetLastError());
    Q3_CUDA(cudaDeviceSynchronize());
    if (kv.f16) {
      Q3_CUDA(cudaMemcpy(h16.data(), kv.k, ring_elems * 2, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < ring_elems; ++i) k_ring[i] = __half2float(h16[i]);
      Q3_CUDA(cudaMemcpy(h16.data(), kv.v, ring_elems * 2, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < ring_elems; ++i) v_ring[i] = __half2float(h16[i]);
    } else {
      Q3_CUDA(cudaMemcpy(k_ring, kv.k, ring_elems * 4, cudaMemcpyDeviceToHost));
      Q3_CUDA(cudaMemcpy(v_ring, kv.v, ring_elems * 4, cudaMemcpyDeviceToHost));
    }
    if (out_f16) {
      std::vector<__half> o((size_t)m * ldo);
      Q3_CUDA(cudaMemcpy(o.data(), dout, o.size() * 2, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < o.size(); ++i) out[i] = __half2float(o[i]);
    } else {
      Q3_CUDA(cudaMemcpy(out, dout, (size_t)m * ldo * 4, cudaMemcpyDeviceToHost));
    }
    for (void* d : allocs) cudaFree(d);
    return Q3TTS_OK;
  } catch (const Error& e) {
    for (void* d : allocs) cudaFree(d);
    g_create_error = e.what();
    cudaGetLastError();
    return e.status;
  }
}

// ------------------------------------------------------------------------------------------------ codec kernel probes
namespace {
// device copies of a probe's host buffers; every allocation is freed when the probe returns, on every path
struct ProbeBuffers {
  std::vector<void*> allocs;
  ProbeBuffers() = default;
  ProbeBuffers(const ProbeBuffers&) = delete;
  ProbeBuffers& operator=(const ProbeBuffers&) = delete;
  ~ProbeBuffers() { for (void* d : allocs) cudaFree(d); }
  void* alloc(size_t bytes) {
    void* d = nullptr;
    Q3_CUDA(cudaMalloc(&d, std::max<size_t>(bytes, 16)));
    allocs.push_back(d);
    return d;
  }
  float* f32(const float* src, size_t n) {  // src == null: uninitialised
    float* d = (float*)alloc(n * 4);
    if (src) Q3_CUDA(cudaMemcpy(d, src, n * 4, cudaMemcpyHostToDevice));
    return d;
  }
  // fp16 copy (round to nearest) of n values, `reps` times, f16_rep_stride_bytes(n) apart: the layout of CodecDecoder::upload_f16
  __half* f16(const float* src, size_t n, int reps = 1) {
    std::vector<__half> h(n);
    for (size_t i = 0; i < n; ++i) h[i] = __float2half_rn(src[i]);
    const size_t stride = f16_rep_stride_bytes(n);
    uint8_t* d = (uint8_t*)alloc(stride * (size_t)reps);
    for (int r = 0; r < reps; ++r) Q3_CUDA(cudaMemcpy(d + (size_t)r * stride, h.data(), n * 2, cudaMemcpyHostToDevice));
    return (__half*)d;
  }
};

void widen_f16(const __half* d, size_t n, float* out) {
  std::vector<__half> h(n);
  Q3_CUDA(cudaMemcpy(h.data(), d, n * 2, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; ++i) out[i] = __half2float(h[i]);
}

q3tts_status probe_failed(const Error& e) {
  g_create_error = e.what();
  cudaGetLastError();
  return e.status;
}

constexpr size_t kProbeMaxElems = (size_t)1 << 31;  // every buffer of a probe stays below 2^31 elements (the kernels' int row math)
}  // namespace

q3tts_status q3tts_codec_attention_probe(int32_t device, int32_t kernel, float* qkv, int32_t B, int32_t T, int32_t nh, int32_t nkv,
                                         const float* inv_freq, float* out) {
  ProbeBuffers buf;
  try {
    Q3_CHECK(qkv && out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(kernel >= 0 && kernel <= 3, Q3TTS_ERR_INVALID_ARG, "kernel must be 0, 1, 2 or 3");
    Q3_CHECK(B >= 1 && B <= 64 && T >= 1 && T <= 2400, Q3TTS_ERR_INVALID_ARG, "B %d / T %d outside 1..64 / 1..2400", B, T);
    Q3_CHECK(nkv >= 1 && nh >= 1 && nh <= 64 && nh % nkv == 0, Q3TTS_ERR_INVALID_ARG, "heads %d / kv heads %d (nh <= 64, nh %% nkv == 0)", nh, nkv);
    const int ld = (nh + 2 * nkv) * 64, ldo = nh * 64;
    const size_t M = (size_t)B * T;
    Q3_CHECK(M * ld < kProbeMaxElems, Q3TTS_ERR_INVALID_ARG, "qkv too large");
    require_device(device);
    LaunchCtx c{nullptr, nullptr};
    float* dqkv = buf.f32(qkv, M * ld);
    if (inv_freq) launch_codec_rope(c, dqkv, ld, (int)M, T, nh + nkv, buf.f32(inv_freq, 32));  // q and k heads, in place (decode_pass_*)
    if (kernel == 1 || kernel == 2) {
      float* dout = buf.f32(nullptr, M * ldo);
      Q3_CUDA(cudaMemset(dout, 0x7f, M * ldo * 4));  // an output no launch writes reads as 3.4e38
      if (kernel == 1) launch_codec_attention(c, dqkv, ld, B, T, nh, nkv, dout, ldo);
      else launch_codec_attention_bidir(c, dqkv, ld, B, T, nh, nkv, dout, ldo);
      Q3_CUDA(cudaGetLastError());
      Q3_CUDA(cudaDeviceSynchronize());
      Q3_CUDA(cudaMemcpy(out, dout, M * ldo * 4, cudaMemcpyDeviceToHost));
    } else {
      __half* dout = (__half*)buf.alloc(M * ldo * 2);
      Q3_CUDA(cudaMemset(dout, 0x7f, M * ldo * 2));  // fp16 NaN
      launch_codec_attention_f16(c, dqkv, ld, B, T, nh, nkv, dout, ldo, kernel == 0);
      Q3_CUDA(cudaGetLastError());
      Q3_CUDA(cudaDeviceSynchronize());
      widen_f16(dout, M * ldo, out);
    }
    if (inv_freq) Q3_CUDA(cudaMemcpy(qkv, dqkv, M * ld * 4, cudaMemcpyDeviceToHost));
    return Q3TTS_OK;
  } catch (const Error& e) {
    return probe_failed(e);
  }
}

q3tts_status q3tts_codec_unit_probe(int32_t device, int32_t form, int32_t B, int32_t T, int32_t C, int32_t dil, const float* a,
                                    const float* w7, const float* b7, const float* ea2, const float* ieb2, const float* w1, const float* b1,
                                    const float* res, const float* ea3, const float* ieb3, int32_t in_place, int32_t emit_residual,
                                    int32_t weight_reps, float* x_out, float* snake_out) {
  ProbeBuffers buf;
  try {
    Q3_CHECK(a && w7 && ea2 && ieb2 && w1 && res && ea3 && ieb3 && snake_out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(form == 0 || form == 1, Q3TTS_ERR_INVALID_ARG, "form must be 0 (two GEMM launches) or 1 (fused unit)");
    Q3_CHECK(!in_place || emit_residual, Q3TTS_ERR_INVALID_ARG, "in_place needs emit_residual");
    Q3_CHECK(!emit_residual == !x_out, Q3TTS_ERR_INVALID_ARG, "x_out must be given exactly when emit_residual is set");
    Q3_CHECK(weight_reps >= 1 && weight_reps <= 32, Q3TTS_ERR_INVALID_ARG, "weight_reps %d outside 1..32", weight_reps);
    Q3_CHECK(B >= 1 && T >= 1 && dil >= 1 && dil <= 64 && C >= 32 && C <= 1536 && C % 32 == 0, Q3TTS_ERR_INVALID_ARG,
             "bad shape (B %d, T %d, C %d, dilation %d)", B, T, C, dil);
    const size_t M = (size_t)B * T;
    Q3_CHECK(M * C < kProbeMaxElems, Q3TTS_ERR_INVALID_ARG, "activations too large");
    Q3_CHECK(form == 0 || codec_unit_shape_supported(B, T, C, dil), Q3TTS_ERR_INVALID_ARG,
             "the fused unit does not run C %d, dilation %d, %d x %d rows", C, dil, B, T);
    require_device(device);
    const size_t n7 = (size_t)7 * C * C, n1 = (size_t)C * C;
    const __half* da = buf.f16(a, M * C);
    const __half* dw7 = buf.f16(w7, n7, weight_reps);
    const __half* dw1 = buf.f16(w1, n1, weight_reps);
    const float* db7 = b7 ? buf.f32(b7, C) : nullptr;
    const float* db1 = b1 ? buf.f32(b1, C) : nullptr;
    const float *dea2 = buf.f32(ea2, C), *dieb2 = buf.f32(ieb2, C), *dea3 = buf.f32(ea3, C), *dieb3 = buf.f32(ieb3, C);
    __half* dres = buf.f16(res, M * C);
    __half* doutr = !emit_residual ? nullptr : in_place ? dres : (__half*)buf.alloc(M * C * 2);
    __half* dout = (__half*)buf.alloc(M * C * 2);
    if (doutr && !in_place) Q3_CUDA(cudaMemset(doutr, 0x7f, M * C * 2));  // fp16 NaN where nothing is written
    Q3_CUDA(cudaMemset(dout, 0x7f, M * C * 2));
    LaunchCtx c{nullptr, nullptr};
    if (form == 1) {
      init_codec_unit();
      CodecUnit u;
      u.Bt = B; u.T = T; u.C = C; u.dil = dil;
      u.a = da; u.w7 = dw7; u.b7 = db7; u.snake2_ea = dea2; u.snake2_ieb = dieb2; u.w1 = dw1; u.b1 = db1;
      u.w7_reps = u.w1_reps = weight_reps;
      u.w7_rep_stride = f16_rep_stride_bytes(n7) / 2; u.w1_rep_stride = f16_rep_stride_bytes(n1) / 2;
      u.res16 = dres; u.outr16 = doutr; u.out16 = dout; u.next_ea = dea3; u.next_ieb = dieb3;
      launch_codec_unit(c, u);
    } else {  // what decode_pass_tc launches for a unit the fused kernel does not take
      init_tc_gemm();
      __half* dh = (__half*)buf.alloc(M * C * 2);
      TcGemm g;
      g.a = da; g.w = dw7; g.w_reps = weight_reps; g.w_rep_stride = f16_rep_stride_bytes(n7) / 2;
      g.Bt = B; g.T = T; g.cin = C; g.N = C; g.ntap = 7; g.dil = dil; g.bias = db7;
      g.out16 = dh; g.ld16 = C; g.snake_ea = dea2; g.snake_ieb = dieb2; g.snake_ch = C;
      launch_tc_gemm(c, g);
      TcGemm g2;
      g2.a = dh; g2.w = dw1; g2.w_reps = weight_reps; g2.w_rep_stride = f16_rep_stride_bytes(n1) / 2;
      g2.Bt = B; g2.T = T; g2.cin = C; g2.N = C; g2.bias = db1;
      g2.ld_res = C; g2.ld32 = C; g2.res16 = dres; g2.allow_skinny = 0; g2.outr16 = doutr;
      g2.out16 = dout; g2.ld16 = C; g2.snake_ea = dea3; g2.snake_ieb = dieb3; g2.snake_ch = C;
      launch_tc_gemm(c, g2);
    }
    Q3_CUDA(cudaGetLastError());
    Q3_CUDA(cudaDeviceSynchronize());
    widen_f16(dout, M * C, snake_out);
    if (doutr) widen_f16(doutr, M * C, x_out);
    return Q3TTS_OK;
  } catch (const Error& e) {
    return probe_failed(e);
  }
}

q3tts_status q3tts_codec_out_conv_probe(int32_t device, int32_t kernel, const float* x, int32_t B, int32_t T, int32_t C, const float* w,
                                        const float* bias, int32_t strip, float* y) {
  ProbeBuffers buf;
  try {
    Q3_CHECK(x && w && bias && y, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(kernel >= 0 && kernel <= 3, Q3TTS_ERR_INVALID_ARG, "kernel must be 0, 1, 2 or 3");
    Q3_CHECK(B >= 1 && T >= 1 && C >= 1, Q3TTS_ERR_INVALID_ARG, "bad shape (B %d, T %d, C %d)", B, T, C);
    const size_t M = (size_t)B * T;
    Q3_CHECK(M * C < kProbeMaxElems, Q3TTS_ERR_INVALID_ARG, "activations too large");
    Q3_CHECK(kernel == 0 || strip == 0, Q3TTS_ERR_INVALID_ARG, "strip applies to kernel 0 only");
    if (kernel == 0)
      Q3_CHECK(out_conv_stream_supported(C) && (strip == 0 || (strip >= 32 && strip <= 65536 && strip % 32 == 0)), Q3TTS_ERR_INVALID_ARG,
               "streaming kernel: C %d not in {32, 64, 96, 128} or strip %d not 0 / a multiple of 32 in 32..65536", C, strip);
    if (kernel == 1 || kernel == 2) Q3_CHECK(C <= 256, Q3TTS_ERR_INVALID_ARG, "C %d > 256 (the tile of 134 rows x C lives in shared memory)", C);
    if (kernel == 3) Q3_CHECK(C % 8 == 0 && C <= 1536, Q3TTS_ERR_INVALID_ARG, "tensor-core form: C %d not a multiple of 8 up to 1536", C);
    require_device(device);
    LaunchCtx c{nullptr, nullptr};
    float* dy = buf.f32(nullptr, M);
    Q3_CUDA(cudaMemset(dy, 0x7f, M * 4));  // an output no launch writes reads as 3.4e38, outside the clip range
    if (kernel == 3) {  // the engine's out_tc_: the one output channel padded to 32 columns, [7][32][C] fp16, 8 copies, bias [32]
      init_tc_gemm();
      std::vector<float> wp((size_t)7 * 32 * C, 0.f), bp(32, 0.f);
      for (int k = 0; k < 7; ++k)
        for (int ch = 0; ch < C; ++ch) wp[(size_t)k * 32 * C + ch] = w[(size_t)k * C + ch];
      bp[0] = bias[0];
      const int reps = 8;
      TcGemm g;
      g.a = buf.f16(x, M * C); g.w = buf.f16(wp.data(), wp.size(), reps); g.w_reps = reps; g.w_rep_stride = f16_rep_stride_bytes(wp.size()) / 2;
      g.Bt = B; g.T = T; g.cin = C; g.N = 32; g.ntap = 7; g.dil = 1; g.bias = buf.f32(bp.data(), 32);
      g.pcm = dy;
      launch_tc_gemm(c, g);
    } else {
      init_codec_kernels();
      const float* dw = buf.f32(w, (size_t)7 * C);
      const float* db = buf.f32(bias, 1);
      if (kernel == 0) launch_out_conv_stream_f16(c, buf.f16(x, M * C), dw, db, C, B, T, dy, strip);
      else if (kernel == 1) launch_out_conv(c, buf.f32(x, M * C), dw, db, C, B, T, dy);
      else launch_out_conv_f16(c, buf.f16(x, M * C), dw, db, C, B, T, dy);
    }
    Q3_CUDA(cudaGetLastError());
    Q3_CUDA(cudaDeviceSynchronize());
    Q3_CUDA(cudaMemcpy(y, dy, M * 4, cudaMemcpyDeviceToHost));
    return Q3TTS_OK;
  } catch (const Error& e) {
    return probe_failed(e);
  }
}

q3tts_status q3tts_codec_rowop_probe(int32_t device, int32_t op, const float* x, int32_t rows, int32_t ldx, int32_t C, int32_t T,
                                     const float* w, const float* b, float eps, float* y) {
  ProbeBuffers buf;
  try {
    Q3_CHECK(x && y, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(op >= 0 && op <= 5, Q3TTS_ERR_INVALID_ARG, "op must be 0..5");
    Q3_CHECK(rows >= 1 && C >= 1 && C <= 65536, Q3TTS_ERR_INVALID_ARG, "bad shape (rows %d, C %d)", rows, C);
    Q3_CHECK(op == 3 || op == 5 || w, Q3TTS_ERR_INVALID_ARG, "op %d needs w", op);
    Q3_CHECK(op == 3 || op == 5 || b, Q3TTS_ERR_INVALID_ARG, "op %d needs b", op);
    const int want_ld = op == 5 ? 2 * C : C;
    Q3_CHECK(op == 3 ? ldx >= C : ldx == want_ld, Q3TTS_ERR_INVALID_ARG, "ldx %d (op %d wants %s %d)", ldx, op, op == 3 ? ">=" : "==", want_ld);
    Q3_CHECK(op != 0 || (T >= 1 && rows % T == 0), Q3TTS_ERR_INVALID_ARG, "dwconv7: rows %d not a multiple of T %d", rows, T);
    Q3_CHECK((size_t)rows * ldx < kProbeMaxElems, Q3TTS_ERR_INVALID_ARG, "input too large");
    require_device(device);
    LaunchCtx c{nullptr, nullptr};
    const size_t ny = (size_t)rows * C;
    const float* dx = buf.f32(x, (size_t)rows * ldx);
    const float* dw = w ? buf.f32(w, (size_t)(op == 0 ? 7 : 1) * C) : nullptr;
    const float* db = b ? buf.f32(b, C) : nullptr;
    if (op == 2 || op == 3) {
      __half* dy = (__half*)buf.alloc(ny * 2);
      Q3_CUDA(cudaMemset(dy, 0x7f, ny * 2));
      if (op == 2) launch_layernorm_f16(c, dx, rows, C, dw, db, eps, dy);
      else launch_rmsnorm_f16(c, dx, ldx, rows, C, dw, eps, dy, C);
      Q3_CUDA(cudaGetLastError());
      Q3_CUDA(cudaDeviceSynchronize());
      widen_f16(dy, ny, y);
    } else {
      float* dy = buf.f32(nullptr, ny);
      Q3_CUDA(cudaMemset(dy, 0x7f, ny * 4));
      if (op == 0) launch_dwconv7(c, dx, dw, db, C, T, rows, dy);
      else if (op == 1) launch_layernorm(c, dx, rows, C, dw, db, eps, dy);
      else if (op == 4) { SnakeW s; s.alpha = dw; s.beta = db; s.ch = C; launch_snake(c, dx, s, rows, dy); }
      else launch_silu_mul(c, dx, rows, C, dy);
      Q3_CUDA(cudaGetLastError());
      Q3_CUDA(cudaDeviceSynchronize());
      Q3_CUDA(cudaMemcpy(y, dy, ny * 4, cudaMemcpyDeviceToHost));
    }
    return Q3TTS_OK;
  } catch (const Error& e) {
    return probe_failed(e);
  }
}

// ------------------------------------------------------------------------------------------------ sampler probes
namespace {
void* upload(ProbeBuffers& buf, const void* src, size_t bytes) {
  void* d = buf.alloc(bytes);
  Q3_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
  return d;
}
// the per-row (or per-slot) sampling fields the sampler reads: a non-finite value or top_p <= 0 has no meaning in sampleToken
void check_sampling_fields(int n, const float* temperature, const float* top_p, const float* rep_penalty) {
  for (int r = 0; r < n; ++r)
    Q3_CHECK(std::isfinite(temperature[r]) && std::isfinite(top_p[r]) && std::isfinite(rep_penalty[r]) && top_p[r] > 0.f, Q3TTS_ERR_INVALID_ARG,
             "row %d: temperature %g, top_p %g, repetition_penalty %g (finite, top_p > 0)", r, temperature[r], top_p[r], rep_penalty[r]);
}
}  // namespace

q3tts_status q3tts_sampler_probe(int32_t device, int32_t form, const float* logits, int32_t n_rows, int32_t V, int32_t ld, int32_t codec_vocab,
                                 const float* temperature, const int32_t* top_k, const float* top_p, const float* repetition_penalty,
                                 const uint32_t* token_sets, const uint64_t* seed, const uint64_t* counter, int32_t* ids_out,
                                 float* processed_out) {
  ProbeBuffers buf;
  try {
    Q3_CHECK(logits && temperature && top_k && top_p && repetition_penalty && seed && counter && ids_out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(form == 0 || form == 1, Q3TTS_ERR_INVALID_ARG, "form must be 0 (sample_kernel) or 1 (frame kernel)");
    Q3_CHECK(V >= 1 && V <= kMaxVocab, Q3TTS_ERR_INVALID_ARG, "V %d outside 1..%d", V, kMaxVocab);
    Q3_CHECK(n_rows >= 1 && n_rows <= 65535, Q3TTS_ERR_INVALID_ARG, "n_rows %d outside 1..65535", n_rows);
    Q3_CHECK(ld == 0 || ld >= V, Q3TTS_ERR_INVALID_ARG, "ld %d (0 or >= V %d)", ld, V);
    check_sampling_fields(n_rows, temperature, top_p, repetition_penalty);
    const size_t n_logits = ld == 0 ? (size_t)V : (size_t)(n_rows - 1) * ld + V;
    Q3_CHECK(n_logits < kProbeMaxElems && (size_t)n_rows * V < kProbeMaxElems, Q3TTS_ERR_INVALID_ARG, "logits too large");
    require_device(device);
    LaunchCtx c{nullptr, nullptr};
    SamplerProbeRows rows;
    rows.temperature = (const float*)upload(buf, temperature, (size_t)n_rows * 4);
    rows.top_k = (const int*)upload(buf, top_k, (size_t)n_rows * 4);
    rows.top_p = (const float*)upload(buf, top_p, (size_t)n_rows * 4);
    rows.rep_penalty = (const float*)upload(buf, repetition_penalty, (size_t)n_rows * 4);
    rows.sets = token_sets ? (const unsigned*)upload(buf, token_sets, (size_t)n_rows * kMaxVocab / 8) : nullptr;
    rows.seed = (const unsigned long long*)upload(buf, seed, (size_t)n_rows * 8);
    rows.counter = (const unsigned long long*)upload(buf, counter, (size_t)n_rows * 8);
    const float* dl = (const float*)upload(buf, logits, n_logits * 4);
    int* dids = (int*)buf.alloc((size_t)n_rows * 4);
    float* dproc = nullptr;
    if (processed_out) {
      dproc = buf.f32(nullptr, (size_t)n_rows * V);
      Q3_CUDA(cudaMemset(dproc, 0x7f, (size_t)n_rows * V * 4));  // an entry the dump does not write reads as 3.4e38
    }
    launch_sampler_probe(c, form, dl, ld, n_rows, V, codec_vocab, rows, dids, dproc);
    Q3_CUDA(cudaGetLastError());
    Q3_CUDA(cudaDeviceSynchronize());
    Q3_CUDA(cudaMemcpy(ids_out, dids, (size_t)n_rows * 4, cudaMemcpyDeviceToHost));
    if (processed_out) Q3_CUDA(cudaMemcpy(processed_out, dproc, (size_t)n_rows * V * 4, cudaMemcpyDeviceToHost));
    return Q3TTS_OK;
  } catch (const Error& e) {
    return probe_failed(e);
  }
}

q3tts_status q3tts_sampler_slot_probe(int32_t device, int32_t form, int32_t group, int32_t n_slots, int32_t V, int32_t codec_vocab, int32_t eos_id,
                                      int32_t pad_id, const float* logits, int32_t* active, int32_t* finished, int32_t* step, int32_t* max_tokens,
                                      int32_t* trailing_idx, int32_t* total_text, int32_t* consecutive_pad, int32_t* n_forced,
                                      int32_t* stream_variant, int32_t* frame_alive, int32_t* logits_cap, const float* temperature,
                                      const int32_t* top_k, const float* top_p, const float* repetition_penalty, const uint64_t* seed,
                                      uint32_t* token_sets, int32_t set_words, const int32_t* forced, int32_t max_frames, float* dump,
                                      int32_t dump_slot, int32_t dump_frames, int32_t* cur_codes) {
  ProbeBuffers buf;
  try {
    int32_t* const fields[] = {active, finished, step, max_tokens, trailing_idx, total_text, consecutive_pad, n_forced, stream_variant, frame_alive,
                               logits_cap};
    for (int32_t* f : fields) Q3_CHECK(f, Q3TTS_ERR_INVALID_ARG, "NULL slot-state field");
    Q3_CHECK(logits && temperature && top_k && top_p && repetition_penalty && seed && token_sets && cur_codes, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(form == 0 || form == 1, Q3TTS_ERR_INVALID_ARG, "form must be 0 (sample_kernel) or 1 (frame kernel)");
    Q3_CHECK(group >= 0 && group < 16, Q3TTS_ERR_INVALID_ARG, "group %d outside 0..15", group);
    Q3_CHECK(V >= 1 && V <= kMaxVocab, Q3TTS_ERR_INVALID_ARG, "V %d outside 1..%d", V, kMaxVocab);
    Q3_CHECK(n_slots >= 1 && n_slots <= 4096, Q3TTS_ERR_INVALID_ARG, "n_slots %d outside 1..4096", n_slots);
    Q3_CHECK(set_words >= (V + 31) / 32 && set_words <= kMaxVocab / 32, Q3TTS_ERR_INVALID_ARG, "set_words %d cannot hold ids < %d", set_words, V);
    check_sampling_fields(n_slots, temperature, top_p, repetition_penalty);
    Q3_CHECK(!forced || (max_frames >= 1 && max_frames <= 65536), Q3TTS_ERR_INVALID_ARG, "max_frames %d outside 1..65536", max_frames);
    Q3_CHECK(!dump || (dump_frames >= 0 && dump_frames <= 65536), Q3TTS_ERR_INVALID_ARG, "dump_frames %d outside 0..65536", dump_frames);
    for (int s = 0; s < n_slots; ++s) {
      Q3_CHECK(step[s] >= 0, Q3TTS_ERR_INVALID_ARG, "slot %d: step %d < 0", s, step[s]);
      Q3_CHECK(!forced || n_forced[s] <= 0 || step[s] < max_frames, Q3TTS_ERR_INVALID_ARG, "slot %d: forced ids end at max_frames %d <= step %d", s,
               max_frames, step[s]);
    }
    Q3_CHECK(!dump || (dump_slot >= 0 && dump_slot < n_slots && logits_cap[dump_slot] <= dump_frames), Q3TTS_ERR_INVALID_ARG,
             "dump: slot %d of %d, logits_cap above dump_frames %d", dump_slot, n_slots, dump_frames);
    require_device(device);
    LaunchCtx c{nullptr, nullptr};
    std::vector<SlotState> st(n_slots);
    for (int s = 0; s < n_slots; ++s) {
      SlotState& x = st[s];
      memset(&x, 0, sizeof(x));
      x.active = active[s]; x.finished = finished[s]; x.step = step[s]; x.max_tokens = max_tokens[s];
      x.trailing_idx = trailing_idx[s]; x.total_text = total_text[s]; x.consecutive_pad = consecutive_pad[s]; x.n_forced = n_forced[s];
      x.stream_variant = stream_variant[s]; x.frame_alive = frame_alive[s]; x.logits_cap = logits_cap[s];
      x.temperature = temperature[s]; x.top_k = top_k[s]; x.top_p = top_p[s]; x.rep_penalty = repetition_penalty[s]; x.seed = seed[s];
    }
    SamplerParams p;
    p.vocab = V; p.group = group; p.codec_vocab = codec_vocab; p.eos_id = eos_id; p.pad_id = pad_id; p.groups = 16; p.set_words = set_words;
    const size_t n_set = (size_t)n_slots * 16 * set_words;
    SlotState* dst = (SlotState*)upload(buf, st.data(), (size_t)n_slots * sizeof(SlotState));
    unsigned* dsets = (unsigned*)upload(buf, token_sets, n_set * 4);
    int* dcodes = (int*)upload(buf, cur_codes, (size_t)n_slots * 16 * 4);
    const int* dforced = forced ? (const int*)upload(buf, forced, (size_t)n_slots * max_frames * 16 * 4) : nullptr;
    float* ddump = nullptr;
    if (dump) {
      ddump = buf.f32(nullptr, (size_t)std::max(dump_frames, 1) * V);
      Q3_CUDA(cudaMemset(ddump, 0x7f, (size_t)std::max(dump_frames, 1) * V * 4));
    }
    const float* dl = (const float*)upload(buf, logits, (size_t)n_slots * V * 4);
    if (form == 0) launch_sample(c, dl, V, n_slots, dst, p, dsets, dcodes, dforced, max_frames, ddump, V, 0, dump_slot);
    else launch_sample_frame_form(c, dl, V, n_slots, dst, p, dsets, dcodes, dforced, max_frames, ddump, V, 0, dump_slot);
    Q3_CUDA(cudaGetLastError());
    Q3_CUDA(cudaDeviceSynchronize());
    Q3_CUDA(cudaMemcpy(st.data(), dst, (size_t)n_slots * sizeof(SlotState), cudaMemcpyDeviceToHost));
    Q3_CUDA(cudaMemcpy(token_sets, dsets, n_set * 4, cudaMemcpyDeviceToHost));
    Q3_CUDA(cudaMemcpy(cur_codes, dcodes, (size_t)n_slots * 16 * 4, cudaMemcpyDeviceToHost));
    if (dump && dump_frames > 0) Q3_CUDA(cudaMemcpy(dump, ddump, (size_t)dump_frames * V * 4, cudaMemcpyDeviceToHost));
    for (int s = 0; s < n_slots; ++s) {
      const SlotState& x = st[s];
      active[s] = x.active; finished[s] = x.finished; step[s] = x.step; max_tokens[s] = x.max_tokens; trailing_idx[s] = x.trailing_idx;
      total_text[s] = x.total_text; consecutive_pad[s] = x.consecutive_pad; n_forced[s] = x.n_forced; stream_variant[s] = x.stream_variant;
      frame_alive[s] = x.frame_alive; logits_cap[s] = x.logits_cap;
    }
    return Q3TTS_OK;
  } catch (const Error& e) {
    return probe_failed(e);
  }
}

static q3tts_status skinny_trace_impl(int32_t device, int32_t M, int32_t N, int32_t K, int32_t bits, int32_t swiglu, int32_t residual, int32_t iters,
                                      uint64_t* stamps_out, int32_t capacity_ctas, int32_t* tiles_out, int32_t* split_out, int32_t* stages_out,
                                      double* avg_us_out) {
  try {
    Q3_CHECK(M > 0 && N > 0 && K > 0 && iters > 0 && stamps_out && tiles_out && split_out && stages_out && avg_us_out, Q3TTS_ERR_INVALID_ARG,
             "bad arguments");
    Q3_CHECK(bits == 0 || bits == 4 || bits == 8, Q3TTS_ERR_INVALID_ARG, "bits must be 0 (fp16 weights), 4 or 8");
    require_device(device);
    init_tc_gemm();
    const int n_out = swiglu ? N / 2 : N;
    __half *x = nullptr, *w = nullptr, *y16 = nullptr;
    float* y32 = nullptr;
    uint32_t* qw = nullptr;
    __half *qs = nullptr, *qb = nullptr;
    unsigned long long* tr = nullptr;
    const size_t wbytes = bits ? (size_t)N * K * bits / 8 : (size_t)N * K * 2, sbytes = (size_t)N * (K / 64) * 2;
    Q3_CUDA(cudaMalloc(&x, (size_t)M * K * 2));
    // `iters` DIFFERENT weight matrices so every launch streams from HBM like consecutive layers do
    if (bits) {
      Q3_CUDA(cudaMalloc(&qw, (size_t)iters * wbytes));
      Q3_CUDA(cudaMalloc(&qs, (size_t)iters * sbytes));
      Q3_CUDA(cudaMalloc(&qb, (size_t)iters * sbytes));
      Q3_CUDA(cudaMemset(qw, 0x5A, (size_t)iters * wbytes));
      Q3_CUDA(cudaMemset(qs, 0x1C, (size_t)iters * sbytes));  // fp16 0x1C1C ~ 4e-3
      Q3_CUDA(cudaMemset(qb, 0x00, (size_t)iters * sbytes));
    } else {
      Q3_CUDA(cudaMalloc(&w, (size_t)iters * wbytes));
      Q3_CUDA(cudaMemset(w, 0, (size_t)iters * wbytes));
    }
    Q3_CUDA(cudaMalloc(&y16, (size_t)M * n_out * 2));
    Q3_CUDA(cudaMalloc(&y32, (size_t)M * n_out * 4));
    Q3_CUDA(cudaMemset(x, 0, (size_t)M * K * 2));
    Q3_CUDA(cudaMemset(y32, 0, (size_t)M * n_out * 4));
    TcGemm g;
    g.a = x; g.w = w; g.Bt = 1; g.T = M; g.cin = K; g.N = N; g.swiglu = swiglu;
    if (bits) { g.q_bits = bits; g.q_group = 64; g.q_sdt = Q3TTS_F16; g.q_halves = swiglu ? 1 : 0; g.q_w = qw; g.q_scales = qs; g.q_biases = qb; }
    if (swiglu) { g.out16 = y16; g.ld16 = n_out; } else { g.out32 = y32; g.ld32 = n_out; }
    if (residual) { g.res = y32; g.ld_res = n_out; g.out32 = y32; g.ld32 = n_out; }
    if (bits) {
      Q3_CHECK(tc_skinny_q_supported(g), Q3TTS_ERR_INVALID_ARG, "shape is not on the dequant-fused skinny path");
      TcGemm gd = g;  // same split rule as the dense kernel: report it through the dense planner
      gd.q_w = nullptr; gd.w = x;
      tc_skinny_grid(gd, tiles_out, split_out, stages_out);
    } else {
      Q3_CHECK(tc_skinny_supported(g), Q3TTS_ERR_INVALID_ARG, "shape is not on the skinny path");
      tc_skinny_grid(g, tiles_out, split_out, stages_out);
    }
    const int ctas = *tiles_out * *split_out;
    Q3_CHECK(ctas <= capacity_ctas, Q3TTS_ERR_CAPACITY, "stamps_out holds %d CTAs, the grid has %d", capacity_ctas, ctas);
    Q3_CUDA(cudaMalloc(&tr, (size_t)ctas * 16 * 8));
    Q3_CUDA(cudaMemset(tr, 0, (size_t)ctas * 16 * 8));
    cudaStream_t st;
    Q3_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    cudaEvent_t e0, e1;
    Q3_CUDA(cudaEventCreate(&e0));
    Q3_CUDA(cudaEventCreate(&e1));
    LaunchCtx c{st, nullptr};
    cudaGraph_t graph;
    cudaGraphExec_t exec;
    tc_skinny_set_trace(tr);
    Q3_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    for (int i = 0; i < iters; ++i) {
      if (bits) {
        g.q_w = qw + (size_t)i * wbytes / 4; g.q_scales = qs + (size_t)i * sbytes / 2; g.q_biases = qb + (size_t)i * sbytes / 2;
        launch_tc_skinny_q(c, g);
      } else {
        g.w = w + (size_t)i * N * K;
        launch_tc_skinny(c, g);
      }
    }
    Q3_CUDA(cudaStreamEndCapture(st, &graph));
    tc_skinny_set_trace(nullptr);
    Q3_CUDA(cudaGraphInstantiate(&exec, graph, 0));
    Q3_CUDA(cudaGraphLaunch(exec, st));
    Q3_CUDA(cudaStreamSynchronize(st));
    Q3_CUDA(cudaEventRecord(e0, st));
    Q3_CUDA(cudaGraphLaunch(exec, st));
    Q3_CUDA(cudaEventRecord(e1, st));
    Q3_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    *avg_us_out = (double)ms * 1e3 / iters;
    Q3_CUDA(cudaMemcpy(stamps_out, tr, (size_t)ctas * 16 * 8, cudaMemcpyDeviceToHost));
    cudaGraphExecDestroy(exec); cudaGraphDestroy(graph);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st);
    cudaFree(x); cudaFree(w); cudaFree(qw); cudaFree(qs); cudaFree(qb); cudaFree(y16); cudaFree(y32); cudaFree(tr);
    return Q3TTS_OK;
  } catch (const Error& e) {
    tc_skinny_set_trace(nullptr);
    g_create_error = e.what();
    cudaGetLastError();
    return e.status;
  }
}

q3tts_status q3tts_skinny_trace(int32_t device, int32_t M, int32_t N, int32_t K, int32_t swiglu, int32_t residual, int32_t iters,
                                uint64_t* stamps_out, int32_t capacity_ctas, int32_t* tiles_out, int32_t* split_out, int32_t* stages_out,
                                double* avg_us_out) {
  return skinny_trace_impl(device, M, N, K, 0, swiglu, residual, iters, stamps_out, capacity_ctas, tiles_out, split_out, stages_out, avg_us_out);
}

q3tts_status q3tts_skinny_trace_q(int32_t device, int32_t M, int32_t N, int32_t K, int32_t bits, int32_t swiglu, int32_t residual, int32_t iters,
                                  uint64_t* stamps_out, int32_t capacity_ctas, int32_t* tiles_out, int32_t* split_out, int32_t* stages_out,
                                  double* avg_us_out) {
  return skinny_trace_impl(device, M, N, K, bits, swiglu, residual, iters, stamps_out, capacity_ctas, tiles_out, split_out, stages_out, avg_us_out);
}

q3tts_status q3tts_profile_linear(q3tts_handle* h, int32_t which, int32_t m, int32_t iters, double* ms_out, int64_t* launches_out,
                                  int64_t* bytes_per_iter_out) {
  return guarded(h, [&] {
    Q3_CHECK(ms_out && launches_out && bytes_per_iter_out && iters > 0, Q3TTS_ERR_INVALID_ARG, "bad arguments");
    Q3_CHECK(h->talker != nullptr, Q3TTS_ERR_MODEL_NOT_LOADED, "Model is not loaded");
    int64_t l = 0, b = 0;
    *ms_out = h->talker->profile_linears(which, m, iters, l, b);
    *launches_out = l;
    *bytes_per_iter_out = b;
  });
}

q3tts_status q3tts_sample_token(q3tts_handle* h, const float* logits, int32_t vocab, float temperature, int32_t top_k, float top_p,
                                float repetition_penalty, const int32_t* token_set, int32_t n_token_set, uint64_t seed,
                                uint64_t counter, int32_t* id_out) {
  return guarded(h, [&] {
    Q3_CHECK(logits && id_out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    Q3_CHECK(h->talker != nullptr, Q3TTS_ERR_MODEL_NOT_LOADED, "Model is not loaded");
    *id_out = h->talker->sample_probe(logits, vocab, temperature, top_k, top_p, repetition_penalty, token_set, n_token_set, seed, counter);
  });
}

q3tts_status q3tts_rvq_embed(q3tts_handle* h, const int32_t* codes, int32_t batch, int32_t frames, float* first_out, float* rest_out,
                             int32_t* dim_out) {
  return guarded(h, [&] {
    Q3_CHECK(h->codec != nullptr, Q3TTS_ERR_DECODER_LOAD_FAILED, "Failed to load MLX audio decoder");
    Q3_CHECK(codes && first_out && rest_out, Q3TTS_ERR_INVALID_ARG, "NULL argument");
    const int M = batch * frames, D = h->codec->vq_dim();
    if (dim_out) *dim_out = D;
    if (M <= 0) return;
    int32_t* dc = nullptr;
    float *d1 = nullptr, *d2 = nullptr;
    Q3_CUDA(cudaMalloc(&dc, (size_t)M * 64)); Q3_CUDA(cudaMalloc(&d1, (size_t)M * D * 4)); Q3_CUDA(cudaMalloc(&d2, (size_t)M * D * 4));
    Q3_CUDA(cudaMemcpyAsync(dc, codes, (size_t)M * 64, cudaMemcpyHostToDevice, h->stream));
    h->codec->rvq_embed(dc, batch, frames, d1, d2);
    Q3_CUDA(cudaMemcpyAsync(first_out, d1, (size_t)M * D * 4, cudaMemcpyDeviceToHost, h->stream));
    Q3_CUDA(cudaMemcpyAsync(rest_out, d2, (size_t)M * D * 4, cudaMemcpyDeviceToHost, h->stream));
    Q3_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(dc); cudaFree(d1); cudaFree(d2);
  });
}

}  // extern "C"
