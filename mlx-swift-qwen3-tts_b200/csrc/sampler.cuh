// Device-side sampler shared by sample_kernel (one CTA per slot) and the frame megakernel (its 512 consumer threads):
// Qwen3Talker.sampleToken (Model/Qwen3Talker.swift:274-322) + the loop's EOS / pad rules (:470-494).
// BAR = 0: the group is the whole CTA (__syncthreads); BAR = 1: named barrier 1 over the first NT threads of the CTA.
#pragma once
#include "kernels.h"

namespace q3 {

template <int BAR, int NT>
__device__ __forceinline__ void block_sync() {
  if constexpr (BAR == 0) __syncthreads();
  else asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
}
__device__ __forceinline__ float smp_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float smp_warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Counter-based uniform in (0,1): splitmix64 finaliser over (seed, counter, index), 23-bit mantissa (+0.5 so neither
// 0 nor 1 occurs).  Same integer arithmetic as oracle/talker.py:counter_uniform.
__device__ __forceinline__ float counter_uniform(unsigned long long seed, unsigned long long counter, unsigned idx) {
  unsigned long long x = seed * 0x9E3779B97F4A7C15ull + counter * 0xD1B54A32D192ED03ull +
                         (unsigned long long)idx * 0x8CB92BA72F3D8DD7ull + 0x2545F4914F6CDD1Dull;
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return (__uint2float_rn((unsigned)(x >> 41)) + 0.5f) * (1.0f / 8388608.0f);
}
// Monotone float -> uint map.  -0.0 is mapped as +0.0: the thresholds compare floats, for which -0.0 == +0.0, so a signed
// zero tied at the top-k or top-p threshold survives like any other tie.
__device__ __forceinline__ unsigned ordered_key(float f) {
  unsigned u = __float_as_uint(f);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

constexpr int kSampleThreads = 512;
constexpr int kFrameSampleThreads = 15 * 32;  // frame_megakernel's consumer warps 0-14 run sample_slot<1, kFrameSampleThreads>
constexpr int kMaxVocab = 4096;

struct BlockRed {
  float fv[16];
  int iv[16];
  float bcast_f;
  int bcast_i;
};

// argmax with first-index tie break over sl[0..V)
template <int BAR, int NT>
__device__ int block_argmax(const float* sl, int V, BlockRed& br) {
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = threadIdx.x; i < V; i += NT) {
    const float v = sl[i];
    if (v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  block_sync<BAR, NT>();
  if ((threadIdx.x & 31) == 0) { br.fv[threadIdx.x >> 5] = bv; br.iv[threadIdx.x >> 5] = bi; }
  block_sync<BAR, NT>();
  if (threadIdx.x == 0) {
    float v = br.fv[0]; int idx = br.iv[0];
    for (int w = 1; w < NT / 32; ++w)
      if (br.fv[w] > v || (br.fv[w] == v && br.iv[w] < idx)) { v = br.fv[w]; idx = br.iv[w]; }
    if (idx == 0x7fffffff) idx = 0;
    br.bcast_i = idx;
  }
  block_sync<BAR, NT>();
  return br.bcast_i;
}
template <int BAR, int NT>
__device__ float block_sum(float v, BlockRed& br) {
  v = smp_warp_sum(v);
  block_sync<BAR, NT>();
  if ((threadIdx.x & 31) == 0) br.fv[threadIdx.x >> 5] = v;
  block_sync<BAR, NT>();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < NT / 32; ++w) s += br.fv[w];
    br.bcast_f = s;
  }
  block_sync<BAR, NT>();
  return br.bcast_f;
}
template <int BAR, int NT>
__device__ float block_max(float v, BlockRed& br) {
  v = smp_warp_max(v);
  block_sync<BAR, NT>();
  if ((threadIdx.x & 31) == 0) br.fv[threadIdx.x >> 5] = v;
  block_sync<BAR, NT>();
  if (threadIdx.x == 0) {
    float s = -INFINITY;
    for (int w = 0; w < NT / 32; ++w) s = fmaxf(s, br.fv[w]);
    br.bcast_f = s;
  }
  block_sync<BAR, NT>();
  return br.bcast_f;
}

// Qwen3Talker.sampleToken (Model/Qwen3Talker.swift:274-322) over sl[0..V) held in shared memory (already carrying
// the EOS/pad suppression of :470-475 where it applies).  Returns the id to every thread.
// DUMP (q3tts_sampler_probe only): processed[0..V) receives the row as it stands just before the Gumbel step -- for a greedy
// row, right after the penalty.
template <int BAR, int NT, bool DUMP = false>
__device__ int sample_block(float* sl, int V, int codec_vocab, float temperature, int top_k, float top_p, float rep_penalty,
                            const unsigned* set_bitmap, unsigned long long seed, unsigned long long counter, BlockRed& br,
                            float* processed = nullptr) {
  if (set_bitmap != nullptr && rep_penalty != 1.0f) {  // set-based, division regardless of sign (:288-299)
    for (int i = threadIdx.x; i < V; i += NT)
      if (set_bitmap[i >> 5] & (1u << (i & 31))) sl[i] = sl[i] / rep_penalty;
  }
  block_sync<BAR, NT>();
  if (!(temperature > 0.f)) {  // greedy: before the valid-token mask (:301-305)
    if constexpr (DUMP) for (int i = threadIdx.x; i < V; i += NT) processed[i] = sl[i];
    return block_argmax<BAR, NT>(sl, V, br);
  }
  for (int i = threadIdx.x; i < V; i += NT) sl[i] = sl[i] / temperature;
  block_sync<BAR, NT>();
  if (top_k > 0 && top_k < V) {  // threshold = k-th largest; ties at the threshold survive (:307-314)
    unsigned t = 0;
    for (int bit = 31; bit >= 0; --bit) {
      const unsigned cand = t | (1u << bit);
      float cnt = 0.f;
      for (int i = threadIdx.x; i < V; i += NT) cnt += (ordered_key(sl[i]) >= cand) ? 1.f : 0.f;
      if (block_sum<BAR, NT>(cnt, br) >= (float)top_k) t = cand;
    }
    for (int i = threadIdx.x; i < V; i += NT)
      if (ordered_key(sl[i]) < t) sl[i] = -INFINITY;
    block_sync<BAR, NT>();
  }
  if (V == codec_vocab) {  // valid ids: < 2048, 2148 (pad), 2150 (eos)  (:19-33, 316-319)
    for (int i = threadIdx.x; i < V; i += NT)
      if (!(i < 2048 || i == 2148 || i == 2150)) sl[i] = -INFINITY;
    block_sync<BAR, NT>();
  }
  if (top_p < 1.0f) {  // extension (no top-p in the reference): keep i iff mass of strictly more probable ids < top_p
    float mx = -INFINITY;
    for (int i = threadIdx.x; i < V; i += NT) mx = fmaxf(mx, sl[i]);
    mx = block_max<BAR, NT>(mx, br);
    float z = 0.f;
    for (int i = threadIdx.x; i < V; i += NT) z += expf(sl[i] - mx);
    z = block_sum<BAR, NT>(z, br);
    unsigned t = 0;  // largest key with mass(key_j > t) >= top_p
    for (int bit = 31; bit >= 0; --bit) {
      const unsigned cand = t | (1u << bit);
      float mass = 0.f;
      for (int i = threadIdx.x; i < V; i += NT)
        if (ordered_key(sl[i]) > cand) mass += expf(sl[i] - mx);
      if (block_sum<BAR, NT>(mass, br) / z >= top_p) t = cand;
    }
    for (int i = threadIdx.x; i < V; i += NT)
      if (ordered_key(sl[i]) <= t) sl[i] = -INFINITY;
    block_sync<BAR, NT>();
  }
  // MLXRandom.categorical == Gumbel-max (:321)
  for (int i = threadIdx.x; i < V; i += NT) {
    const float l = sl[i];
    if constexpr (DUMP) processed[i] = l;
    if (l > -INFINITY) {
      const float u = counter_uniform(seed, counter, (unsigned)i);
      sl[i] = l + (-logf(-logf(u)));
    }
  }
  block_sync<BAR, NT>();
  return block_argmax<BAR, NT>(sl, V, br);
}

// One slot's sampleToken + loop bookkeeping (the body of sample_kernel), callable from any 512-thread group that owns
// `sl` / `br`: group 0 applies the EOS / pad stop rules and sets frame_alive, groups >= 1 record into the per-group sets.
template <int BAR, int NT>
__device__ void sample_slot(int slot, const float* __restrict__ logits, int ld, SlotState* __restrict__ st, const SamplerParams& p,
                            unsigned* __restrict__ token_sets, int* __restrict__ cur_codes, const int* __restrict__ forced,
                            int max_frames, float* __restrict__ dump, int dump_stride_frame, int dump_offset, int dump_slot,
                            float* sl, BlockRed& br) {
  SlotState& s = st[slot];
  const int V = p.vocab;
  if (p.group == 0) {
    const bool alive = s.active && !s.finished && s.step < s.max_tokens;
    if (!alive) {
      if (threadIdx.x == 0) { s.frame_alive = 0; if (s.active && s.step >= s.max_tokens) s.finished = 1; }
      return;
    }
  } else if (!s.frame_alive) {
    return;
  }
  const float* lg = logits + (size_t)slot * ld;
  const int step = s.step;
  if (dump != nullptr && slot == dump_slot && step < s.logits_cap) {
    float* d = dump + (size_t)step * dump_stride_frame + dump_offset;
    for (int i = threadIdx.x; i < V; i += NT) d[i] = lg[i];
  }
  const bool suppress = (p.group == 0) && (s.trailing_idx < s.total_text);  // EOS/pad masked while text remains (:470-475)
  for (int i = threadIdx.x; i < V; i += NT) {
    float v = lg[i];
    if (suppress && (i == p.eos_id || i == p.pad_id)) v = -INFINITY;
    sl[i] = v;
  }
  block_sync<BAR, NT>();
  unsigned* set = token_sets + ((size_t)slot * p.groups + p.group) * p.set_words;
  const bool use_set = (p.group == 0) || !s.stream_variant;  // generateStream: no penalty on CP groups (:821)
  int tok = sample_block<BAR, NT>(sl, V, p.codec_vocab, s.temperature, s.top_k, s.top_p, s.rep_penalty, use_set ? set : nullptr, s.seed,
                         (unsigned long long)step * p.groups + p.group, br);
  if (threadIdx.x != 0) return;
  const bool is_forced = s.n_forced > 0 && forced != nullptr;
  if (is_forced) tok = forced[((size_t)slot * max_frames + step) * p.groups + p.group];
  if (p.group == 0) {
    if (!is_forced) {  // stop rules (:485-494)
      if (tok == p.eos_id) { s.finished = 1; s.frame_alive = 0; return; }
      if (tok == p.pad_id) {
        s.consecutive_pad += 1;
        if (s.consecutive_pad > 6) { s.finished = 1; s.frame_alive = 0; return; }
      } else {
        s.consecutive_pad = 0;
      }
    }
    s.frame_alive = 1;
  } else if (tok >= 0 && tok < V) {
    set[tok >> 5] |= 1u << (tok & 31);  // generatedCodePredictorSets[g-1].insert (:522)
  }
  cur_codes[slot * p.groups + p.group] = tok;
}
}  // namespace q3
