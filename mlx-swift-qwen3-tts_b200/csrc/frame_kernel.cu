// Persistent frame kernel (sm_100a).  Grid = one CTA per SM (cooperative launch), 16 warps per CTA:
//   warps 0-14 : consumers.  Every Qwen3DecoderLayer is five phases — [RMSNorm + qkv GEMV] | [q/k norm + RoPE + KV append +
//                split-key window attention] | [split combine + o GEMV + residual] | [RMSNorm + gate/up GEMV + SwiGLU] |
//                [down GEMV + residual].  There is NO grid barrier: every value a phase hands to the next one travels as an
//                8-byte (value, phase tag) pair ("LL" exchange) that the consumer polls directly in L2, so a phase boundary
//                costs one store->load round trip instead of fence + atomic + poll + reload.
//                Each CTA owns a contiguous slice of every linear's output rows; a warp owns a row: 128-bit reads of the
//                packed row from shared memory, dequant in registers, activations lane-major in shared memory, shuffle reduce.
//   warp 15    : weight producer.  Walks the frame's linears in execution order and copies this CTA's row slices (weights,
//                scales, biases) global -> shared with 1-D TMA bulk copies (UBLKCP) into a ring of slots, mbarrier
//                complete_tx to the consumers.  Weight addresses never depend on activations, so the stream runs several
//                phases ahead and the dependency chain waits only on L2-resident activations.
// Sampling (Qwen3Talker.sampleToken), the next-input embedding sum and all loop bookkeeping run inside the same kernel.
//
// Batch-1 decode is bound by the LATENCY of ~660 dependent phases per frame, not by bandwidth: each warp runs nearly alone on
// its scheduler, so what counts is the number of dependent instructions per phase.  Hence: one copy of every phase body
// (instruction cache), no integer division on the per-phase path, descriptors prefetched a phase ahead into shared memory,
// 16 warps so that ptxas may use 128 registers, and shared-memory pointers the compiler can prove are shared (LDS, not LD).
#include "device_utils.cuh"
#include "frame_kernel.h"
#include "sampler.cuh"

namespace q3 {

namespace {

constexpr int kCWarps = 15;            // consumer warps
constexpr int kCons = kCWarps * 32;    // 480 consumer threads (named barrier 1)
static_assert(kCons == kFrameSampleThreads, "q3tts_sampler_probe runs the sampler form of the frame kernel with kFrameSampleThreads");
constexpr int kMegaThreads = 512;
constexpr int kKeyTile = 128;          // keys per attention item (host sizes nsplit so that a split never exceeds it)
constexpr int kKeyGroups = 3;          // P.V key groups: 3 x 128 threads

__device__ __forceinline__ void cbar() { asm volatile("bar.sync 1, %0;" ::"n"(kCons) : "memory"); }
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded waits: a protocol bug must surface as a trapped kernel (an error on the host), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) __trap();
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// ---- LL exchange: element = (tag << 32) | value bits, written / read with single 64-bit (or paired 2 x 64-bit) accesses.
// A reader spins until the tag equals the producing phase's id; buffers are zeroed per launch and tags start at 1.
typedef unsigned long long u64;
__device__ __forceinline__ void ll_store(u64* p, uint32_t bits, uint32_t tag) {
  asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(((u64)tag << 32) | bits) : "memory");
}
__device__ __forceinline__ void ll_ld2(const u64* p, u64& a, u64& b) {
  asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ bool ll_ok(u64 v, uint32_t tag) { return (uint32_t)(v >> 32) == tag; }
__device__ __forceinline__ float ll_f(u64 v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ uint32_t ll_load1(const u64* p, uint32_t tag) {
  u64 v;
  uint32_t spins = 0;
  while (true) {
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    if (ll_ok(v, tag)) break;
    if (++spins > (1u << 22)) __trap();
  }
  return (uint32_t)v;
}
__device__ __forceinline__ float4 ll_load4(const u64* p, uint32_t tag) {  // 4 consecutive elements, 32-byte aligned
  u64 a, b, c, d;
  uint32_t spins = 0;
  while (true) {
    ll_ld2(p, a, b);
    ll_ld2(p + 2, c, d);
    if (ll_ok(a, tag) && ll_ok(b, tag) && ll_ok(c, tag) && ll_ok(d, tag)) break;
    if (++spins > (1u << 22)) __trap();
  }
  return make_float4(ll_f(a), ll_f(b), ll_f(c), ll_f(d));
}
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ uint32_t lop3_and_or(uint32_t a, uint32_t b, uint32_t c) {  // (a & b) | c in ONE LOP3
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// Shared-memory plan.  Everything is addressed from the one extern array so the compiler keeps the shared address space.
extern __shared__ __align__(128) uint8_t smem[];

struct Sm {   // byte offsets into smem (from MegaParams) resolved once
  uint8_t* ring;
  uint64_t *full, *empty;
  float4* xs;       // lane-major staged activations; also the scratch of the attention / sampling phases
  float* xsum;
  float* xraw;      // raw residual rows of the current layer input
  float* red;       // [rows][16] partial sums of squares
  MegaLinear* dsc;  // [2] descriptor of the current / next linear
  float* hl;        // [slots][raw_ld] h_last of the previous talker step (every CTA keeps its own copy)
  float* rope;      // [slots][2 rows][64 freqs][cos, sin] of the current unit's positions
  __half* xh;       // tensor-core path: fp16 activation columns, permuted k (aliases xs)
  float* part;      // tensor-core path: partial [16 x 8] tiles of the K slices
};

struct Slice { int r0, rows, rch, nch; };
// no integer division on the per-phase path: the unit split over the grid and the chunk size come precomputed from the host
__device__ __forceinline__ Slice slice_of(const MegaLinear& L) {
  const int c = blockIdx.x;
  Slice s;
  s.rows = (L.ubase + (c < L.urem ? 1 : 0)) * L.unit;
  s.r0 = (c * L.ubase + min(c, L.urem)) * L.unit;
  s.rch = L.rch;
  s.nch = s.rows == 0 ? 0 : (s.rows <= s.rch ? 1 : (s.rows + s.rch - 1) / s.rch);
  return s;
}

// ------------------------------------------------------------------------------------------------ producer warp
__device__ void producer_loop(const MegaParams& p, uint8_t* ring, uint64_t* full, uint64_t* empty) {
  int slot = 0;
  uint32_t ph = 0;
  for (int f = 0; f < p.n_frames; ++f) {
    for (int li = 0; li < p.n_lin; ++li) {
      const MegaLinear L = p.lin[li];
      const Slice s = slice_of(L);
      for (int c = 0; c < s.nch; ++c) {
        {  // the ring is usually full: sleep between probes so this lone thread does not steal issue slots from the consumers
          uint32_t spins = 0;
          while (!mbar_try_wait(&empty[slot], ph ^ 1u)) {
            __nanosleep(256);
            if (++spins > (1u << 24)) __trap();
          }
        }
        const int row0 = s.r0 + c * s.rch;
        const int rows = min(s.rch, s.rows - c * s.rch);
        const uint32_t wb = (uint32_t)rows * L.row_bytes, sb = (uint32_t)rows * L.srow_bytes;
        mbar_expect_tx(&full[slot], (uint32_t)L.nsub * (wb + 2u * sb));
        uint8_t* dst = ring + (size_t)slot * p.slot_bytes;
        for (int sub = 0; sub < L.nsub; ++sub) {
          const size_t grow = (size_t)sub * L.out_eff + row0;
          bulk_g2s(dst, reinterpret_cast<const uint8_t*>(L.w) + grow * L.row_bytes, wb, &full[slot]);
          dst += wb;
          if (sb) {
            bulk_g2s(dst, reinterpret_cast<const uint8_t*>(L.scales) + grow * L.srow_bytes, sb, &full[slot]);
            dst += sb;
            bulk_g2s(dst, reinterpret_cast<const uint8_t*>(L.biases) + grow * L.srow_bytes, sb, &full[slot]);
            dst += sb;
          }
        }
        if (++slot == p.n_ring) { slot = 0; ph ^= 1u; }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ per-thread state
struct Ctx {
  int slot;          // ring position of the next chunk (consumer side)
  uint32_t ring_ph;
  uint32_t ph;       // id of the phase being executed (identical in every CTA); values written carry it as their tag
  uint32_t fseq;     // 1 + frame index within the launch: tag of the per-frame messages
  int tid, lane, warp;
  long long* trace;  // per-phase cycle stamps of this CTA's thread 0 (diagnostics; null = off)
  long long wait_full, wait_poll;
};

__device__ __forceinline__ void trace_close(Ctx& cx) {
  if (cx.trace) { cx.trace[5] = clock64(); cx.trace += 8; }
}

// per-frame message of unit u for `slot`: 4 LL elements {code_u, pos, win_start, text row (-1: tts_pad)} (the last three: unit 0)
__device__ __forceinline__ u64* msg_at(const MegaParams& p, uint32_t fseq, int u, int slot) {
  return p.ex_msg + ((size_t)((fseq & 1u) * 16 + u) * kMegaMaxSlots + slot) * 4;
}

// ------------------------------------------------------------------------------------------------ activation staging
__device__ __forceinline__ float4 ld_emb4(const Embedding& e, int id, int f) {  // 4 consecutive elements of row `id`
  if (id < 0 || id >= e.rows) return make_float4(0.f, 0.f, 0.f, 0.f);
  const size_t i = (size_t)id * e.dim + (size_t)f * 4;
  if (e.dt == Q3TTS_F32) return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(e.w) + i);
  const uint2 r = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(e.w) + i);
  if (e.dt == Q3TTS_F16) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
    return make_float4(a.x, a.y, b.x, b.y);
  }
  return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xFFFF0000u), __uint_as_float(r.y << 16), __uint_as_float(r.y & 0xFFFF0000u));
}
__device__ __forceinline__ void add4(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }

enum InKind {
  IN_GX = 0,        // residual rows from the exchange buffer
  IN_GX_LAST,       // last row of each slot (code-predictor head)
  IN_CP0,           // pass 0: rows (2s, 2s+1) = [h_last[s], codec_embedding(code0)]          (Model/Qwen3Talker.swift:503-505)
  IN_CPG,           // pass g: row s = code_predictor.codec_embedding[g-1](code_g)            (:509-510)
  IN_TALKER,        // next talker input = (trailing text | tts_pad) + sum of 16 code embeddings  (:531-549)
  IN_ATTN,          // attention output: combine of the split-key partials
  IN_ACT            // SwiGLU activations
};

struct InArgs {
  int kind;
  int pass;      // code-predictor pass (IN_CPG) ; rows per slot (IN_GX_LAST)
  int nsplit, heads;
};

// softmax-weighted merge of NSPLIT key splits (flash-decoding combine); every load of a round is in flight together
template <int NSPLIT>
__device__ __forceinline__ float4 combine_splits(const MegaParams& p, int mi, int f, int heads, uint32_t tag) {
  const int h = f >> 5;
  u64 o[NSPLIT][4], ml[NSPLIT][2];
  uint32_t spins = 0;
  while (true) {
    bool ok = true;
#pragma unroll
    for (int sp = 0; sp < NSPLIT; ++sp) {
      const u64* base = p.ex_part + (size_t)(mi * NSPLIT + sp) * p.part_stride;
      ll_ld2(base + heads * 128 + 2 * h, ml[sp][0], ml[sp][1]);
      ll_ld2(base + (size_t)f * 4, o[sp][0], o[sp][1]);
      ll_ld2(base + (size_t)f * 4 + 2, o[sp][2], o[sp][3]);
    }
#pragma unroll
    for (int sp = 0; sp < NSPLIT; ++sp)
      ok = ok && ll_ok(ml[sp][0], tag) && ll_ok(ml[sp][1], tag) && ll_ok(o[sp][0], tag) && ll_ok(o[sp][1], tag) && ll_ok(o[sp][2], tag) && ll_ok(o[sp][3], tag);
    if (ok) break;
    if (++spins > (1u << 22)) __trap();
  }
  float M = -INFINITY;
#pragma unroll
  for (int sp = 0; sp < NSPLIT; ++sp) M = fmaxf(M, ll_f(ml[sp][0]));
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float den = 0.f;
#pragma unroll
  for (int sp = 0; sp < NSPLIT; ++sp) {
    const float l = ll_f(ml[sp][1]);
    if (l > 0.f) {
      const float w = expf(ll_f(ml[sp][0]) - M);
      acc.x += w * ll_f(o[sp][0]); acc.y += w * ll_f(o[sp][1]); acc.z += w * ll_f(o[sp][2]); acc.w += w * ll_f(o[sp][3]);
      den += w * l;
    }
  }
  const float inv = 1.0f / den;
  return make_float4(acc.x * inv, acc.y * inv, acc.z * inv, acc.w * inv);
}

__device__ __forceinline__ float4 load_in(const MegaParams& p, const Ctx& cx, const float* hl, const InArgs& a, int mi, int f) {
  const uint32_t tag = cx.ph - 1u;  // every exchanged value was produced by the immediately preceding phase
  switch (a.kind) {
    case IN_GX: return ll_load4(p.ex_x + (size_t)mi * p.ld_x + (size_t)f * 4, tag);
    case IN_GX_LAST: return ll_load4(p.ex_x + (size_t)(mi * a.pass + a.pass - 1) * p.ld_x + (size_t)f * 4, tag);
    case IN_ACT: return ll_load4(p.ex_act + (size_t)mi * p.ld_act + (size_t)f * 4, tag);
    case IN_CP0: {
      const int slot = mi >> 1;
      if ((mi & 1) == 0) return reinterpret_cast<const float4*>(hl + slot * p.raw_ld)[f];
      return ld_emb4(p.codec, (int)ll_load1(msg_at(p, cx.fseq, 0, slot), cx.fseq), f);
    }
    case IN_CPG: return ld_emb4(p.cp_emb[a.pass - 1], (int)ll_load1(msg_at(p, cx.fseq, a.pass, mi), cx.fseq), f);
    case IN_TALKER: {
      u64 c[16], hdr;
      uint32_t spins = 0;
      while (true) {  // the 16 codes of this frame + the text cursor: all loads in flight together
        bool ok = true;
#pragma unroll
        for (int g = 0; g < 16; ++g) asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(c[g]) : "l"(msg_at(p, cx.fseq, g, mi)) : "memory");
        asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(hdr) : "l"(msg_at(p, cx.fseq, 0, mi) + 3) : "memory");
#pragma unroll
        for (int g = 0; g < 16; ++g) ok = ok && ll_ok(c[g], cx.fseq);
        if (ok && ll_ok(hdr, cx.fseq)) break;
        if (++spins > (1u << 22)) __trap();
      }
      const int ti = (int)(uint32_t)hdr;
      const float* text = ti >= 0 ? p.trailing + ((size_t)mi * p.max_trailing + ti) * p.H : p.tts_pad;
      float4 sum = ld_emb4(p.codec, (int)(uint32_t)c[0], f);
#pragma unroll
      for (int g = 1; g < 16; ++g) add4(sum, ld_emb4(p.cp_emb[g - 1], (int)(uint32_t)c[g], f));
      float4 t = *reinterpret_cast<const float4*>(text + (size_t)f * 4);
      add4(t, sum);
      return t;
    }
    default:  // IN_ATTN
      return a.nsplit == 1 ? combine_splits<1>(p, mi, f, a.heads, tag) : combine_splits<4>(p, mi, f, a.heads, tag);
  }
}

// Stage `m` rows of K values: raw copy (residual) when keep_raw, RMSNorm weight folded in, lane-major layout, per-lane sums
// for the group-bias term.  Leaves sum(x^2) per row in sm.red (the RMS scale is applied to the finished dot products).
template <int FMT>
__device__ __forceinline__ void stage_rows(const MegaParams& p, const Sm& sm, const Ctx& cx, const InArgs& in, int m, int K, const float* norm_w,
                                           bool keep_raw) {
  constexpr int VPL = FmtTraits<FMT>::VPL;
  constexpr int KC = 32 * VPL;
  constexpr bool QUANT = (FMT == W_Q4 || FMT == W_Q8);
  constexpr int LPG = VPL / 4;
  const int nchunk = (K + KC - 1) / KC;
  const int xstride = nchunk * (KC / 4);
  const int in4 = K >> 2;
  for (int mi = 0; mi < m; ++mi) {
    float ss = 0.f;
    for (int f0 = 0; f0 < in4; f0 += kCons) {
      const int f = f0 + cx.tid;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (f < in4) {
        float4 nw = make_float4(1.f, 1.f, 1.f, 1.f);
        if (norm_w != nullptr) nw = __ldg(reinterpret_cast<const float4*>(norm_w) + f);  // in flight with the poll below
        const long long tp0 = cx.trace ? clock64() : 0;
        v = load_in(p, cx, sm.hl, in, mi, f);
        if (cx.trace) const_cast<Ctx&>(cx).wait_poll += clock64() - tp0;
        ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
        if (keep_raw) reinterpret_cast<float4*>(sm.xraw + mi * p.raw_ld)[f] = v;
        v.x *= nw.x; v.y *= nw.y; v.z *= nw.z; v.w *= nw.w;
        const int e = f << 2;
        const int ch = e / KC, ec = e - ch * KC;
        const int l = ec / VPL, j = (ec - l * VPL) >> 2;
        sm.xs[mi * xstride + ch * (KC / 4) + j * 32 + l] = v;
      }
      if constexpr (QUANT) {
        float s4 = (v.x + v.y) + (v.z + v.w);
#pragma unroll
        for (int o = 1; o < LPG; o <<= 1) s4 += __shfl_xor_sync(0xffffffffu, s4, o);
        if ((cx.tid & (LPG - 1)) == 0 && f < in4) {
          const int e = f << 2;
          const int ch = e / KC;
          sm.xsum[mi * (nchunk * 32) + ch * 32 + (e - ch * KC) / VPL] = s4;
        }
      }
    }
    if (norm_w != nullptr) {
      ss = warp_sum(ss);
      if (cx.lane == 0) sm.red[mi * 16 + cx.warp] = ss;
    }
  }
  cbar();
}

// ------------------------------------------------------------------------------------------------ GEMV over the ring
enum EpiKind { E_STORE = 0, E_ADD_RAW = 1, E_SWIGLU = 2 };

__device__ __forceinline__ float scale_to_f32(uint32_t raw16, int sdt) {  // bf16 / f16 payload of a 16-bit shared-memory load
  const float as_bf16 = __uint_as_float(raw16 << 16);
  const float as_f16 = __half2float(__ushort_as_half((unsigned short)raw16));
  return sdt == Q3TTS_F16 ? as_f16 : as_bf16;
}

// R rows of the warp are in flight together (independent FMA chains, the staged activations are read once for all of them).
template <int FMT, int M, int R>
__device__ __forceinline__ void gemv_rows(const MegaParams& p, const Sm& sm, Ctx& cx, const MegaLinear& L, int m, bool has_norm, float eps, int epi,
                                          u64* out, int ld_out, float* plain_out, int plain_ld) {
  constexpr int VPL = FmtTraits<FMT>::VPL;
  constexpr int KC = 32 * VPL;
  constexpr bool QUANT = (FMT == W_Q4 || FMT == W_Q8);
  const int K = L.in;
  const int nchunk = (K + KC - 1) / KC;
  const int xstride = nchunk * (KC / 4);
  const int row_bytes = L.row_bytes, srow_bytes = L.srow_bytes, nsub = L.nsub, sdt = L.sdt, gshift = L.group_shift;
  float inv_rms[M];
#pragma unroll
  for (int mi = 0; mi < M; ++mi) {
    inv_rms[mi] = 1.0f;
    if (has_norm && mi < m) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kCWarps; ++w) s += sm.red[mi * 16 + w];
      inv_rms[mi] = rsqrtf(s / (float)K + eps);
    }
  }
  const Slice s = slice_of(L);
  for (int c = 0; c < s.nch; ++c) {
    const int slot = cx.slot;
    const long long tw0 = cx.trace ? clock64() : 0;
    mbar_wait(&sm.full[slot], cx.ring_ph);
    if (cx.trace) { cx.wait_full += clock64() - tw0; cx.trace[3] = clock64(); }
    const int row0 = s.r0 + c * s.rch;
    const int rows = min(s.rch, s.rows - c * s.rch);
    const int wb = rows * row_bytes, sb = rows * srow_bytes;
    const uint8_t* base = sm.ring + slot * p.slot_bytes;
    for (int r = cx.warp; r < rows; r += R * kCWarps) {
      float res[R][2][M];
#pragma unroll
      for (int q = 0; q < R; ++q) {
#pragma unroll
        for (int sub = 0; sub < 2; ++sub) {
#pragma unroll
          for (int mi = 0; mi < M; ++mi) res[q][sub][mi] = 0.f;
        }
      }
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        if (sub < nsub) {
          const uint8_t* sbase = base + sub * (wb + 2 * sb);
          float acc[R][M][2];
#pragma unroll
          for (int q = 0; q < R; ++q) {
#pragma unroll
            for (int mi = 0; mi < M; ++mi) acc[q][mi][0] = acc[q][mi][1] = 0.f;
          }
          for (int ch = 0; ch < nchunk; ++ch) {
            const int e0 = ch * KC + cx.lane * VPL;
            if (e0 < K) {
#pragma unroll
              for (int q = 0; q < R; ++q) {
                const int rq = r + q * kCWarps;
                if (q == 0 || rq < rows) {
                  const uint4 wv = reinterpret_cast<const uint4*>(sbase + rq * row_bytes)[ch * 32 + cx.lane];
                  const uint8_t* scp = sbase + wb + rq * srow_bytes;
                  float scv = 1.f, biv = 0.f;
                  if constexpr (QUANT) {
                    const int gi = e0 >> gshift;
                    if (sdt == Q3TTS_F32) {
                      scv = reinterpret_cast<const float*>(scp)[gi];
                      biv = reinterpret_cast<const float*>(scp + sb)[gi];
                    } else {
                      scv = scale_to_f32(reinterpret_cast<const unsigned short*>(scp)[gi], sdt);
                      biv = scale_to_f32(reinterpret_cast<const unsigned short*>(scp + sb)[gi], sdt);
                    }
                  }
                  float wf[VPL];
                  if constexpr (FMT == W_Q4) {  // m = 1 + q/16: shift + one LOP3 per value, no FADD
                    const uint32_t ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
#pragma unroll
                      for (int n = 0; n < 8; ++n) {
                        const uint32_t sh = (19 - 4 * n) >= 0 ? (ww[i] << ((19 - 4 * n) & 31)) : (ww[i] >> ((4 * n - 19) & 31));
                        wf[i * 8 + n] = __uint_as_float(lop3_and_or(sh, 0x00780000u, 0x3F800000u));
                      }
                    }
                    scv *= 16.0f;  // s*q.x + b*sum(x) = 16s*(m.x) + (b - 16s)*sum(x)
                    biv -= scv;
                  } else {
                    lane_expand<FMT>(wv, wf);
                  }
#pragma unroll
                  for (int mi = 0; mi < M; ++mi) {
                    const float4* xp = sm.xs + mi * xstride + ch * (KC / 4) + cx.lane;
                    float d0 = 0.f, d1 = 0.f;  // two independent FMA chains per (row, activation row)
#pragma unroll
                    for (int j = 0; j < VPL / 4; ++j) {
                      const float4 x = xp[j * 32];
                      d0 = fmaf(wf[4 * j], x.x, d0);
                      d1 = fmaf(wf[4 * j + 1], x.y, d1);
                      d0 = fmaf(wf[4 * j + 2], x.z, d0);
                      d1 = fmaf(wf[4 * j + 3], x.w, d1);
                    }
                    if constexpr (QUANT) {
                      acc[q][mi][0] = fmaf(scv, d0 + d1, acc[q][mi][0]);
                      acc[q][mi][1] = fmaf(biv, sm.xsum[mi * (nchunk * 32) + ch * 32 + cx.lane], acc[q][mi][1]);
                    } else {
                      acc[q][mi][0] += d0;
                      acc[q][mi][1] += d1;
                    }
                  }
                }
              }
            }
          }
#pragma unroll
          for (int q = 0; q < R; ++q) {
#pragma unroll
            for (int mi = 0; mi < M; ++mi) res[q][sub][mi] = warp_sum(acc[q][mi][0] + acc[q][mi][1]) * inv_rms[mi];
          }
        }
      }
      if (cx.trace) cx.trace[4] = clock64();
#pragma unroll
      for (int q = 0; q < R; ++q) {
        const int rq = r + q * kCWarps;
        if (q == 0 || rq < rows) {
          const int grow = row0 + rq;
#pragma unroll
          for (int mi = 0; mi < M; ++mi) {
            if (cx.lane == mi && mi < m) {
              float v = res[q][0][mi];
              if (epi == E_SWIGLU) {
                float g = v, u = res[q][1][mi];
                if (L.bias) { g += L.bias[grow]; u += L.bias[grow + L.out_eff]; }
                v = silu_f(g) * u;
              } else {
                if (L.bias) v += L.bias[grow];
                if (epi == E_ADD_RAW) v += sm.xraw[mi * p.raw_ld + grow];
              }
              ll_store(out + (size_t)mi * ld_out + grow, __float_as_uint(v), cx.ph);
              if (plain_out) plain_out[(size_t)mi * plain_ld + grow] = v;
            }
          }
        }
      }
    }
    __syncwarp();
    if (cx.lane == 0) mbar_arrive(&sm.empty[slot]);
    if (++cx.slot == p.n_ring) { cx.slot = 0; cx.ring_ph ^= 1u; }
  }
}

// ------------------------------------------------------------------------------------------------ tensor-core GEMV (packed formats)
// The packed 4/8-bit linears run on mma.sync.m16n8k16 (fp16 x fp16 -> fp32): 16 weight rows are the M side of the tile, up
// to 8 activation rows (slots x rows-per-slot) are the N side, so several utterances cost the same issue slots as one.
// Integer codes go to fp16 through the 0x6400 exponent trick (shift + LOP3 give 1024 + q for a PAIR of values, one exact
// HSUB2 removes the 1024 — leaving it in costs the accumulator seven bits); the group scale / bias are applied once per
// 64-wide group to the fp32 accumulator:  s * sum(q x) + b * sum(x)  =  s * C + b * sum(x).
// K is split across the warps (whole groups), partial tiles meet in shared memory.  Within a block of 32 k the activations
// are stored permuted (k -> (k % 4) * 8 + (k / 16) * 4 + (k % 16) / 4) so that the pair of nibbles (t, t + 4) a thread
// peels off a packed word lines up with the (b0, b1) fragment it reads with one 128-bit load.
__device__ __forceinline__ uint32_t hsub2_u32(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("sub.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ void mma_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// Stage `m` activation rows as fp16 columns of the B operand (permuted k), their per-group sums, the raw fp32 residual copy
// and sum(x^2) per row.
__device__ __forceinline__ void stage_rows_mma(const MegaParams& p, const Sm& sm, const Ctx& cx, const InArgs& in, int m, int K, int gshift,
                                               const float* norm_w, bool keep_raw) {
  const int in4 = K >> 2;
  const int ngroups = K >> gshift;
  const int lanes_per_group = 1 << (gshift - 2);  // float4 chunks per scale group (16 for group 64)
  for (int mi = 0; mi < m; ++mi) {
    float ss = 0.f;
    __half* xcol = sm.xh + (size_t)mi * p.xh_stride;
    for (int f0 = 0; f0 < in4; f0 += kCons) {
      const int f = f0 + cx.tid;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      float s4 = 0.f;
      if (f < in4) {
        float4 nw = make_float4(1.f, 1.f, 1.f, 1.f);
        if (norm_w != nullptr) nw = __ldg(reinterpret_cast<const float4*>(norm_w) + f);  // in flight with the poll below
        const long long tp0 = cx.trace ? clock64() : 0;
        v = load_in(p, cx, sm.hl, in, mi, f);
        if (cx.trace) const_cast<Ctx&>(cx).wait_poll += clock64() - tp0;
        ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
        if (keep_raw) reinterpret_cast<float4*>(sm.xraw + mi * p.raw_ld)[f] = v;
        v.x *= nw.x; v.y *= nw.y; v.z *= nw.z; v.w *= nw.w;
        // x = hi + lo, both fp16: column mi carries hi, column mi + 4 carries lo, ONE MMA multiplies both (fp32-grade products)
        const __half h0 = __float2half_rn(v.x), h1 = __float2half_rn(v.y), h2 = __float2half_rn(v.z), h3 = __float2half_rn(v.w);
        const __half l0 = __float2half_rn(v.x - __half2float(h0)), l1 = __float2half_rn(v.y - __half2float(h1));
        const __half l2 = __float2half_rn(v.z - __half2float(h2)), l3 = __float2half_rn(v.w - __half2float(h3));
        s4 = (v.x + v.y) + (v.z + v.w);
        // k = 4f + i  ->  block 32: (k % 4) * 8 + (k / 16 % 2) * 4 + (k % 16) / 4
        const int blk = f >> 3, fin = f & 7;
        __half* dst = xcol + blk * 32 + (fin >> 2) * 4 + (fin & 3);
        dst[0] = h0; dst[8] = h1; dst[16] = h2; dst[24] = h3;
        __half* dlo = dst + (size_t)4 * p.xh_stride;
        dlo[0] = l0; dlo[8] = l1; dlo[16] = l2; dlo[24] = l3;
      }
      // per-group sums: the float4 chunks of one group sit in consecutive lanes
      for (int o = 1; o < lanes_per_group && o < 32; o <<= 1) s4 += __shfl_xor_sync(0xffffffffu, s4, o);
      if (f < in4 && (cx.tid & (lanes_per_group - 1)) == 0) sm.xsum[mi * ngroups + (f >> (gshift - 2))] = s4;
    }
    if (norm_w != nullptr) {
      ss = warp_sum(ss);
      if (cx.lane == 0) sm.red[mi * 16 + cx.warp] = ss;
    }
  }
  cbar();
}

template <int FMT>
__device__ __forceinline__ void gemv_mma(const MegaParams& p, const Sm& sm, Ctx& cx, const MegaLinear& L, int m, bool has_norm, float eps, int epi,
                                         u64* out, int ld_out, float* plain_out, int plain_ld) {
  const int K = L.in;
  const int row_bytes = L.row_bytes, srow_bytes = L.srow_bytes, nsub = L.nsub, sdt = L.sdt, gshift = L.group_shift;
  const int ngroups = K >> gshift;
  const int steps = 1 << (gshift - 5);  // 32-wide steps per group
  const Slice s = slice_of(L);
  const int g = cx.lane >> 2, t = cx.lane & 3;
  float* part = sm.part;
  for (int c = 0; c < s.nch; ++c) {
    const int slot = cx.slot;
    const long long tw0 = cx.trace ? clock64() : 0;
    mbar_wait(&sm.full[slot], cx.ring_ph);
    if (cx.trace) { cx.wait_full += clock64() - tw0; cx.trace[3] = clock64(); }
    const int row0 = s.r0 + c * s.rch;
    const int rows = min(s.rch, s.rows - c * s.rch);
    const int wb = rows * row_bytes, sb = rows * srow_bytes;
    const uint8_t* base = sm.ring + slot * p.slot_bytes;
    const int tiles = (rows + 15) >> 4;
    const int units = tiles * nsub;
    int nks = kCWarps / units;           // K slices (whole groups) per (tile, sub)
    if (nks > ngroups) nks = ngroups;
    if (nks < 1) nks = 1;
    // ---- partial tiles
    for (int w = cx.warp; w < units * nks; w += kCWarps) {
      const int unit = w / nks, ks = w - unit * nks;
      const int sub = unit / tiles, tile = unit - sub * tiles;
      const int g0 = (ks * ngroups) / nks, g1 = ((ks + 1) * ngroups) / nks;
      const uint8_t* sbase = base + sub * (wb + 2 * sb);
      const int ra = min(tile * 16 + g, rows - 1), rb = min(tile * 16 + g + 8, rows - 1);
      const uint8_t* wa = sbase + ra * row_bytes;
      const uint8_t* wbp = sbase + rb * row_bytes;
      const uint8_t* sca = sbase + wb + ra * srow_bytes;
      const uint8_t* scb = sbase + wb + rb * srow_bytes;
      const __half* xcol = sm.xh + (size_t)g * p.xh_stride + t * 8;
      const bool colv = (g & 3) < m;  // columns 0..3: hi halves of the activation rows, 4..7: their lo halves
      const int c0 = 2 * t, c1 = 2 * t + 1;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int grp = g0; grp < g1; ++grp) {
        float C[4] = {0.f, 0.f, 0.f, 0.f};
        for (int st = 0; st < steps; ++st) {
          const int k32 = grp * steps + st;
          uint4 xb = make_uint4(0u, 0u, 0u, 0u);
          if (colv) xb = *reinterpret_cast<const uint4*>(xcol + k32 * 32);
          if constexpr (FMT == W_Q4) {
            const uint4 va = *reinterpret_cast<const uint4*>(wa + k32 * 16);
            const uint4 vb = *reinterpret_cast<const uint4*>(wbp + k32 * 16);
            const int sh = 4 * t;
            auto dq = [&](uint32_t w) { return hsub2_u32(lop3_and_or(w >> sh, 0x000F000Fu, 0x64006400u), 0x64006400u); };  // (1024 + q) - 1024: exact
            mma_16816(C, dq(va.x), dq(vb.x), dq(va.y), dq(vb.y), xb.x, xb.y);
            mma_16816(C, dq(va.z), dq(vb.z), dq(va.w), dq(vb.w), xb.z, xb.w);
          } else {  // W_Q8: 4 codes per word, the pair (t, t + 4) is byte t of two consecutive words
            const uint4 va0 = *reinterpret_cast<const uint4*>(wa + k32 * 32), va1 = *reinterpret_cast<const uint4*>(wa + k32 * 32 + 16);
            const uint4 vb0 = *reinterpret_cast<const uint4*>(wbp + k32 * 32), vb1 = *reinterpret_cast<const uint4*>(wbp + k32 * 32 + 16);
            const uint32_t sel = (uint32_t)t | ((uint32_t)(4 + t) << 8);  // byte t of a -> byte 0, byte t of b -> byte 2
            auto pk = [&](uint32_t lo, uint32_t hi) { return hsub2_u32(lop3_and_or(__byte_perm(lo, hi, sel), 0x00FF00FFu, 0x64006400u), 0x64006400u); };
            mma_16816(C, pk(va0.x, va0.y), pk(vb0.x, vb0.y), pk(va0.z, va0.w), pk(vb0.z, vb0.w), xb.x, xb.y);
            mma_16816(C, pk(va1.x, va1.y), pk(vb1.x, vb1.y), pk(va1.z, va1.w), pk(vb1.z, vb1.w), xb.z, xb.w);
          }
        }
        float sa, ba, sbv, bb;
        if (sdt == Q3TTS_F32) {
          sa = reinterpret_cast<const float*>(sca)[grp]; ba = reinterpret_cast<const float*>(sca + sb)[grp];
          sbv = reinterpret_cast<const float*>(scb)[grp]; bb = reinterpret_cast<const float*>(scb + sb)[grp];
        } else {
          sa = scale_to_f32(reinterpret_cast<const unsigned short*>(sca)[grp], sdt); ba = scale_to_f32(reinterpret_cast<const unsigned short*>(sca + sb)[grp], sdt);
          sbv = scale_to_f32(reinterpret_cast<const unsigned short*>(scb)[grp], sdt); bb = scale_to_f32(reinterpret_cast<const unsigned short*>(scb + sb)[grp], sdt);
        }
        const float x0 = c0 < m ? sm.xsum[c0 * ngroups + grp] : 0.f, x1 = c1 < m ? sm.xsum[c1 * ngroups + grp] : 0.f;  // bias term: hi columns only
        acc[0] += sa * C[0] + ba * x0; acc[1] += sa * C[1] + ba * x1;
        acc[2] += sbv * C[2] + bb * x0; acc[3] += sbv * C[3] + bb * x1;
      }
      float* pt = part + w * 128;  // [16 rows][8 cols]
      pt[g * 8 + c0] = acc[0]; pt[g * 8 + c1] = acc[1];
      pt[(g + 8) * 8 + c0] = acc[2]; pt[(g + 8) * 8 + c1] = acc[3];
    }
    cbar();
    if (cx.trace) cx.trace[4] = clock64();
    // ---- reduce the K slices + epilogue: one thread per (row, activation row)
    for (int e = cx.tid; e < rows * m; e += kCons) {
      const int r = e / m, col = e - r * m;
      const int tile = r >> 4, r16 = r & 15;
      float inv_rms = 1.0f;
      if (has_norm) {
        float ssum = 0.f;
#pragma unroll
        for (int w = 0; w < kCWarps; ++w) ssum += sm.red[col * 16 + w];
        inv_rms = rsqrtf(ssum / (float)K + eps);
      }
      float res[2] = {0.f, 0.f};
      for (int sub = 0; sub < nsub; ++sub) {
        const float* pt = part + ((sub * tiles + tile) * nks) * 128 + r16 * 8 + col;
        float v = 0.f;
        for (int ks = 0; ks < nks; ++ks) v += pt[ks * 128] + pt[ks * 128 + 4];  // hi + lo columns
        res[sub] = v * inv_rms;
      }
      const int grow = row0 + r;
      float v = res[0];
      if (epi == E_SWIGLU) {
        float gg = v, uu = res[1];
        if (L.bias) { gg += L.bias[grow]; uu += L.bias[grow + L.out_eff]; }
        v = silu_f(gg) * uu;
      } else {
        if (L.bias) v += L.bias[grow];
        if (epi == E_ADD_RAW) v += sm.xraw[col * p.raw_ld + grow];
      }
      ll_store(out + (size_t)col * ld_out + grow, __float_as_uint(v), cx.ph);
      if (plain_out) plain_out[(size_t)col * plain_ld + grow] = v;
    }
    cbar();  // `part` and the ring slot are free again
    if (cx.lane == 0) mbar_arrive(&sm.empty[slot]);
    if (++cx.slot == p.n_ring) { cx.slot = 0; cx.ring_ph ^= 1u; }
  }
}

// ------------------------------------------------------------------------------------------------ attention phase
// item = (slot, kv head, key split).  rps rows per slot (2 only in code-predictor pass 0).  Writes unnormalised partial
// outputs + (max, sum) per head; the o-projection staging merges the splits.  A lane owns 4 consecutive head dims
// (one LL poll of 4 elements); the rotate-half partner of dim d is dim d ^ 64, i.e. lane ^ 16.
template <int G>
__device__ void attn_phase(const MegaParams& p, const Sm& sm, const Ctx& cx, const MegaStack& S, const float* q_norm, const float* k_norm, int rps,
                           bool talker, int cp_pos0, int l) {
  float* sc0 = reinterpret_cast<float*>(sm.xs);
  float* q = sc0;                        // [2][G][128]
  float* kcur = q + 2 * G * 128;         // [2][128]
  float* vcur = kcur + 256;              // [2][128]
  float* sc = vcur + 256;                // [G][kKeyTile]
  float* ored = sc + G * kKeyTile;       // [kKeyGroups][G][128]
  float* stat = ored + kKeyGroups * G * 128;  // [G][2]
  const int heads = S.heads, kv_heads = S.kv_heads, nsplit = S.nsplit, cap = S.capacity;
  const int n_items = p.n_slots * kv_heads * nsplit;
  const float scale = 0.08838834764831845f;  // 1 / sqrt(128)
  const uint32_t tag = cx.ph - 1u;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int slot = item / (kv_heads * nsplit);
    const int rem = item - slot * (kv_heads * nsplit);
    const int kvh = rem / nsplit, sp = rem - kvh * nsplit;
    int pos0 = cp_pos0, w0 = 0;
    if (talker) {  // position / window of this frame's talker step: published by CTA 0 with code0
      pos0 = (int)ll_load1(msg_at(p, cx.fseq, 0, slot) + 1, cx.fseq);
      w0 = (int)ll_load1(msg_at(p, cx.fseq, 0, slot) + 2, cx.fseq);
    }
    const int w0r = w0 % cap;  // ring index of the window start; later keys wrap with one conditional subtract
    float* kb = S.k + (size_t)slot * S.slot_stride + (size_t)l * S.layer_stride + (size_t)kvh * cap * 128;
    float* vb = S.v + (size_t)slot * S.slot_stride + (size_t)l * S.layer_stride + (size_t)kvh * cap * 128;
    if (l == 0) {  // cos / sin of this unit's position(s): once per unit, not once per layer (precise sincosf is ~100 instructions)
      if (cx.tid < rps * 64) {
        const int rr = cx.tid >> 6, i = cx.tid & 63;
        float sn, cs;
        sincosf((float)(pos0 + rr) * S.inv_freq[i], &sn, &cs);
        sm.rope[(slot * 128 + cx.tid) * 2] = cs;
        sm.rope[(slot * 128 + cx.tid) * 2 + 1] = sn;
      }
      cbar();
    }
    // (a) per-head RMSNorm + rotate-half RoPE of q (G warps) and k (1 warp), v copy (1 warp) for each of the rps rows
    if (cx.warp < rps * (G + 2)) {
      const int rr = cx.warp / (G + 2), role = cx.warp - rr * (G + 2);
      const int row = slot * rps + rr, pos = pos0 + rr;
      const int ring = pos % cap;
      const u64* rowp = p.ex_qkv + (size_t)row * p.ld_qkv;
      const int lane = cx.lane;
      if (role <= G) {
        const int head = role < G ? (kvh * G + role) : (heads + kvh);
        const float4 a = ll_load4(rowp + (size_t)head * 128 + lane * 4, tag);
        const float ss = warp_sum(a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w);
        const float inv = rsqrtf(ss * (1.0f / 128.0f) + S.eps);
        const float4 nw = __ldg(reinterpret_cast<const float4*>(role < G ? q_norm : k_norm) + lane);
        const float4 x = make_float4(a.x * inv * nw.x, a.y * inv * nw.y, a.z * inv * nw.z, a.w * inv * nw.w);
        const float4* cs4 = reinterpret_cast<const float4*>(sm.rope + (slot * 128 + rr * 64 + 4 * (lane & 15)) * 2);  // [freq][cos, sin]
        const float4 t0 = cs4[0], t1 = cs4[1];
        const float4 cs = make_float4(t0.x, t0.z, t1.x, t1.z), sn = make_float4(t0.y, t0.w, t1.y, t1.w);
        float4 y;  // partner dims (d ^ 64)
        y.x = __shfl_xor_sync(0xffffffffu, x.x, 16); y.y = __shfl_xor_sync(0xffffffffu, x.y, 16);
        y.z = __shfl_xor_sync(0xffffffffu, x.z, 16); y.w = __shfl_xor_sync(0xffffffffu, x.w, 16);
        // q*cos + rotate_half(q)*sin, rotate_half = [-x2, x1]  (Model/Qwen3Layers.swift:187-195)
        const float sg = lane < 16 ? -1.0f : 1.0f;
        const float4 o = make_float4(x.x * cs.x + sg * y.x * sn.x, x.y * cs.y + sg * y.y * sn.y, x.z * cs.z + sg * y.z * sn.z, x.w * cs.w + sg * y.w * sn.w);
        float* dst = role < G ? q + (rr * G + role) * 128 : kcur + rr * 128;
        reinterpret_cast<float4*>(dst)[lane] = o;
        if (role == G && sp == 0) reinterpret_cast<float4*>(kb + (size_t)ring * 128)[lane] = o;  // append k (Model/Qwen3Layers.swift:197-201)
      } else {
        const float4 v = ll_load4(rowp + (size_t)(heads + kv_heads + kvh) * 128 + lane * 4, tag);
        reinterpret_cast<float4*>(vcur + rr * 128)[lane] = v;
        if (sp == 0) reinterpret_cast<float4*>(vb + (size_t)ring * 128)[lane] = v;
      }
    }
    cbar();
    for (int rr = 0; rr < rps; ++rr) {
      const int row = slot * rps + rr, pos = pos0 + rr;
      const int Sk = pos - w0 + 1;
      const int per = (Sk + nsplit - 1) / nsplit;
      const int j0 = sp * per, j1 = min(Sk, j0 + per);
      const int n = max(0, j1 - j0);
      if (n > kKeyTile) __trap();
      // (b) scores: one warp per key, the row of 128 floats is one coalesced 512-byte read
      for (int jb = cx.warp; jb < n; jb += 4 * kCWarps) {
        float4 kk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int jj = jb + u * kCWarps;
          kk[u] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (jj < n) {
            const int j = j0 + jj, back = (Sk - 1) - j;  // keys of this launch's own rows come from shared memory
            const int rj = w0r + j >= cap ? w0r + j - cap : w0r + j;
            kk[u] = (back <= rr) ? reinterpret_cast<const float4*>(kcur + (rr - back) * 128)[cx.lane] : ldcg4(kb + (size_t)rj * 128 + cx.lane * 4);
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int jj = jb + u * kCWarps;
          if (jj < n) {
#pragma unroll
            for (int g = 0; g < G; ++g) {
              const float4 qq = reinterpret_cast<const float4*>(q + (rr * G + g) * 128)[cx.lane];
              const float d = warp_sum(kk[u].x * qq.x + kk[u].y * qq.y + kk[u].z * qq.z + kk[u].w * qq.w);
              if (cx.lane == 0) sc[g * kKeyTile + jj] = d * scale;
            }
          }
        }
      }
      cbar();
      if (cx.warp < G) {  // softmax statistics of this split
        const int g = cx.warp;
        float mx = -INFINITY;
        for (int jj = cx.lane; jj < n; jj += 32) mx = fmaxf(mx, sc[g * kKeyTile + jj]);
        mx = warp_max(mx);
        float sum = 0.f;
        for (int jj = cx.lane; jj < n; jj += 32) { const float e = expf(sc[g * kKeyTile + jj] - mx); sc[g * kKeyTile + jj] = e; sum += e; }
        sum = warp_sum(sum);
        if (cx.lane == 0) { stat[2 * g] = mx; stat[2 * g + 1] = sum; }
      }
      cbar();
      if (cx.tid < kKeyGroups * 128) {  // (c) P.V: key groups x 128 dims
        const int d = cx.tid & 127, kg = cx.tid >> 7;
        float o[G];
#pragma unroll
        for (int g = 0; g < G; ++g) o[g] = 0.f;
        for (int jb = kg; jb < n; jb += 4 * kKeyGroups) {
          float vv[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int jj = jb + kKeyGroups * u;
            vv[u] = 0.f;
            if (jj < n) {
              const int j = j0 + jj, back = (Sk - 1) - j;
              const int rj = w0r + j >= cap ? w0r + j - cap : w0r + j;
              vv[u] = (back <= rr) ? vcur[(rr - back) * 128 + d] : __ldcg(vb + (size_t)rj * 128 + d);
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int jj = jb + kKeyGroups * u;
            if (jj < n) {
#pragma unroll
              for (int g = 0; g < G; ++g) o[g] = fmaf(sc[g * kKeyTile + jj], vv[u], o[g]);
            }
          }
        }
#pragma unroll
        for (int g = 0; g < G; ++g) ored[(kg * G + g) * 128 + d] = o[g];
      }
      cbar();
      u64* part = p.ex_part + (size_t)(row * nsplit + sp) * p.part_stride;
      if (cx.tid < G * 128) {
        const int g = cx.tid >> 7, d = cx.tid & 127;
        float o = 0.f;
#pragma unroll
        for (int kg = 0; kg < kKeyGroups; ++kg) o += ored[(kg * G + g) * 128 + d];
        ll_store(part + (kvh * G + g) * 128 + d, __float_as_uint(o), cx.ph);
      }
      if (cx.tid < 2 * G) ll_store(part + heads * 128 + 2 * kvh * G + cx.tid, __float_as_uint(stat[cx.tid]), cx.ph);
      cbar();
    }
  }
}

// ------------------------------------------------------------------------------------------------ bookkeeping (CTA 0)
// record the frame, add code0 to its set, advance the trailing-text cursor (Model/Qwen3Talker.swift:526-549)
__device__ void finalize_bookkeeping(const MegaParams& p, int slot) {
  {
    SlotState& s = p.st[slot];
    if (!s.frame_alive) return;
    const int* codes = p.cur_codes + slot * 16;
    if (s.n_frames < p.max_frames) {
      for (int g = 0; g < 16; ++g) p.frames[((size_t)slot * p.max_frames + s.n_frames) * 16 + g] = codes[g];
      s.n_frames += 1;
    }
    const int c0 = codes[0];
    if (c0 >= 0 && c0 < p.set_words * 32) {
      unsigned* set0 = p.sets + (size_t)slot * 16 * p.set_words;
      set0[c0 >> 5] |= 1u << (c0 & 31);
    }
    if (s.trailing_idx < s.total_text) s.trailing_idx += 1;
  }
}

// pos++, step++, window trim every 15th step, max_tokens stop (Model/Qwen3Talker.swift:554-558; Qwen3Layers.swift:111-124)
__device__ void step_advance(const MegaParams& p, int slot) {
  {
    SlotState& s = p.st[slot];
    if (!s.frame_alive) return;
    s.pos += 1;
    s.step += 1;
    if (s.step % 15 == 0 && s.pos - s.win_start > p.window) s.win_start = s.pos - p.window;
    if (s.step >= s.max_tokens) s.finished = 1;
    s.frame_alive = 0;
  }
}

// CTA 0: code_u = sampleToken(logits of the previous unit); the id (and, for unit 0, position / window / text cursor of
// this frame) is published to every CTA as a per-frame message.  All SlotState traffic stays inside CTA 0.
__device__ __forceinline__ void sample_phase(const MegaParams& p, const Sm& sm, const Ctx& cx, int group, bool plain_logits) {
  float* sl = reinterpret_cast<float*>(sm.xs);
  BlockRed& br = *reinterpret_cast<BlockRed*>(sl + kMaxVocab);
  float* lg = sl + kMaxVocab + 64;  // staged logits of this CTA's slot
  const int s = blockIdx.x;          // the slot this CTA owns
  SamplerParams sp;
  sp.vocab = group == 0 ? p.V : p.Vc; sp.group = group; sp.codec_vocab = p.V; sp.eos_id = p.eos_id; sp.pad_id = p.pad_id;
  sp.groups = 16; sp.set_words = p.set_words;
  const int V = sp.vocab;
  if (plain_logits) {  // first unit of a launch: logits written by the prefill / the previous launch
    for (int i = cx.tid; i < V; i += kCons) lg[i] = p.logits0[(size_t)s * V + i];
  } else {
    for (int f = cx.tid; f < (V >> 2); f += kCons)
      reinterpret_cast<float4*>(lg)[f] = ll_load4(p.ex_logit + (size_t)s * p.ld_logit + (size_t)f * 4, cx.ph - 1u);
  }
  cbar();
  float* dump = group == 0 ? p.dump0 : p.dumpcp;
  const int dump_stride = group == 0 ? p.V : 15 * p.Vc, dump_off = group == 0 ? 0 : (group - 1) * p.Vc;
  // sample_slot indexes logits by slot: hand it a base that makes row `s` land on the staged copy
  sample_slot<1, kCons>(s, lg - (size_t)s * V, V, p.st, sp, p.sets, p.cur_codes, p.forced, p.max_frames, dump, dump_stride, dump_off, 0, sl, br);
  cbar();
  if (cx.tid == 0) {
    const SlotState& st = p.st[s];
    u64* m = msg_at(p, cx.fseq, group, s);
    if (group == 0) {
      ll_store(m + 1, (uint32_t)st.pos, cx.fseq);
      ll_store(m + 2, (uint32_t)st.win_start, cx.fseq);
      ll_store(m + 3, (uint32_t)(st.trailing_idx < st.total_text ? st.trailing_idx : -1), cx.fseq);
    }
    ll_store(m, (uint32_t)p.cur_codes[s * 16 + group], cx.fseq);
  }
}

// ------------------------------------------------------------------------------------------------ the frame loop
// ONE copy of every phase body: the 16 units of a frame (15 code-predictor passes + the talker step) run through the same
// loop over linear phases [mtp?] + layers x {qkv, o, gate|up, down} + head.

template <int FMT, int NS>
__global__ void __launch_bounds__(kMegaThreads, 1) frame_megakernel(const __grid_constant__ MegaParams p) {
  constexpr int M = 2 * NS;
  // packed formats with more than one utterance per launch: tensor-core GEMV (one utterance stays on the fp32 SIMT GEMV)
  constexpr bool kMma = (FMT == W_Q4 || FMT == W_Q8) && NS > 1;
  Sm sm;
  sm.ring = smem;
  sm.xs = reinterpret_cast<float4*>(smem + p.off_xs);
  sm.xsum = reinterpret_cast<float*>(smem + p.off_xsum);
  sm.xraw = reinterpret_cast<float*>(smem + p.off_xraw);
  sm.red = reinterpret_cast<float*>(smem + p.off_red);
  sm.full = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  sm.empty = sm.full + p.n_ring;
  sm.dsc = reinterpret_cast<MegaLinear*>(smem + p.off_dsc);
  sm.hl = reinterpret_cast<float*>(smem + p.off_hl);
  sm.rope = reinterpret_cast<float*>(smem + p.off_rope);
  sm.xh = reinterpret_cast<__half*>(smem + p.off_xs);
  sm.part = reinterpret_cast<float*>(smem + p.off_part);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int kDscVec = (int)(sizeof(MegaLinear) / 16);
  if (tid == 0) {
    for (int s = 0; s < p.n_ring; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], kCWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (tid < kDscVec) reinterpret_cast<uint4*>(&sm.dsc[0])[tid] = __ldg(reinterpret_cast<const uint4*>(&p.lin[0]) + tid);
  for (int s = 0; s < p.n_slots; ++s)  // h_last of the prefill / the previous launch
    for (int i = tid; i < p.H; i += kMegaThreads) sm.hl[s * p.raw_ld + i] = p.hlast[(size_t)s * p.H + i];
  __syncthreads();
  if (warp == kCWarps) {
    if (lane == 0) producer_loop(p, sm.ring, sm.full, sm.empty);
    return;
  }
  Ctx cx;
  cx.slot = 0; cx.ring_ph = 0; cx.ph = 0; cx.fseq = 0; cx.tid = tid; cx.lane = lane; cx.warp = warp;
  cx.trace = nullptr; cx.wait_full = 0; cx.wait_poll = 0;
  if (p.trace != nullptr && tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x / 2))
    cx.trace = p.trace + (size_t)(blockIdx.x == 0 ? 0 : 1) * p.trace_stride;
  const int ns = p.n_slots;
  int cur = 0;  // which of the two descriptor slots holds the current linear

  for (int f = 0; f < p.n_frames; ++f) {
    cx.fseq = (uint32_t)f + 1u;
    const bool last_frame = (f == p.n_frames - 1);
    for (int li = 0; li < p.n_lin; ++li) {
      const MegaLinear& L = sm.dsc[cur];
      const int flags = L.flags;
      const bool talker = (flags & MF_TALKER) != 0;
      const MegaStack& S = talker ? p.tk : p.cp;
      // next phase's descriptor: loaded now, parked in the other slot at the end of the phase (never on the critical path)
      uint4 nd = make_uint4(0u, 0u, 0u, 0u);
      if (tid < kDscVec) nd = __ldg(reinterpret_cast<const uint4*>(&p.lin[li + 1 < p.n_lin ? li + 1 : 0]) + tid);
      if (flags & MF_UNIT_START) {  // ---- sample phase (CTA 0): code_u from the logits of the previous unit
        ++cx.ph;
        if (blockIdx.x < (unsigned)ns) {  // CTA s owns slot s: its sampler state, its messages, its bookkeeping
          if (cx.trace) { cx.trace[0] = clock64(); cx.trace[1] = cx.trace[0]; cx.trace[6] = 0; cx.trace[7] = 20; }
          sample_phase(p, sm, cx, L.uidx, f == 0 && li == 0);
          if (cx.trace) cx.trace[2] = clock64();
          trace_close(cx);
          cbar();
        }
      }
      ++cx.ph;                       // ---- linear phase
      const int rps = (flags & MF_ROWS2) ? 2 : 1;
      const int rows = (flags & MF_HEAD) ? ns : ns * rps;
      const bool head0 = (flags & (MF_HEAD | MF_TALKER)) == (MF_HEAD | MF_TALKER);
      InArgs in;
      in.kind = L.in_kind; in.pass = L.pass; in.nsplit = S.nsplit; in.heads = S.heads;
      const int out_sel = L.out_sel;
      u64* out = out_sel == 0 ? p.ex_x : (out_sel == 1 ? p.ex_qkv : (out_sel == 2 ? p.ex_act : p.ex_logit));
      const int ld_out = out_sel == 0 ? p.ld_x : (out_sel == 1 ? p.ld_qkv : (out_sel == 2 ? p.ld_act : p.ld_logit));
      float* plain_out = (head0 && last_frame) ? p.logits0 : nullptr;  // the next launch (or the graph path) starts from plain logits
      const float* norm_w = L.norm_w;
      const float eps = S.eps;
      if (cx.trace) { cx.trace[0] = clock64(); cx.wait_full = 0; cx.wait_poll = 0; cx.trace[3] = cx.trace[4] = 0; }
      if constexpr (kMma) stage_rows_mma(p, sm, cx, in, rows, L.in, L.group_shift, norm_w, (flags & MF_KEEP_RAW) != 0);
      else stage_rows<FMT>(p, sm, cx, in, rows, L.in, norm_w, (flags & MF_KEEP_RAW) != 0);
      if (cx.trace) cx.trace[1] = clock64();
      if (head0) {  // h_last = final norm of the talker step: next frame's pass-0 input, kept per CTA
        for (int s = 0; s < ns; ++s) {
          float ss = 0.f;
          for (int w = 0; w < kCWarps; ++w) ss += sm.red[s * 16 + w];
          const float inv = rsqrtf(ss / (float)p.H + eps);
          for (int i = tid; i < p.H; i += kCons) {
            const float hv = sm.xraw[s * p.raw_ld + i] * inv * norm_w[i];
            sm.hl[s * p.raw_ld + i] = hv;
            if (last_frame && blockIdx.x == 0) p.hlast[(size_t)s * p.H + i] = hv;
          }
        }
      }
      if constexpr (kMma) {
        gemv_mma<FMT>(p, sm, cx, L, rows, norm_w != nullptr, eps, L.epi, out, ld_out, plain_out, p.V);
      } else {
        if (rps == 2 && !(flags & MF_HEAD)) gemv_rows<FMT, M, 1>(p, sm, cx, L, rows, norm_w != nullptr, eps, L.epi, out, ld_out, plain_out, p.V);
        else gemv_rows<FMT, NS, 2>(p, sm, cx, L, rows, norm_w != nullptr, eps, L.epi, out, ld_out, plain_out, p.V);
      }
      if (cx.trace) { cx.trace[2] = clock64(); cx.trace[6] = cx.wait_full; cx.trace[7] = L.tkind + (cx.wait_poll << 8); }
      if (head0 && blockIdx.x < (unsigned)ns && tid == 0) step_advance(p, blockIdx.x);
      const float* q_norm = L.q_norm;
      const float* k_norm = L.k_norm;
      const int layer = L.layer, unit = L.uidx;
      if (tid < kDscVec) reinterpret_cast<uint4*>(&sm.dsc[cur ^ 1])[tid] = nd;
      cur ^= 1;
      trace_close(cx);
      cbar();  // xs / xraw / descriptors are reused by the next phase
      if (flags & MF_ATTN) {
        ++cx.ph;                     // ---- attention phase (participants: one CTA per (slot, kv head, split))
        if ((flags & MF_FINALIZE) && blockIdx.x < (unsigned)ns && tid == 0) finalize_bookkeeping(p, blockIdx.x);
        if (blockIdx.x < (unsigned)(ns * S.kv_heads * S.nsplit)) {
          if (cx.trace) { cx.trace[0] = clock64(); cx.trace[1] = cx.trace[0]; cx.trace[6] = 0; cx.trace[7] = 10; }
          const int G = S.heads / S.kv_heads;
          const int cp_pos0 = unit == 0 ? 0 : unit + 1;
          if (G == 2) attn_phase<2>(p, sm, cx, S, q_norm, k_norm, rps, talker, cp_pos0, layer);
          else if (G == 1) attn_phase<1>(p, sm, cx, S, q_norm, k_norm, rps, talker, cp_pos0, layer);
          else attn_phase<4>(p, sm, cx, S, q_norm, k_norm, rps, talker, cp_pos0, layer);
          if (cx.trace) cx.trace[2] = clock64();
          trace_close(cx);
        }
      }
    }
  }
}

template <int FMT, int NS>
void launch_fmt(const LaunchCtx& c, const MegaPlan& plan, const MegaParams& p) {
  void* args[] = {const_cast<MegaParams*>(&p)};
  Q3_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(&frame_megakernel<FMT, NS>), dim3(plan.grid), dim3(kMegaThreads), args, plan.smem, c.stream));
}

template <int FMT, int NS>
void init_fmt() {
  Q3_CUDA(cudaFuncSetAttribute(frame_megakernel<FMT, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
}

}  // namespace

void init_mega_kernels() {
  init_fmt<W_Q4, 1>();
  init_fmt<W_Q4, kMegaMaxSlots>();
  init_fmt<W_Q8, 1>();
  init_fmt<W_Q8, kMegaMaxSlots>();
  init_fmt<W_BF16, 1>();
  init_fmt<W_F16, 1>();
  init_fmt<W_F32, 1>();
}

int mega_max_blocks_per_sm(int fmt, int slots, size_t smem_bytes) {
  int n = 0;
  cudaError_t e = cudaErrorInvalidValue;
  const bool multi = slots > 1;
  switch (fmt) {
    case W_Q4: e = multi ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, frame_megakernel<W_Q4, kMegaMaxSlots>, kMegaThreads, smem_bytes)
                         : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, frame_megakernel<W_Q4, 1>, kMegaThreads, smem_bytes); break;
    case W_Q8: e = multi ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, frame_megakernel<W_Q8, kMegaMaxSlots>, kMegaThreads, smem_bytes)
                         : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, frame_megakernel<W_Q8, 1>, kMegaThreads, smem_bytes); break;
    case W_BF16: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, frame_megakernel<W_BF16, 1>, kMegaThreads, smem_bytes); break;
    case W_F16: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, frame_megakernel<W_F16, 1>, kMegaThreads, smem_bytes); break;
    case W_F32: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, frame_megakernel<W_F32, 1>, kMegaThreads, smem_bytes); break;
    default: break;
  }
  return e == cudaSuccess ? n : 0;
}

void launch_frame_megakernel(const LaunchCtx& c, const MegaPlan& plan, int n_slots, int n_frames, float* dump0, float* dumpcp) {
  Q3_CHECK(plan.ok && n_slots >= 1 && n_slots <= plan.max_slots && n_frames >= 1, Q3TTS_ERR_INVALID_ARG, "frame megakernel: bad launch");
  MegaParams p = plan.p;
  p.n_slots = n_slots; p.n_frames = n_frames; p.dump0 = dump0; p.dumpcp = dumpcp;
  Q3_CUDA(cudaMemsetAsync(p.ex_base, 0, p.ex_bytes, c.stream));  // LL tags start from 0 in every launch
  switch (plan.fmt) {
    case W_Q4: if (plan.max_slots > 1) launch_fmt<W_Q4, kMegaMaxSlots>(c, plan, p); else launch_fmt<W_Q4, 1>(c, plan, p); break;
    case W_Q8: if (plan.max_slots > 1) launch_fmt<W_Q8, kMegaMaxSlots>(c, plan, p); else launch_fmt<W_Q8, 1>(c, plan, p); break;
    case W_BF16: launch_fmt<W_BF16, 1>(c, plan, p); break;
    case W_F16: launch_fmt<W_F16, 1>(c, plan, p); break;
    case W_F32: launch_fmt<W_F32, 1>(c, plan, p); break;
    default: fail(Q3TTS_ERR_BAD_CONFIG, "frame megakernel: unknown weight format %d", plan.fmt);
  }
  c.tick();
}

}  // namespace q3
