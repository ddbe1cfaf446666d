// Pieces shared by the two <= 128-row split-K cluster GEMMs (gemm_skinny.cu: fp16 dense weights through TMA; gemm_skinny_q.cu:
// MLX-packed 4/8-bit weights dequantised inside the kernel): K split, parameter block, trace hooks, epilogue.
#pragma once
#include <cuda.h>

#include "gemm_tc.h"
#include "tc_ptx.cuh"

namespace q3 {
namespace skinny {

using namespace tcptx;

constexpr int kRowsW = 128;                     // weight rows per CTA = UMMA M
constexpr int kBlockK = 64;                     // fp16 elements per k-block = one 128-byte swizzle row
constexpr int kWBytes = kRowsW * kBlockK * 2;   // 16 KB of fp16 weights per stage
constexpr int kThreads = 192;
constexpr int kMaxSplit = 8;                    // K slices = cluster size; > 8 is a non-portable cluster size (B200 allows 16)
// up to ~1.3 waves: 48 weight tiles (gate|up) take 4 K slices = 192 CTAs of 4 k-blocks (two co-resident per SM on 44 SMs)
// rather than 96 CTAs of 8 k-blocks; measured 13.5 -> ~9 us per launch at 64 rows
constexpr int kCtaTarget = 200;

// The K split (= the fp32 summation order of the partial sums) of both kernels: it depends on the weight shape and the row bucket
// only, so the packed-weight kernel and the fp16-copy kernel produce the same bits.
inline int k_split(int tiles, int num_kb, int m_pad) {
  int split = 1;
  while (split * 2 <= kMaxSplit && tiles * split * 2 <= kCtaTarget && split * 2 <= num_kb && m_pad / (split * 2) >= 4) split *= 2;
  return split;
}

struct SkParams {
  int M, N, K;
  int m_pad, mc, mc_shift, split, stages, num_kb, tmem_cols;
  const float* bias;
  const float* res;
  int ld_res;
  const float* scale;
  int act, swiglu;
  float* out32;
  int ld32;
  __half* out16;
  int ld16;
  float out16_scale;
  const __half* rms_x;      // folded RMSNorm: fp16 activation rows [M][K] (= the B operand), or null
  float rms_a, rms_eps, rms_mult;  // row factor = rms_mult * rsqrt(sum(x16^2) * rms_a + rms_eps)
  unsigned long long* trace;  // measurement hook (q3tts_skinny_trace): 16 stamps per CTA, or null
  // ---- packed-weight kernel only (gemm_skinny_q.cu)
  const void* q_scales;     // [N][K / q_group] of q_sdt
  const void* q_biases;
  const float* q_fold;      // fp32 [K] multiplied into the dequantised columns (the RMSNorm weight in front of this linear), or null
  int q_group, q_sdt;
  int q_pstages;            // packed-tile ring depth
  int q_xstages, q_xown;    // activation stages in total / outside the (dead after dequantisation) packed region
  int q_half_rows;          // SwiGLU over a [gate ; up] matrix: rows of one half (N / 2); tile row 2i = gate i, 2i + 1 = up i.  0: plain rows
  int split_shift;          // log2(split)
};

__device__ __forceinline__ unsigned long long sk_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define SK_STAMP(slot)                                                                                        \
  do {                                                                                                        \
    if (p.trace) p.trace[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + (slot)] = (unsigned long long)clock64(); \
  } while (0)

__device__ __forceinline__ float sk_gelu_erf(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }
__device__ __forceinline__ float sk_silu(float v) { return v / (1.0f + expf(-v)); }
// SwiGLU feeds an fp16 operand (2^-11 relative rounding): the SFU exponential and reciprocal (2 ulp each) are invisible behind it
__device__ __forceinline__ float sk_silu_fast(float v) { return __fdividef(v, 1.0f + __expf(-v)); }

__device__ __forceinline__ float4 lds_f4(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

// sk_load_res: the residual values of the chunk (issued by the caller BEFORE it waits for the peers' partial sums).
// sk_finish: epilogue for `valid` (<= NC) consecutive activation rows m0.. of this thread's weight row (all 32 lanes call it together: the
// SwiGLU pairing is a lane shuffle).  Residual loads are issued first, stores last, so the round trips overlap; row pointers
// advance by their leading dimension (no 64-bit multiply per element: code size matters here, see below).
// ACT / SWIGLU are template parameters on purpose: with the exact erf and exponential expanded inline for every element of an
// unrolled chunk, one all-purpose epilogue was ~50 KB of SASS that ran once per launch at instruction-fetch speed (2.6 us
// per 16-column chunk measured); each instantiation now carries only its own math, at ONE call site.
template <int NC>
__device__ __forceinline__ void sk_load_res(const SkParams& p, float (&r)[NC], int valid, int m0, int ob) {
  if (p.res) {
    const float* rp = p.res + (size_t)m0 * p.ld_res + ob;
#pragma unroll
    for (int e = 0; e < NC; ++e, rp += p.ld_res) r[e] = e < valid ? *rp : 0.f;
  }
}
template <int NC, int ACT, bool SWIGLU>
__device__ __forceinline__ void sk_finish(const SkParams& p, float (&acc)[NC], const float (&r)[NC], int valid, int m0, int ob, float bias,
                                          float scale, const float* rowscale) {
#pragma unroll
  for (int e = 0; e < NC; ++e) {
    float v = acc[e];
    if (rowscale) v *= rowscale[e];  // folded RMSNorm of the input rows (shared memory, same value for the whole warp)
    v += bias;
    if (ACT == TC_ACT_GELU) v = sk_gelu_erf(v);
    else if (ACT == TC_ACT_SILU) v = sk_silu(v);
    if (SWIGLU) {  // weight rows (2i, 2i+1) = (gate_i, up_i): adjacent TMEM lanes = adjacent threads
      const float up = __shfl_xor_sync(0xffffffffu, v, 1);
      v = sk_silu_fast(v) * up;
    }
    if (p.res) v = r[e] + scale * v;
    acc[e] = v;
  }
  if (p.out32) {
    float* op = p.out32 + (size_t)m0 * p.ld32 + ob;
#pragma unroll
    for (int e = 0; e < NC; ++e, op += p.ld32)
      if (e < valid) *op = acc[e];
  }
  if (p.out16) {
    __half* hp = p.out16 + (size_t)m0 * p.ld16 + ob;
#pragma unroll
    for (int e = 0; e < NC; ++e, hp += p.ld16)
      if (e < valid) *hp = __float2half_rn(acc[e] * p.out16_scale);
  }
}

// The part of both kernels that follows "accumulator complete": TMEM -> shared staging grouped by owner, one bulk DSMEM copy
// per peer, fixed-order sum of the K slices of this CTA's activation rows, fused epilogue.  Called by the four epilogue warps
// (threads 64..191); `stage_out` (>= 128 * m_pad * 4 bytes, 16-byte aligned) may alias operand buffers no MMA reads any more.
template <int ACT, bool SWIGLU>
__device__ __forceinline__ void sk_reduce_epilogue(const SkParams& p, float* stage_out, float* red, uint64_t* red_full, uint64_t* ack, const float* rowscale_s,
                                                   uint32_t tmem_base, uint32_t rank, int n0) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = warp & 3;
  const int row = q * 32 + lane;
  const int n = n0 + row;
  const bool n_ok = n < p.N;
  const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
  const float bias = (p.bias && n_ok) ? p.bias[n] : 0.f;
  const int so = SWIGLU ? (n >> 1) : n;
  const float scale = (p.scale && n_ok) ? p.scale[so] : 1.f;
  // 1. TMEM -> local staging [owner][row][mc]
  for (int c0 = 0; c0 < p.m_pad; c0 += 32) {
    uint32_t raw[32];
    tmem_ld32(taddr + (uint32_t)c0, raw);
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const int col = c0 + j;
      const int dst = col >> p.mc_shift;          // owner of activation rows [dst*mc, +mc)
      const int off = col & (p.mc - 1);
      // slice of owner dst = [mc/4 column groups][128 rows][4]: a warp writes 512 contiguous bytes (no bank conflicts)
      *reinterpret_cast<float4*>(stage_out + (size_t)dst * kRowsW * p.mc + ((size_t)(off >> 2) * kRowsW + row) * 4) =
          make_float4(__uint_as_float(raw[j]), __uint_as_float(raw[j + 1]), __uint_as_float(raw[j + 2]), __uint_as_float(raw[j + 3]));
    }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the bulk-copy engine
  asm volatile("bar.sync 1, 128;" ::: "memory");                // the four epilogue warps
  // 2. one bulk DSMEM copy per peer: slice [owner = d] of my partial sums -> slot [src = rank] of d's `red`, signalling d's mbarrier
  const uint32_t slice_bytes = (uint32_t)(kRowsW * p.mc * 4);
  if (threadIdx.x == 64 && p.split > 1) {
    mbar_expect_tx(red_full, slice_bytes * (uint32_t)(p.split - 1));
    for (int i = 1; i < p.split; ++i) {
      const uint32_t d = (rank + (uint32_t)i) & (uint32_t)(p.split - 1);
      bulk_copy_to_rank(map_to_rank(smem_u32(red + (size_t)rank * kRowsW * p.mc), d), smem_u32(stage_out + (size_t)d * kRowsW * p.mc), slice_bytes,
                        map_to_rank(smem_u32(red_full), d));
    }
  }
  if (threadIdx.x == 64) SK_STAMP(5);
  // residual rows of the first chunk: requested now, they arrive while the peers' partial sums are still in flight
  const int m_base = (int)rank * p.mc;
  const bool lane_out = n_ok && (!SWIGLU || (n & 1) == 0);  // lanes without an output column compute (shuffle partners) but do not touch memory
  float r16[16];
  {
    int valid0 = p.M - m_base;
    valid0 = valid0 < 16 ? valid0 : 16;
    valid0 = valid0 < p.mc ? valid0 : p.mc;
    sk_load_res<16>(p, r16, lane_out ? valid0 : 0, m_base, so);
  }
  if (p.split > 1) mbar_wait(red_full, 0);  // the other K slices of MY activation rows have landed
  if (threadIdx.x == 96) SK_STAMP(10);
  if (threadIdx.x == 64) {
    SK_STAMP(6);
    // tell every peer that its copy into this CTA is complete (it may retire its staging buffer / exit)
    for (int i = 1; i < p.split; ++i) mbar_arrive_remote_relaxed(map_to_rank(smem_u32(ack), (rank + (uint32_t)i) & (uint32_t)(p.split - 1)));
  }
  const uint32_t own_s = smem_u32(stage_out), red_s = smem_u32(red);
  for (int cb = 0; cb < p.mc; cb += 16) {
    const int nc = p.mc - cb < 16 ? p.mc - cb : 16;
    float a16[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) a16[j] = 0.f;
    for (int s = 0; s < p.split; ++s) {  // fixed order: deterministic
      const uint32_t base = (s == (int)rank ? own_s : red_s) + (uint32_t)s * slice_bytes + (uint32_t)row * 16u;
#pragma unroll
      for (int c = 0; c < 16; c += 4) {
        if (c < nc) {
          const float4 v = lds_f4(base + (uint32_t)((cb + c) >> 2) * (uint32_t)(kRowsW * 16));
          a16[c] += v.x; a16[c + 1] += v.y; a16[c + 2] += v.z; a16[c + 3] += v.w;
        }
      }
    }
    if (threadIdx.x == 96 && cb == 0) SK_STAMP(11);
    int valid = p.M - (m_base + cb);
    valid = valid < nc ? valid : nc;
    if (!lane_out) valid = 0;
    if (cb > 0) sk_load_res<16>(p, r16, valid, m_base + cb, so);
    sk_finish<16, ACT, SWIGLU>(p, a16, r16, valid, m_base + cb, so, bias, scale, p.rms_x ? rowscale_s + cb : nullptr);
    if (threadIdx.x == 96 && cb == 0) SK_STAMP(12);
  }
  if (threadIdx.x == 96) SK_STAMP(13);
  if (threadIdx.x == 64 && p.split > 1) {
    SK_STAMP(7);
    mbar_wait(ack, 0);  // every peer has received my partial sums: my staging buffer is no longer being read
  }
}

// folded RMSNorm: factors of this CTA's activation rows, 8 lanes per row, 16 rows per pass of the four epilogue warps
__device__ __forceinline__ void sk_row_factors(const SkParams& p, float* rowscale_s, uint32_t rank) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = warp & 3;
  const int m_lo = (int)rank * p.mc, j = lane & 7;
  for (int r0 = 0; r0 < p.mc; r0 += 16) {
    const int r = r0 + q * 4 + (lane >> 3), m = m_lo + r;
    float ss = (r < p.mc && m < p.M) ? tc_row_sumsq_f16(p.rms_x + (size_t)m * p.K, p.K, j) : 0.f;
    ss = tc_group8_sum(ss);
    if (j == 0 && r < p.mc) rowscale_s[r] = p.rms_mult * rsqrtf(ss * p.rms_a + p.rms_eps);
  }
}

}  // namespace skinny
}  // namespace q3
