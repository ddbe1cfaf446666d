// Dequant-fused skinny tcgen05 GEMM (sm_100a): MLXNN.QuantizedLinear / quantized_matmul (Model/QuantizedLayerFactory.swift:49-66)
// for <= 128 activation rows with the MLX-packed 4/8-bit weights as the STREAMED operand.
//
//   Y[m, n] = epilogue( sum_k X[m, k] * fp16( (scale[n, k/g] * q[n, k] + bias[n, k/g]) * fold[k] ) ),   m < M <= 128
//
// Same decomposition as gemm_skinny.cu (weight tile = UMMA A operand of 128 rows, activation rows = N dimension, K split over a
// thread-block cluster, K slices reduced through distributed shared memory, fused epilogue) -- but HBM is read in the
// checkpoint's own format: 0.5625 B / weight at 4-bit g64 instead of the 2 B / weight of an fp16 copy (SURVEY.md §8d).
//   * warp 0 (TMA producer) requests EVERY packed k-block of this CTA's K slice at kernel entry (uint32 tensor map, no swizzle:
//     a k-block is [128 rows][32 B] at 4 bits) -- weights never depend on the predecessor kernel -- then, after
//     griddepcontrol.wait, streams the fp16 activation k-blocks through a short ring;
//   * warps 2-5: one thread per weight row.  Per k-block it reads its 32 / 64 packed bytes, expands the codes with the
//     0x6400 exponent trick (4-bit) / PRMT (8-bit), applies scale and bias in fp32 exactly as MLX `dequantized` does
//     (deq32 = fp32(s) * q + fp32(b): the product is exact, so mul + add == fma), multiplies by the folded RMSNorm weight,
//     rounds ONCE to fp16 and writes the row into its own lane of tensor memory (tcgen05.st); an mbarrier hands the tile to the
//     MMA thread.  The bits that enter the tensor core are identical to the fp16 copies the engine used to keep
//     (q3tts_dequantize contract), so parity numbers do not move;
//   * warp 1 issues tcgen05.mma 128 x m_pad x 16 from (A in TMEM, X tile in shared memory) into TMEM, commits each stage back to the ring;
//   * warps 2-5 then run the shared reduce + epilogue (skinny_common.cuh).
#include <cuda.h>

#include <algorithm>

#include "skinny_common.cuh"

namespace q3 {

namespace {

using namespace skinny;

__device__ __forceinline__ uint32_t lop3_and_or(uint32_t a, uint32_t b, uint32_t c) {  // (a & b) | c in ONE LOP3
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t hsub2_u32(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("sub.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {  // round-to-nearest-even, lo in bits [0,16)
  uint32_t d;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
// Scales and biases of `ng` consecutive groups of one weight row -> column `my_sb` of the [2 * group + (0: scale, 1: bias)][128] table.
// SDT: 0 = bf16, 1 = f16, 2 = f32.  Batches of 8 groups: sixteen independent loads in flight, then the conversions and stores.
template <int SDT>
__device__ __forceinline__ void fill_sb_table(float* my_sb, const void* scales, const void* biases, size_t g_first, int ng, bool live) {
  for (int j0 = 0; j0 < ng; j0 += 8) {
    uint32_t rs[8], rb[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      rs[u] = rb[u] = 0u;
      if (live && j0 + u < ng) {
        if constexpr (SDT == 2) {
          rs[u] = __ldg(reinterpret_cast<const uint32_t*>(scales) + g_first + j0 + u);
          rb[u] = __ldg(reinterpret_cast<const uint32_t*>(biases) + g_first + j0 + u);
        } else {
          rs[u] = __ldg(reinterpret_cast<const unsigned short*>(scales) + g_first + j0 + u);
          rb[u] = __ldg(reinterpret_cast<const unsigned short*>(biases) + g_first + j0 + u);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (j0 + u < ng) {
        float fs, fb;
        if constexpr (SDT == 2) { fs = __uint_as_float(rs[u]); fb = __uint_as_float(rb[u]); }
        else if constexpr (SDT == 1) { fs = __half2float(__ushort_as_half((unsigned short)rs[u])); fb = __half2float(__ushort_as_half((unsigned short)rb[u])); }
        else { fs = __uint_as_float(rs[u] << 16); fb = __uint_as_float(rb[u] << 16); }
        my_sb[(2 * (j0 + u)) * kRowsW] = fs;
        my_sb[(2 * (j0 + u) + 1) * kRowsW] = fb;
      }
    }
  }
}
__device__ __forceinline__ uint4 lds_u4(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
  return v;
}

// 8 consecutive k of one weight row -> four packed fp16 pairs (one 16-byte chunk of the row).  q[8] are the integer codes as floats.
// MLX `dequantized` rounds the product and the sum separately (q3tts_dequantize contract).  With 16-bit scales the product s * q has
// <= 19 significant bits, i.e. it is exact, and one FMA gives the same bits; fp32 scales (24 + 8 bits) need the two roundings.
template <bool F32S>
__device__ __forceinline__ void pack_chunk(uint32_t* out4, const float (&q)[8], float sc, float bi, const float* fold8) {
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = F32S ? __fadd_rn(__fmul_rn(sc, q[e]), bi) : fmaf(sc, q[e], bi);
  if (fold8 != nullptr) {
    const float4 f0 = *reinterpret_cast<const float4*>(fold8), f1 = *reinterpret_cast<const float4*>(fold8 + 4);
    v[0] *= f0.x; v[1] *= f0.y; v[2] *= f0.z; v[3] *= f0.w;
    v[4] *= f1.x; v[5] *= f1.y; v[6] *= f1.z; v[7] *= f1.w;
  }
  out4[0] = pack_f16x2(v[0], v[1]); out4[1] = pack_f16x2(v[2], v[3]); out4[2] = pack_f16x2(v[4], v[5]); out4[3] = pack_f16x2(v[6], v[7]);
}

// One weight row of one k-block (64 k): packed bytes in shared memory -> 64 fp16 values in registers (out[4j .. 4j+3] = chunk j).
//   prow_s : shared address of the row's packed bytes (32 B at 4 bits, 64 B at 8 bits)
//   sc/bi  : scale and bias of the (up to two) groups the k-block touches: index 0 = k in [0, 32), 1 = k in [32, 64)
template <int BITS, bool F32S>
__device__ __forceinline__ void dequant_row(uint32_t prow_s, const float (&sc)[2], const float (&bi)[2], const float* fold64, uint32_t (&out)[32]) {
  if constexpr (BITS == 4) {
    const uint4 w0 = lds_u4(prow_s), w1 = lds_u4(prow_s + 16);
    const uint32_t w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {  // word j = k 8j .. 8j+7, nibble n at bits [4n, 4n+4)
      float q[8];
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        // (1024 + q_n, 1024 + q_{n+4}) as an fp16 pair in one shift + one LOP3; the subtraction is exact
        const uint32_t h = hsub2_u32(lop3_and_or(w[j] >> (4 * n), 0x000F000Fu, 0x64006400u), 0x64006400u);
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h));
        q[n] = f.x;
        q[n + 4] = f.y;
      }
      pack_chunk<F32S>(out + 4 * j, q, sc[j >> 2], bi[j >> 2], fold64 ? fold64 + 8 * j : nullptr);
    }
  } else {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const uint4 w0 = lds_u4(prow_s + 32 * half), w1 = lds_u4(prow_s + 32 * half + 16);
      const uint32_t w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {  // chunk = words 2jj, 2jj+1: byte b of word i = k 4i + b
        float q[8];
#pragma unroll
        for (int e = 0; e < 8; ++e)  // byte -> mantissa of 2^23 in one PRMT, exact subtraction
          q[e] = __uint_as_float(__byte_perm(w[2 * jj + (e >> 2)], 0x4B000000u, 0x7440u + (uint32_t)(e & 3))) - 8388608.0f;
        const int j = half * 4 + jj;
        pack_chunk<F32S>(out + 4 * j, q, sc[half], bi[half], fold64 ? fold64 + 8 * j : nullptr);
      }
    }
  }
}

// The dequantised weight tile is the MMA's A operand straight from TENSOR MEMORY: every k-block is written there once by its row's
// thread (tcgen05.st).
template <int BITS, bool SWIGLU>
__global__ void __launch_bounds__(kThreads, 1)
tc_skinny_q_kernel(const __grid_constant__ CUtensorMap tmP, const __grid_constant__ CUtensorMap tmX, const SkParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int kPBytes = kRowsW * kBlockK * BITS / 8;   // packed bytes of one k-block: 4 KB / 8 KB
  constexpr int kPRow = kBlockK * BITS / 8;              // per row and k-block: 32 B / 64 B
  const int x_bytes = p.m_pad * kBlockK * 2;
  const int PS = p.q_pstages, XS = p.q_xstages, XOWN = p.q_xown;
  uint8_t* sX = smem;                                             // [XOWN][m_pad rows][128 B] activation tiles (TMA, swizzled)
  uint8_t* sP = sX + (size_t)XOWN * x_bytes;                      // [PS][128 rows][kPRow] packed weight k-blocks (TMA, dense)
  float* red = reinterpret_cast<float*>(sP + (size_t)PS * kPBytes);  // [split][128][mc] landing buffer of the peers' partial sums
  // Activation stages XOWN .. XS-1 ALIAS the packed-weight region: every packed block has been dequantised (and is dead) before the
  // first activation tile is requested -- the producer waits for `pdone` -- so all XS = min(nkb, ...) activation k-blocks are in
  // flight at once after the dependency resolves, instead of two at a time behind the MMAs (measured: +0.9 us per launch).
  auto x_stage = [&](int xs) -> uint8_t* { return xs < XOWN ? sX + (size_t)xs * x_bytes : sP + (size_t)(xs - XOWN) * x_bytes; };
  uint64_t* afull = reinterpret_cast<uint64_t*>(red + (size_t)kRowsW * p.m_pad);  // every k-block of A is in tensor memory
  uint64_t* xfull = afull + 1;
  uint64_t* xempty = xfull + XS;
  uint64_t* pfull = xempty + XS;   // [0] only: the whole packed slice arrives with one (two: gate | up) tensor load(s)
  uint64_t* pdone = pfull + PS;
  uint64_t* tmem_full = pdone + 1;
  uint64_t* red_full = tmem_full + 1;
  uint64_t* ack = red_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ack + 1);
  // 16-byte aligned whatever the barrier count: rowscale [mc <= 128], then the [PS * 64] slice of the folded norm weight
  float* rowscale_s = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 15) & ~(uintptr_t)15);
  float* fold_s = rowscale_s + kRowsW;
  float* sb_s = fold_s + PS * kBlockK;  // [2 * q_ngm][128] scale / bias table of the CTA's K slice (thread = row owns a column)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = p.split > 1 ? cluster_ctarank() : 0u;
  const int n0 = blockIdx.x * kRowsW;
  const int kb0 = (int)((rank * (uint32_t)p.num_kb) >> p.split_shift);  // split is a power of two: no 64-bit division in front of the first request
  const int kb1 = (int)(((rank + 1u) * (uint32_t)p.num_kb) >> p.split_shift);
  const int nkb = kb1 - kb0;   // <= PS (host plan)

  pdl_launch_dependents();
  if (threadIdx.x == 32) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmP) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmX) : "memory");
  }
  if (threadIdx.x == 0) {
    if (p.trace) p.trace[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + 0] = sk_globaltimer();
    SK_STAMP(1);
    mbar_init(afull, 4);
    for (int s = 0; s < XS; ++s) { mbar_init(&xfull[s], 1); mbar_init(&xempty[s], 1); }
    for (int s = 0; s < PS; ++s) mbar_init(&pfull[s], 1);
    mbar_init(pdone, 4);
    mbar_init(tmem_full, 1);
    mbar_init(red_full, 1);
    mbar_init(ack, p.split > 1 ? p.split - 1 : 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) SK_STAMP(2);
  if (p.split > 1) cluster_arrive_release();  // phase A: "this CTA is running" (peers may write its shared memory after wait A)

  if (warp == 0) {
    if (lane == 0) {  // ---------------- TMA producer
      // The packed K slice of this CTA's 128 weight rows, now (weights are static): ONE box of [128 rows][PS k-blocks] -- rows of
      // PS * 32 B (4-bit) are whole 128-byte lines at PS = 4, where per-k-block boxes of 32-byte rows cost the TMA unit and DRAM a
      // request per row and k-block (measured: the dominant part of +2.7 us per launch against the fp16-copy kernel).
      const int wpk = kBlockK * BITS / 32;  // uint32 words of one packed row of a k-block
      mbar_expect_tx(&pfull[0], (uint32_t)(PS * kPBytes));
      if (p.q_half_rows) {  // tile rows (2i, 2i+1) = (gate_i, up_i): 64 rows of each half of the [gate ; up] matrix
        tma_load_2d(sP, &tmP, &pfull[0], kb0 * wpk, n0 / 2);
        tma_load_2d(sP + (size_t)PS * kPBytes / 2, &tmP, &pfull[0], kb0 * wpk, p.q_half_rows + n0 / 2);
      } else {
        tma_load_2d(sP, &tmP, &pfull[0], kb0 * wpk, n0);
      }
      pdl_wait();
      int xs = 0;
      uint32_t xph = 1;  // parity of (round - 1): ring positions are wrapping counters, no integer division per k-block
      for (int i = 0; i < nkb; ++i) {
        if (xs >= XOWN && i < XS) mbar_wait(pdone, 0);                        // the packed region is dead: its bytes may be overwritten
        if (i >= XS) mbar_wait(&xempty[xs], xph);                             // the MMAs of k-block i - XS have read this stage
        mbar_expect_tx(&xfull[xs], (uint32_t)x_bytes);
        tma_load_2d(x_stage(xs), &tmX, &xfull[xs], (kb0 + i) * kBlockK, 0);
        if (++xs == XS) { xs = 0; xph ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    {  // ---------------- MMA issuer: D[128 weight rows, m_pad activation rows] (+)= W_tile . X^T; warp-uniform loop, one elected lane issues
      const bool lead = elect_one();
      const uint32_t idesc = (1u << 4) | ((uint32_t)(p.m_pad >> 3) << 17) | ((uint32_t)(kRowsW >> 4) << 24);
      int xs = 0;
      uint32_t xph = 0;
      for (int i = 0; i < nkb; ++i) {
        if (i == 0) mbar_wait(afull, 0);
        mbar_wait(&xfull[xs], xph);
        tc_fence_after();
        if (lead && i == 0) SK_STAMP(3);
        const uint64_t bd = umma_desc(smem_u32(x_stage(xs)));
        const uint32_t at = tmem_base + (uint32_t)p.m_pad + (uint32_t)i * 32u;  // k-block i: 32 columns = 64 fp16 per lane
        if (lead) {
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) umma_f16_ts(tmem_base, at + (uint32_t)(8 * k), bd + (uint64_t)(2 * k), idesc, (i | k) != 0 ? 1u : 0u);
        }
        if (lead && i + XS < nkb) umma_commit(&xempty[xs]);
        if (++xs == XS) { xs = 0; xph ^= 1u; }
      }
      if (lead) umma_commit(tmem_full);
    }
    __syncwarp();
  } else {
    // ---------------- warps 2-5: dequantise this CTA's weight rows (thread = row), then reduce + epilogue
    const int q = warp & 3;
    const int row = q * 32 + lane;
    // weight row behind tile row `row`
    const int grow = p.q_half_rows ? ((row & 1) * p.q_half_rows + n0 / 2 + (row >> 1)) : (n0 + row);
    const int prow = p.q_half_rows ? ((row & 1) * (kRowsW / 2) + (row >> 1)) : row;
    const bool row_ok = p.q_half_rows ? (n0 / 2 + (row >> 1) < p.q_half_rows) : (grow < p.N);
    const int gpk = p.q_group >= kBlockK ? 1 : kBlockK / p.q_group;          // groups per k-block: 1 or 2
    const int gdiv = p.q_group >= kBlockK ? p.q_group / kBlockK : 1;         // k-blocks per group: 1 or 2
    const size_t srow = (size_t)grow * (size_t)(p.K / p.q_group);
    // The fold slice (the RMSNorm weight of the K slice) is requested FIRST and parked in registers, so that its DRAM round trip overlaps
    // the scale / bias loads' instead of following them (the stores of the table fill wait for their loads).
    constexpr int kFoldRegs = 8;  // nkb <= 16 (host plan): 16 * 64 / 128 threads
    float fv[kFoldRegs];
#pragma unroll
    for (int u = 0; u < kFoldRegs; ++u) {
      const int e = (int)threadIdx.x - 64 + u * 128, k = kb0 * kBlockK + e;
      fv[u] = (p.q_fold && e < nkb * kBlockK && k < p.K) ? __ldg(p.q_fold + k) : 0.f;
    }
    // Scales and biases of this row for EVERY k-block of the CTA's K slice, requested up front: all the loads of a batch of 8 groups are
    // in flight together and land in this thread's column of a shared-memory table.  (One k-block ahead, as the first version did, left
    // two dependent DRAM round trips in front of the first block and one L2 round trip inside every later one: measured 2000 of the 4600
    // cycles before the first block and 850 of the 1950 cycles of each later block.)
    const int g_lo = (kb0 * gpk) / gdiv;
    const int ng = nkb > 0 ? ((kb1 - 1) * gpk + gpk - 1) / gdiv - g_lo + 1 : 0;
    float* my_sb = sb_s + row;  // [2 * group + (0: scale, 1: bias)][128 rows]
    {
      const size_t g_first = srow + (size_t)g_lo;
      if (p.q_sdt == Q3TTS_F32) fill_sb_table<2>(my_sb, p.q_scales, p.q_biases, g_first, ng, row_ok);
      else if (p.q_sdt == Q3TTS_F16) fill_sb_table<1>(my_sb, p.q_scales, p.q_biases, g_first, ng, row_ok);
      else fill_sb_table<0>(my_sb, p.q_scales, p.q_biases, g_first, ng, row_ok);
    }
    auto load_sb = [&](int kb, float (&sc)[2], float (&bi)[2]) {  // this thread's own table column: no barrier needed
      const int gi = (kb * gpk) / gdiv - g_lo;
      sc[0] = my_sb[(2 * gi) * kRowsW];
      bi[0] = my_sb[(2 * gi + 1) * kRowsW];
      if (gpk == 2) {
        sc[1] = my_sb[(2 * gi + 2) * kRowsW];
        bi[1] = my_sb[(2 * gi + 3) * kRowsW];
      } else {
        sc[1] = sc[0];
        bi[1] = bi[0];
      }
    };
    if (p.q_fold) {
#pragma unroll
      for (int u = 0; u < kFoldRegs; ++u) {
        const int e = (int)threadIdx.x - 64 + u * 128;
        if (e < nkb * kBlockK) fold_s[e] = fv[u];
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
    const uint32_t prow0 = smem_u32(sP) + (uint32_t)prow * (uint32_t)(PS * kPRow);  // row pitch = the whole slice: PS k-blocks
    // Every k-block is dequantised NOW, ahead of the dependency on the predecessor kernel, into its own 32 TMEM columns (thread = TMEM
    // lane, packed fp16 pairs): k-block i is columns [m_pad + 32 i, +32) of this warp's lanes, the A operand of its MMAs.
    const uint32_t a0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)p.m_pad;
    for (int i = 0; i < nkb; ++i) {
      float sc[2], bi[2];
      load_sb(kb0 + i, sc, bi);
      if (i == 0) mbar_wait(&pfull[0], 0);
      uint32_t v[32];
      const float* fold = p.q_fold ? fold_s + i * kBlockK : nullptr;
      if (p.q_sdt == Q3TTS_F32) dequant_row<BITS, true>(prow0 + (uint32_t)i * (uint32_t)kPRow, sc, bi, fold, v);
      else dequant_row<BITS, false>(prow0 + (uint32_t)i * (uint32_t)kPRow, sc, bi, fold, v);
      tmem_st32(a0 + (uint32_t)i * 32u, v);
    }
    if (nkb > 0) tmem_st_wait();
    tc_fence_before();  // the tensor-memory writes are ordered before the barrier the MMA thread waits on
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(pdone);  // this warp has read its last packed byte
      mbar_arrive(afull);
    }
    if (threadIdx.x == 96) SK_STAMP(14);
    pdl_wait();  // residual rows and the activation rows were written by earlier kernels
    if (threadIdx.x == 96) SK_STAMP(15);
    if (p.rms_x) sk_row_factors(p, rowscale_s, rank);
    if (p.split > 1) cluster_wait_acquire();  // A: every peer CTA is resident, its mbarriers initialised
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    if (threadIdx.x == 64) SK_STAMP(4);
    // the X ring and the packed region are free (every MMA of this CTA has completed): they hold the outgoing partial sums
    sk_reduce_epilogue<TC_ACT_NONE, SWIGLU>(p, reinterpret_cast<float*>(smem), red, red_full, ack, rowscale_s, tmem_base, rank, n0);
  }
  if (p.split > 1 && warp < 2) cluster_wait_acquire();  // A (the epilogue warps passed it above)
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0 && p.trace) {
    SK_STAMP(8);
    p.trace[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + 9] = sk_globaltimer();
  }
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

struct SkqPlan {
  int m_pad, split, tiles, num_kb, nkb_max, x_own, x_stages, tmem_cols, ngm;
  size_t smem;
  bool ok;
};

SkqPlan plan(const TcGemm& g) {
  SkqPlan s{};
  const int M = g.Bt * g.T;
  s.m_pad = M <= 32 ? 32 : (M <= 64 ? 64 : 128);
  s.tiles = (g.N + kRowsW - 1) / kRowsW;
  s.num_kb = (g.cin + kBlockK - 1) / kBlockK;
  s.split = k_split(s.tiles, s.num_kb, s.m_pad);
  s.nkb_max = (s.num_kb + s.split - 1) / s.split;
  const int x_bytes = s.m_pad * kBlockK * 2, red_bytes = kRowsW * s.m_pad * 4;
  const int p_bytes = kRowsW * kBlockK * g.q_bits / 8;
  // quantisation groups a CTA's K slice can touch (scale / bias table rows)
  s.ngm = g.q_group == 32 ? 2 * s.nkb_max : (g.q_group == 64 ? s.nkb_max : s.nkb_max / 2 + 1);
  // the activation stages + the (dead) packed region double as the outgoing staging buffer
  s.x_own = 2;                                                                             // activation stages of their own ...
  while (s.x_own * x_bytes + s.nkb_max * p_bytes < red_bytes) ++s.x_own;
  s.x_stages = std::min(s.nkb_max, s.x_own + (s.nkb_max * p_bytes) / x_bytes);           // ... plus those that alias the packed region
  s.smem = (size_t)s.x_own * x_bytes + (size_t)s.nkb_max * p_bytes + red_bytes + 1024 +
           (size_t)(1 + 2 * s.x_stages + s.nkb_max + 4) * 8 + 16 + kRowsW * 4 + (size_t)s.nkb_max * kBlockK * 4 + (size_t)2 * s.ngm * kRowsW * 4 + 64;
  // TMEM: the fp32 accumulator [128 lanes x m_pad columns] + 32 columns per k-block of the dequantised A operand
  int cols = s.m_pad + 32 * s.nkb_max;
  s.tmem_cols = 32;
  while (s.tmem_cols < cols) s.tmem_cols <<= 1;
  // the packed slice is one TMA box: <= 256 elements in the inner dimension
  s.ok = s.smem <= 220 * 1024 && s.tmem_cols <= 512 && s.nkb_max * (kBlockK * g.q_bits / 32) <= 256 && s.nkb_max <= 16;
  return s;
}

using SkqKernel = void (*)(const CUtensorMap, const CUtensorMap, const SkParams);
SkqKernel pick_kernel(int bits, int swiglu) {
  if (bits == 4) return swiglu ? tc_skinny_q_kernel<4, true> : tc_skinny_q_kernel<4, false>;
  return swiglu ? tc_skinny_q_kernel<8, true> : tc_skinny_q_kernel<8, false>;
}

CUtensorMap make_packed_map(const void* base, uint64_t words_per_row, uint64_t rows, uint32_t box_words, uint32_t box_rows) {
  CUtensorMap m;
  const uint64_t dims[2] = {words_per_row, rows};
  const uint64_t strides[1] = {words_per_row * 4};
  const uint32_t box[2] = {box_words, box_rows};
  const uint32_t estr[2] = {1, 1};
  // L2 promotion 256 B: one row's consecutive k-blocks (32 B each at 4 bits) arrive with one DRAM burst for the whole cluster
  CUresult r = tc_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  Q3_CHECK(r == CUDA_SUCCESS, Q3TTS_ERR_CUDA, "cuTensorMapEncodeTiled (packed weights) failed with CUresult %d", (int)r);
  return m;
}

}  // namespace

bool tc_skinny_q_supported(const TcGemm& g) {
  if (!g.q_w || !(g.q_bits == 4 || g.q_bits == 8)) return false;
  if (!(g.q_group == 32 || g.q_group == 64 || g.q_group == 128)) return false;
  const long long M = (long long)g.Bt * g.T;
  if (!(g.allow_skinny && !g.res16 && !g.outr16 && g.ntap == 1 && M >= 1 && M <= 128 && !g.snake_ea && !g.pcm)) return false;
  if (g.act != TC_ACT_NONE || g.row_scale) return false;
  if (g.cin % kBlockK != 0 || g.cin % g.q_group != 0 || g.N % 32 != 0) return false;
  if (g.q_halves && (!g.swiglu || (g.N / 2) % (kRowsW / 2) != 0)) return false;
  if ((reinterpret_cast<uintptr_t>(g.q_w) & 15) != 0 || (reinterpret_cast<uintptr_t>(g.a) & 15) != 0) return false;
  return plan(g).ok;
}

void init_tc_skinny_q() {
  tc_resolve_encode();
  for (int bits : {4, 8})
    for (int sw : {0, 1}) {
      Q3_CUDA(cudaFuncSetAttribute(pick_kernel(bits, sw), cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
      Q3_CUDA(cudaFuncSetAttribute(pick_kernel(bits, sw), cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    }
}

void launch_tc_skinny_q(const LaunchCtx& c, const TcGemm& g) {
  Q3_CHECK(tc_skinny_q_supported(g), Q3TTS_ERR_INVALID_ARG, "tc_skinny_q: unsupported shape (rows %d, cin %d, N %d, bits %d, group %d)", g.Bt * g.T, g.cin, g.N,
           g.q_bits, g.q_group);
  tc_resolve_encode();
  const SkqPlan s = plan(g);
  SkParams p{};
  p.M = g.Bt * g.T; p.N = g.N; p.K = g.cin;
  p.m_pad = s.m_pad; p.split = s.split; p.mc = s.m_pad / s.split; p.num_kb = s.num_kb;
  p.mc_shift = 0;
  while ((1 << p.mc_shift) < p.mc) ++p.mc_shift;
  p.split_shift = 0;
  while ((1 << p.split_shift) < p.split) ++p.split_shift;
  p.tmem_cols = s.tmem_cols;
  p.bias = g.bias; p.res = g.res; p.ld_res = g.ld_res; p.scale = g.scale; p.act = g.act; p.swiglu = g.swiglu;
  p.out32 = g.out32; p.ld32 = g.ld32; p.out16 = g.out16; p.ld16 = g.ld16;
  p.out16_scale = g.out16_scale;
  p.rms_x = g.rms_in ? g.a : nullptr;
  p.rms_a = 1.0f / (g.in_scale * g.in_scale * (float)g.cin); p.rms_eps = g.rms_eps; p.rms_mult = 1.0f / g.in_scale;
  p.trace = tc_skinny_trace_buf();
  p.q_scales = g.q_scales; p.q_biases = g.q_biases; p.q_fold = g.q_fold; p.q_group = g.q_group; p.q_sdt = g.q_sdt;
  p.q_pstages = s.nkb_max;
  p.q_xstages = s.x_stages; p.q_xown = s.x_own;
  p.q_half_rows = g.q_halves ? g.N / 2 : 0;

  const uint32_t wpk = (uint32_t)(kBlockK * g.q_bits / 32) * (uint32_t)s.nkb_max;  // one box = the whole K slice of a row
  const CUtensorMap mp = make_packed_map(g.q_w, (uint64_t)g.cin * g.q_bits / 32, (uint64_t)g.N, wpk, (uint32_t)(g.q_halves ? kRowsW / 2 : kRowsW));
  const uint64_t xdims[2] = {(uint64_t)g.cin, (uint64_t)p.M};
  const uint64_t xstr[1] = {(uint64_t)g.cin * 2};
  const uint32_t xbox[2] = {(uint32_t)kBlockK, (uint32_t)s.m_pad};
  const CUtensorMap mx = tc_make_map(g.a, 2, xdims, xstr, xbox);

  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)s.tiles, (unsigned)s.split);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = s.smem;
  cfg.stream = c.stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (s.split > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = 1; attr[na].val.clusterDim.y = (unsigned)s.split; attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  Q3_CUDA(cudaLaunchKernelEx(&cfg, pick_kernel(g.q_bits, g.swiglu), mp, mx, p));
  c.tick();
}

}  // namespace q3
