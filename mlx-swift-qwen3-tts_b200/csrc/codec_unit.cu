// One DecoderResidualUnit of the vocoder (Vocoder/SpeechTokenizer.swift:696-718) as ONE persistent tcgen05 kernel:
//
//     x' = x + conv1x1( snake2( conv7_dilated( snake1(x) ) ) ),      also emitted: snake_next(x') as the next contraction's operand
//
// for the thin stages (C = 96 / 192 channels, 16 640 - 49 920 rows per 26-frame window) where the two-kernel form was bound by
// its HBM round trips and epilogues, not by the tensor pipe (ncu, profiles/r01_ncu_full_codec_tc_gemm.md: the 1x1 convolutions ran
// at 4-5 % tensor / 35 % DRAM, and every unit wrote and re-read a [rows, C] fp16 intermediate).  Per 128-row tile:
//
//   warp 0    TMA producer: the snake1(x) tile WITH its causal halo (128 + 6*dil rows, once per 64-channel block -- every tap reads it
//             through a UMMA descriptor whose start is shifted by tap*dil rows), the 7 x kcs weight tiles of the dilated
//             convolution and the kcs weight tiles of the 1x1, all through one ring
//   warp 1    MMA issuer: conv7 of tile i+1 is issued BEFORE the 1x1 of tile i (two accumulators), so the tensor pipe works on the
//             next tile while the epilogue warps turn accumulator i into the 1x1's operand
//   warps 2+  epilogue sets (4 warps each, 32-column chunks round-robin):
//             E1: acc1 (+bias) -> snake2 -> fp16 -> TENSOR MEMORY (tcgen05.st): the intermediate is the A operand of the 1x1 straight
//                 from TMEM (tcgen05.mma with a TMEM A operand); it never touches shared or global memory
//             E2: acc2 (+bias) + residual x -> x' (fp16 stream) and snake_next(x') (fp16 operand of the next unit / block)
//
// HBM traffic per unit: read snake1(x) (+42 % halo, mostly L2) and x, write x' and snake_next(x'): 4 tile-sized streams instead of 7.
#include <cuda.h>

#include <algorithm>
#include <cstdio>
#include <vector>

#include "codec_unit.h"
#include "epi_io.cuh"
#include "gemm_tc.h"
#include "tc_ptx.cuh"

namespace q3 {

namespace {

using namespace tcptx;

constexpr int kTileM = 128;
constexpr int kBlockK = 64;
constexpr int kHaloRowsMax = 192;
constexpr int kHaloBytes = kHaloRowsMax * kBlockK * 2;  // 24 KB
constexpr int kTaps = 7;
constexpr int kMaxEpiSets = 3;                       // sets of 4 epilogue warps
constexpr int kMaxThreads = 64 + 128 * kMaxEpiSets;
constexpr int kMaxC = 192;
constexpr int kTraceTiles = 8;
constexpr int kTraceSlots = 12;
#define UNIT_STAMP(ti, slot)                                                                                              \
  do {                                                                                                                    \
    if (p.trace && (ti) < kTraceTiles) p.trace[((size_t)blockIdx.x * kTraceTiles + (ti)) * kTraceSlots + (slot)] = (unsigned long long)clock64(); \
  } while (0)

struct UnitParams {
  int Bt, T, C, dil;
  int tiles_per_batch, total_tiles, kcs, halo_rows;
  int a_stages, n_acc, b_stages, b_bytes;
  int h_col0, tmem_cols, epi_sets, tps, w7_reps, w1_reps;
  unsigned long long* trace;  // measurement hook (Q3TTS_CODEC_UNIT_TRACE): [CTA][kTraceTiles][kTraceSlots] clock stamps, or null
  const float *b7, *ea2, *ieb2, *b1, *ea3, *ieb3;
  const __half* res16;
  __half* outr16;
  __half* out16;
};

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]),
      "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}

__global__ void __launch_bounds__(kMaxThreads, 1)
codec_unit_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW7, const __grid_constant__ CUtensorMap tmW1,
                  const UnitParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int AST = p.a_stages, NACC = p.n_acc;
  uint8_t* sA = smem;                                   // [2][192 rows][128 B] halo tiles of snake1(x)
  uint8_t* sB = smem + (size_t)AST * kHaloBytes;        // [b_stages][tps][C rows][128 B] weight tiles (conv7 taps, then the 1x1)
  uint64_t* a_full = reinterpret_cast<uint64_t*>(sB + (size_t)p.b_stages * p.tps * p.b_bytes);
  uint64_t* a_empty = a_full + AST;
  uint64_t* b_full = a_empty + AST;
  uint64_t* b_empty = b_full + p.b_stages;
  uint64_t* acc1_full = b_empty + p.b_stages;  // [NACC] conv7 accumulator of a tile complete         (MMA -> epilogue)
  uint64_t* acc2_full = acc1_full + 3;         // [NACC] 1x1 accumulator complete                      (MMA -> epilogue)
  uint64_t* acc_empty = acc2_full + 3;         // [NACC] accumulator drained by E2                     (epilogue -> MMA)
  uint64_t* h_full = acc_empty + 3;            // [1] intermediate of a tile written to tensor memory   (epilogue -> MMA)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(h_full + 1);
  uint8_t* patches = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 127) & ~(uintptr_t)127);  // [epilogue warps][2 KB]

  __shared__ __align__(16) float s_b7[kMaxC], s_ea2[kMaxC], s_ieb2[kMaxC], s_b1[kMaxC], s_ea3[kMaxC], s_ieb3[kMaxC];
  for (int c = threadIdx.x; c < p.C; c += blockDim.x) {  // static parameters: no dependency on the predecessor kernel
    s_b7[c] = p.b7 ? p.b7[c] : 0.f;
    s_ea2[c] = p.ea2[c]; s_ieb2[c] = p.ieb2[c];
    s_b1[c] = p.b1 ? p.b1[c] : 0.f;
    s_ea3[c] = p.ea3[c]; s_ieb3[c] = p.ieb3[c];
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    for (int s = 0; s < AST; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    for (int s = 0; s < p.b_stages; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
    for (int s = 0; s < 3; ++s) { mbar_init(&acc1_full[s], 1); mbar_init(&acc2_full[s], 1); mbar_init(&acc_empty[s], 4 * p.epi_sets); }
    mbar_init(h_full, 4 * p.epi_sets);
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
  const int n_local = p.total_tiles > (int)blockIdx.x ? (p.total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  // k-steps (K = 16 each) of channel block kc that hold real channels (C = 96: the second block is half zero fill)
  auto ksteps = [&](int kc) { return p.C - kc * kBlockK >= kBlockK ? 4 : 2; };  // C % 32 == 0: a tail block holds 32 channels

  // Ring positions are counters that wrap (stage, parity of the round), never `it % stages` / `it / stages`: a runtime integer division is
  // ~35 dependent instructions (I2F, MUFU.RCP, F2I, fix-ups), and five of them per 12 KB weight stage in the single MMA-issuing thread WERE
  // the stage time of the first version (1 000 cycles per stage whatever the ring depth, tap alignment or L2 placement: the thread, not
  // the memory system or the tensor pipe, was the bottleneck -- tensor pipe 13 % active, L2 20 %).
  struct Ring {
    int s = 0, n;
    uint32_t ph = 0;
    bool wrapped = false;
    __device__ explicit Ring(int stages) : n(stages) {}
    __device__ void next() { if (++s == n) { s = 0; ph ^= 1u; wrapped = true; } }
  };
  // A ring stage holds p.tps weight tiles (two taps of one channel block, or two channel blocks of the 1x1, when a tile is <= 16 KB):
  // every wait / fence / commit / descriptor set-up of the issuing warps is paid once per stage, and at C <= 128 a single 12-16 KB
  // tile carries only ~150 cycles of tensor work against ~500 cycles of issue overhead.
  const int TPS = p.tps;
  const int stage_bytes = TPS * p.b_bytes;

  if (warp == 0) {
    {  // ---------------- TMA producer: warp-uniform loop, one elected lane issues
      const bool lead = elect_one();
      Ring ra(AST), rb(p.b_stages);
      bool waited = false;
      const int rep7 = (int)(blockIdx.x % (unsigned)p.w7_reps), rep1 = (int)(blockIdx.x % (unsigned)p.w1_reps);
      // n (<= TPS) weight tiles into the next ring stage: tile u = rows [row0 + u * row_step, + C) x channels [c0 + u * c_step, + 64)
      auto issue_stage = [&](const CUtensorMap* map, int n, int c0, int c_step, int row0, int row_step, int rep) {
        if (rb.wrapped) mbar_wait(&b_empty[rb.s], rb.ph ^ 1u);  // the MMAs of this stage's previous tenant have read it
        if (lead) {
          uint8_t* dst = sB + (size_t)rb.s * stage_bytes;
          mbar_expect_tx(&b_full[rb.s], (uint32_t)(n * p.b_bytes));
          for (int u = 0; u < n; ++u) tma_load_3d(dst + (size_t)u * p.b_bytes, map, &b_full[rb.s], c0 + u * c_step, row0 + u * row_step, rep);
        }
        rb.next();
      };
      int tile = (int)blockIdx.x;
      int bidx = tile / p.tiles_per_batch, tin = tile - bidx * p.tiles_per_batch;  // the only divisions: once per CTA
      const int step_b = (int)gridDim.x / p.tiles_per_batch, step_t = (int)gridDim.x - step_b * p.tiles_per_batch;
      for (int ti = 0; ti <= n_local; ++ti) {
        if (ti < n_local) {  // operands of conv7(ti)
          const int t0 = tin * kTileM;
          if (lead) UNIT_STAMP(ti, 7);  // producer: starts requesting the operands of conv7(ti)
          for (int kc = 0; kc < p.kcs; ++kc) {
            int tap = 0;
            if (!waited) {  // the first weight stages do not depend on the predecessor kernel
              for (int st = 0; st < p.b_stages && tap < kTaps; ++st) {
                const int n = kTaps - tap < TPS ? kTaps - tap : TPS;
                issue_stage(&tmW7, n, kc * kBlockK, 0, tap * p.C, p.C, rep7);
                tap += n;
              }
              pdl_wait();
              waited = true;
            }
            if (ra.wrapped) mbar_wait(&a_empty[ra.s], ra.ph ^ 1u);
            if (lead) {
              mbar_expect_tx(&a_full[ra.s], (uint32_t)(p.halo_rows * kBlockK * 2));
              tma_load_3d(sA + (size_t)ra.s * kHaloBytes, &tmA, &a_full[ra.s], kc * kBlockK, t0 - (kTaps - 1) * p.dil, bidx);
            }
            ra.next();
            while (tap < kTaps) {
              const int n = kTaps - tap < TPS ? kTaps - tap : TPS;
              issue_stage(&tmW7, n, kc * kBlockK, 0, tap * p.C, p.C, rep7);
              tap += n;
            }
          }
          if (lead) UNIT_STAMP(ti, 8);  // producer: last operand of conv7(ti) requested (stamps stay OUT of the per-stage loops)
          bidx += step_b; tin += step_t;  // next tile of this CTA: tile + gridDim.x
          if (tin >= p.tiles_per_batch) { tin -= p.tiles_per_batch; ++bidx; }
        }
        if (ti > 0)  // operands of conv1(ti - 1): the channel blocks of the 1x1 weight, TPS per stage
          for (int kc = 0; kc < p.kcs; kc += TPS) issue_stage(&tmW1, p.kcs - kc < TPS ? p.kcs - kc : TPS, kc * kBlockK, kBlockK, 0, 0, rep1);
      }
      if (!waited) pdl_wait();
    }
  } else if (warp == 1) {
    {  // ---------------- MMA issuer: the whole warp walks the loop, one elected lane issues
      const bool lead = elect_one();
      const uint32_t idesc = (1u << 4) | ((uint32_t)(p.C >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
      const uint32_t h_base = tmem_base + (uint32_t)p.h_col0;
      const uint32_t sA0 = smem_u32(sA), sB0 = smem_u32(sB);
      Ring ra(AST), rb(p.b_stages);
      int buf7 = 0, buf1 = 0;            // accumulator of conv7(ti) / conv1(ti - 1): ti % NACC without the division
      uint32_t use_par = 1;              // parity of (ti / NACC - 1): flips each time buf7 wraps
      bool reuse = false;                // ti >= NACC: the accumulator had a previous tenant
      uint32_t hpar = 0;
      for (int ti = 0; ti <= n_local; ++ti) {
        if (ti < n_local) {  // conv7(ti) -> accumulator buf7
          if (reuse) {
            mbar_wait(&acc_empty[buf7], use_par);
            tc_fence_after();
          }
          const uint32_t acc = tmem_base + (uint32_t)(buf7 * p.C);
          if (lead) UNIT_STAMP(ti, 0);  // conv7(ti): accumulator free, issue starts
          for (int kc = 0; kc < p.kcs; ++kc) {
            const int ks = ksteps(kc);
            const uint32_t a_base = sA0 + (uint32_t)ra.s * (uint32_t)kHaloBytes;
            for (int tap = 0; tap < kTaps; tap += TPS) {
              const int n = kTaps - tap < TPS ? kTaps - tap : TPS;
              mbar_wait(&b_full[rb.s], rb.ph);
              if (tap == 0) mbar_wait(&a_full[ra.s], ra.ph);
              tc_fence_after();
              const uint32_t b_base = sB0 + (uint32_t)rb.s * (uint32_t)stage_bytes;
              if (lead) {
                for (int u = 0; u < n; ++u) {
                  const uint64_t ad = umma_desc_rows(a_base + (uint32_t)((tap + u) * p.dil) * 128u);
                  const uint64_t bd = umma_desc(b_base + (uint32_t)u * (uint32_t)p.b_bytes);
                  umma_f16(acc, ad, bd, idesc, (kc | tap | u) != 0 ? 1u : 0u);
                  umma_f16(acc, ad + 2u, bd + 2u, idesc, 1u);
                  if (ks == 4) {
                    umma_f16(acc, ad + 4u, bd + 4u, idesc, 1u);
                    umma_f16(acc, ad + 6u, bd + 6u, idesc, 1u);
                  }
                }
                umma_commit(&b_empty[rb.s]);
              }
              rb.next();
            }
            if (lead) umma_commit(&a_empty[ra.s]);
            ra.next();
          }
          if (lead) {
            umma_commit(&acc1_full[buf7]);
            UNIT_STAMP(ti, 1);  // conv7(ti): all MMAs issued
          }
          if (++buf7 == NACC) { buf7 = 0; reuse = true; use_par ^= 1u; }
        }
        if (ti > 0) {  // conv1(ti - 1): A = the intermediate in tensor memory, D = the same accumulator columns (drained by E1)
          const uint32_t acc = tmem_base + (uint32_t)(buf1 * p.C);
          mbar_wait(h_full, hpar);
          hpar ^= 1u;
          tc_fence_after();
          if (lead) UNIT_STAMP(ti - 1, 2);  // conv1(ti - 1): intermediate ready, issue starts
          for (int kc0 = 0; kc0 < p.kcs; kc0 += TPS) {
            const int n = p.kcs - kc0 < TPS ? p.kcs - kc0 : TPS;
            mbar_wait(&b_full[rb.s], rb.ph);
            tc_fence_after();
            const uint32_t b_base = sB0 + (uint32_t)rb.s * (uint32_t)stage_bytes;
            if (lead) {
              for (int u = 0; u < n; ++u) {
                const int kc = kc0 + u;
                const uint64_t bd = umma_desc(b_base + (uint32_t)u * (uint32_t)p.b_bytes);
                const uint32_t ha = h_base + (uint32_t)(kc * 32);
                umma_f16_ts(acc, ha, bd, idesc, kc != 0 ? 1u : 0u);
                umma_f16_ts(acc, ha + 8u, bd + 2u, idesc, 1u);
                if (ksteps(kc) == 4) {
                  umma_f16_ts(acc, ha + 16u, bd + 4u, idesc, 1u);
                  umma_f16_ts(acc, ha + 24u, bd + 6u, idesc, 1u);
                }
              }
              umma_commit(&b_empty[rb.s]);
            }
            rb.next();
          }
          if (lead) umma_commit(&acc2_full[buf1]);
          if (++buf1 == NACC) buf1 = 0;
        }
      }
    }
  } else {
    // ---------------- epilogue warps: warp w touches TMEM lanes [32*(w%4), +32); set e takes chunks e, e + sets, ...
    const int q = warp & 3, set = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const uint32_t h_base = tmem_base + (uint32_t)p.h_col0 + lane_off;
    const uint32_t patch = smem_u32(patches + (size_t)(warp - 2) * epiio::kPatchBytes);
    pdl_wait();
    int bidx = (int)blockIdx.x / p.tiles_per_batch, tin = (int)blockIdx.x - bidx * p.tiles_per_batch;
    const int step_b = (int)gridDim.x / p.tiles_per_batch, step_t = (int)gridDim.x - step_b * p.tiles_per_batch;
    int buf = 0;
    uint32_t upar = 0;  // parity of ti / NACC
    for (int ti = 0; ti < n_local; ++ti) {
      const int t0 = tin * kTileM;
      const uint32_t acc = tmem_base + (uint32_t)(buf * p.C) + lane_off;
      const int t = t0 + row;
      const bool row_ok = t < p.T;
      const size_t m = (size_t)bidx * p.T + t;
      // global memory is touched 8 rows x 64 B per warp instruction (epi_io.cuh), never one row per lane.  The residual rows of this
      // warp's first two chunks are requested now: their DRAM round trip hides behind E1
      const size_t wrow0 = (size_t)bidx * p.T + (size_t)(t0 + q * 32);
      const int wvalid = min(32, max(0, p.T - (t0 + q * 32)));
      uint4 rpre[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int c = (set + u * p.epi_sets) * 32;
        if (c < p.C) epiio::warp_load_64B_rows_issue(reinterpret_cast<const uint8_t*>(p.res16), wrow0, (size_t)p.C * 2, c * 2, rpre[u], lane, wvalid);
      }
      // ---- E1: conv7 accumulator -> bias -> snake2 -> fp16 pairs -> tensor memory
      mbar_wait(&acc1_full[buf], upar);
      tc_fence_after();
      if (threadIdx.x == 64) UNIT_STAMP(ti, 3);  // conv7(ti) complete (seen by the epilogue)
      for (int c = set * 32; c < p.C; c += 32 * p.epi_sets) {
        uint32_t raw[32];
        tmem_ld32(acc + (uint32_t)c, raw);
        uint32_t h[16];
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(s_b7 + c + j), a4 = *reinterpret_cast<const float4*>(s_ea2 + c + j),
                       i4 = *reinterpret_cast<const float4*>(s_ieb2 + c + j);
          float v0 = __uint_as_float(raw[j]) + b4.x, v1 = __uint_as_float(raw[j + 1]) + b4.y, v2 = __uint_as_float(raw[j + 2]) + b4.z,
                v3 = __uint_as_float(raw[j + 3]) + b4.w;
          const float s0 = __sinf(v0 * a4.x), s1 = __sinf(v1 * a4.y), s2 = __sinf(v2 * a4.z), s3 = __sinf(v3 * a4.w);
          v0 += i4.x * (s0 * s0); v1 += i4.y * (s1 * s1); v2 += i4.z * (s2 * s2); v3 += i4.w * (s3 * s3);
          h[j >> 1] = pack_h2(v0, v1);
          h[(j >> 1) + 1] = pack_h2(v2, v3);
        }
        tmem_st16(h_base + (uint32_t)(c >> 1), h);
      }
      tmem_st_wait();
      tc_fence_before();  // the accumulator reads and the tensor-memory writes are ordered before the barrier the MMA thread waits on
      __syncwarp();
      if (lane == 0) mbar_arrive(h_full);
      if (threadIdx.x == 64) UNIT_STAMP(ti, 4);  // E1 done
      // ---- E2: 1x1 accumulator -> bias + residual -> x' (fp16 stream) and snake_next(x') (fp16 operand)
      mbar_wait(&acc2_full[buf], upar);
      tc_fence_after();
      if (threadIdx.x == 64) UNIT_STAMP(ti, 5);  // conv1(ti) complete
      int ci = 0;
      for (int c = set * 32; c < p.C; c += 32 * p.epi_sets, ++ci) {
        uint32_t raw[32];
        tmem_ld32_issue(acc + (uint32_t)c, raw);
        uint4 rres[4];
        if (ci < 2) {
          if (ci == 0) epiio::warp_load_64B_rows_complete(rpre[0], rres, patch, lane);
          else epiio::warp_load_64B_rows_complete(rpre[1], rres, patch, lane);
        } else {
          uint4 tmp[4];
          epiio::warp_load_64B_rows_issue(reinterpret_cast<const uint8_t*>(p.res16), wrow0, (size_t)p.C * 2, c * 2, tmp, lane, wvalid);
          epiio::warp_load_64B_rows_complete(tmp, rres, patch, lane);
        }
        tmem_ld_wait32(raw);
        float v[32];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t w4[4] = {rres[j].x, rres[j].y, rres[j].z, rres[j].w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float2 r2 = __half22float2(*reinterpret_cast<const __half2*>(&w4[i]));
            const int e = 8 * j + 2 * i;
            v[e] = r2.x + (__uint_as_float(raw[e]) + s_b1[c + e]);
            v[e + 1] = r2.y + (__uint_as_float(raw[e + 1]) + s_b1[c + e + 1]);
          }
        }
        uint4 o4[4];
        if (p.outr16) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            o4[j] = make_uint4(pack_h2(v[8 * j], v[8 * j + 1]), pack_h2(v[8 * j + 2], v[8 * j + 3]), pack_h2(v[8 * j + 4], v[8 * j + 5]),
                               pack_h2(v[8 * j + 6], v[8 * j + 7]));
          epiio::warp_store_64B_rows(reinterpret_cast<uint8_t*>(p.outr16), wrow0, (size_t)p.C * 2, c * 2, o4, patch, lane, wvalid);
        }
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 a4 = *reinterpret_cast<const float4*>(s_ea3 + c + j), i4 = *reinterpret_cast<const float4*>(s_ieb3 + c + j);
          const float s0 = __sinf(v[j] * a4.x), s1 = __sinf(v[j + 1] * a4.y), s2 = __sinf(v[j + 2] * a4.z), s3 = __sinf(v[j + 3] * a4.w);
          v[j] += i4.x * (s0 * s0); v[j + 1] += i4.y * (s1 * s1); v[j + 2] += i4.z * (s2 * s2); v[j + 3] += i4.w * (s3 * s3);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          o4[j] = make_uint4(pack_h2(v[8 * j], v[8 * j + 1]), pack_h2(v[8 * j + 2], v[8 * j + 3]), pack_h2(v[8 * j + 4], v[8 * j + 5]),
                             pack_h2(v[8 * j + 6], v[8 * j + 7]));
        epiio::warp_store_64B_rows(reinterpret_cast<uint8_t*>(p.out16), wrow0, (size_t)p.C * 2, c * 2, o4, patch, lane, wvalid);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
      if (threadIdx.x == 64) UNIT_STAMP(ti, 6);  // E2 done
      if (++buf == NACC) { buf = 0; upar ^= 1u; }
      bidx += step_b; tin += step_t;
      if (tin >= p.tiles_per_batch) { tin -= p.tiles_per_batch; ++bidx; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

}  // namespace

bool codec_unit_shape_supported(int Bt, int T, int C, int dil) {
  if (C % 32 != 0 || C < 32 || C > kMaxC) return false;             // one CTA owns all C columns; 2.5 * C tensor-memory columns
  if (dil < 1 || kTileM + (kTaps - 1) * dil > kHaloRowsMax) return false;  // the halo tile is one 192-row stage
  if (Bt < 1 || T < 1 || (long long)Bt * ((T + kTileM - 1) / kTileM) < 32) return false;  // a few tiles: the two-kernel form (its <= 128-row variants) is fine
  return true;
}

static bool codec_unit_launchable(const CodecUnit& u) {
  if (!u.res16 || !u.out16 || !u.a || !u.w7 || !u.w1 || !u.snake2_ea || !u.next_ea) return false;
  return codec_unit_shape_supported(u.Bt, u.T, u.C, u.dil);
}

bool codec_unit_supported(const CodecUnit& u) {
  const char* e = getenv("Q3TTS_CODEC_UNIT");  // read per call: the A/B test flips it between two handles of one process
  if (e && atoi(e) == 0) return false;
  return codec_unit_launchable(u);
}

void init_codec_unit() {
  tc_resolve_encode();
  Q3_CUDA(cudaFuncSetAttribute(codec_unit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
}

void launch_codec_unit(const LaunchCtx& c, const CodecUnit& u) {
  Q3_CHECK(codec_unit_launchable(u), Q3TTS_ERR_INVALID_ARG, "codec_unit: unsupported shape (C %d, dilation %d, %d x %d rows)", u.C, u.dil, u.Bt, u.T);
  UnitParams p{};
  p.Bt = u.Bt; p.T = u.T; p.C = u.C; p.dil = u.dil;
  p.tiles_per_batch = (u.T + kTileM - 1) / kTileM;
  p.total_tiles = u.Bt * p.tiles_per_batch;
  p.kcs = (u.C + kBlockK - 1) / kBlockK;
  p.halo_rows = kTileM + (kTaps - 1) * u.dil;
  p.b_bytes = u.C * kBlockK * 2;
  // three accumulators when tensor memory allows (C <= 128): conv7 of tile i+2 runs while E2 drains tile i (with two, the tensor
  // pipe idles for the length of an E2 per tile); the halo ring holds two tiles' worth of channel blocks so that the next tile's
  // activations are in flight while this tile's MMAs run
  p.n_acc = 3 * u.C + u.C / 2 <= 512 ? 3 : 2;
  p.a_stages = 3;
  const int ring_budget = 212 * 1024 - 12 * epiio::kPatchBytes;  // 188 KB for the two operand rings
  p.tps = p.b_bytes <= 16 * 1024 ? 2 : 1;  // C <= 128: two weight tiles per ring stage
  const int sbytes = p.tps * p.b_bytes;
  if (sbytes * 3 + p.a_stages * kHaloBytes > ring_budget) p.a_stages = std::max(2, (ring_budget - 3 * sbytes) / kHaloBytes);
  p.b_stages = std::max(2, std::min(12, (ring_budget - p.a_stages * kHaloBytes) / sbytes));
  p.h_col0 = p.n_acc * u.C;
  int cols = 32;
  while (cols < p.n_acc * u.C + u.C / 2) cols <<= 1;
  p.tmem_cols = cols;
  p.epi_sets = std::max(1, std::min(kMaxEpiSets, u.C / 32));
  p.b7 = u.b7; p.ea2 = u.snake2_ea; p.ieb2 = u.snake2_ieb; p.b1 = u.b1; p.ea3 = u.next_ea; p.ieb3 = u.next_ieb;
  p.res16 = u.res16; p.outr16 = u.outr16; p.out16 = u.out16;

  const uint64_t adims[3] = {(uint64_t)u.C, (uint64_t)u.T, (uint64_t)u.Bt};
  const uint64_t astr[2] = {(uint64_t)u.C * 2, (uint64_t)u.T * u.C * 2};
  const uint32_t abox[3] = {(uint32_t)kBlockK, (uint32_t)p.halo_rows, 1};
  const CUtensorMap ma = tc_make_map(u.a, 3, adims, astr, abox);
  p.w7_reps = std::max(1, u.w7_reps); p.w1_reps = std::max(1, u.w1_reps);
  const uint64_t w7dims[3] = {(uint64_t)u.C, (uint64_t)kTaps * u.C, (uint64_t)p.w7_reps};
  const uint64_t w7str[2] = {(uint64_t)u.C * 2, p.w7_reps > 1 ? (uint64_t)u.w7_rep_stride * 2 : (uint64_t)kTaps * u.C * u.C * 2};
  const uint32_t wbox[3] = {(uint32_t)kBlockK, (uint32_t)u.C, 1};
  const CUtensorMap m7 = tc_make_map(u.w7, 3, w7dims, w7str, wbox);
  const uint64_t w1dims[3] = {(uint64_t)u.C, (uint64_t)u.C, (uint64_t)p.w1_reps};
  const uint64_t w1str[2] = {(uint64_t)u.C * 2, p.w1_reps > 1 ? (uint64_t)u.w1_rep_stride * 2 : (uint64_t)u.C * u.C * 2};
  const CUtensorMap m1 = tc_make_map(u.w1, 3, w1dims, w1str, wbox);

  const size_t smem = (size_t)p.a_stages * kHaloBytes + (size_t)p.b_stages * p.tps * p.b_bytes + 1024 + (size_t)(2 * p.a_stages + 2 * p.b_stages + 12) * 8 + 256 + (size_t)4 * p.epi_sets * epiio::kPatchBytes;
  Q3_CHECK(smem <= 220 * 1024 && p.tmem_cols <= 512, Q3TTS_ERR_CAPACITY, "codec_unit: resources (smem %zu, tmem %d)", smem, p.tmem_cols);
  dim3 grid((unsigned)std::min(p.total_tiles, 148));
  // measurement hook: Q3TTS_CODEC_UNIT_TRACE=<file> dumps the per-tile clock stamps of the first launch with C == Q3TTS_CODEC_UNIT_TRACE_C (96)
  static const char* trace_path = getenv("Q3TTS_CODEC_UNIT_TRACE");
  static bool traced = false;
  static const int trace_c = [] { const char* e = getenv("Q3TTS_CODEC_UNIT_TRACE_C"); return e ? atoi(e) : 96; }();
  unsigned long long* tbuf = nullptr;
  const size_t tn = (size_t)grid.x * kTraceTiles * kTraceSlots;
  if (trace_path && !traced && u.C == trace_c && !(c.counter && c.counter->capturing)) {
    traced = true;
    Q3_CUDA(cudaMalloc(&tbuf, tn * 8));
    Q3_CUDA(cudaMemsetAsync(tbuf, 0, tn * 8, c.stream));
  }
  p.trace = tbuf;
  launch_kernel_pdl(codec_unit_kernel, grid, dim3(64 + 128 * p.epi_sets), smem, c.stream, pdl_enabled(), ma, m7, m1, p);
  c.tick();
  if (tbuf) {
    std::vector<unsigned long long> h(tn);
    Q3_CUDA(cudaStreamSynchronize(c.stream));
    Q3_CUDA(cudaMemcpy(h.data(), tbuf, tn * 8, cudaMemcpyDeviceToHost));
    cudaFree(tbuf);
    if (FILE* f = fopen(trace_path, "w")) {
      fprintf(f, "{\"C\": %d, \"dil\": %d, \"ctas\": %u, \"tiles\": %d, \"slots\": %d, \"b_stages\": %d, \"a_stages\": %d, \"stamps\": [", u.C, u.dil, grid.x, kTraceTiles, kTraceSlots, p.b_stages, p.a_stages);
      for (size_t i = 0; i < tn; ++i) fprintf(f, "%s%llu", i ? "," : "", h[i]);
      fprintf(f, "]}\n");
      fclose(f);
    }
  }
}

}  // namespace q3
