// Skinny tcgen05 GEMM for <= 128 activation rows (sm_100a): the linears of a batched decode step
// (Model/Qwen3Layers.swift:128-238 at L = 1 for many utterances at once) and of short codec windows.
//
//   Y[m, n] = epilogue( sum_k X[m, k] * W[n, k] ),   m < M <= 128
//
// At M <= 128 a [128 x bn] output tile per CTA (gemm_tc.cu) leaves N/bn CTAs each walking ALL of K and re-reading every
// activation row: the launch is bound by per-SM load latency (13-24 us for a 4-12 MB weight matrix).  Here the roles are
// swapped and K is split:
//   * the WEIGHT tile (128 rows of W) is the UMMA A operand, the activation rows are the N dimension (m_pad = 32/64/128
//     columns of the TMEM accumulator), so every weight byte enters exactly one CTA and the activation re-read is m_pad/128
//     of the weight traffic;
//   * the grid is (N/128 weight tiles) x (split K slices), one thread-block CLUSTER per weight tile; every CTA streams a
//     128 x (K/split) slice through a short TMA ring, so ~all SMs pull weights concurrently;
//   * the K slices are reduced through DISTRIBUTED SHARED MEMORY: CTA r of the cluster owns activation rows
//     [r*mc, (r+1)*mc); every CTA stages its TMEM accumulator in its own shared memory grouped by owner and ships each
//     owner's slice with ONE bulk copy (cp.async.bulk.shared::cluster, completion on the owner's mbarrier); the owner then
//     finishes bias / activation / SwiGLU / residual for its rows in a fixed summation order (deterministic, no atomics, no
//     zero-init, epilogues stay fused).  (Per-thread st.shared::cluster stores were measured at ~3 B/cycle: 2.9 us per 32
//     accumulator columns; the bulk engine moves the same bytes in a fraction of that.)
// Warp roles as in gemm_tc.cu: warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer, warps 2-5 epilogue.  Programmatic
// dependent launch: the first ring-full of WEIGHT tiles is requested before griddepcontrol.wait.
#include <cuda.h>

#include <algorithm>

#include "skinny_common.cuh"

namespace q3 {

namespace {

using namespace skinny;

template <int ACT, bool SWIGLU>
__global__ void __launch_bounds__(kThreads, 1)
tc_skinny_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX, const SkParams p) {
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B needs 1024-B aligned stages; the dynamic window starts at the same offset in every CTA of the kernel, so the
  // aligned offsets (and with them the DSMEM addresses of `red`) agree across the cluster.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int x_bytes = p.m_pad * kBlockK * 2;
  uint8_t* sW = smem;
  uint8_t* sX = smem + (size_t)p.stages * kWBytes;
  float* red = reinterpret_cast<float*>(sX + (size_t)p.stages * x_bytes);            // [split][128][mc]
  uint64_t* full = reinterpret_cast<uint64_t*>(red + (size_t)kRowsW * p.m_pad);
  uint64_t* empty = full + p.stages;
  uint64_t* tmem_full = empty + p.stages;
  uint64_t* red_full = tmem_full + 1;
  uint64_t* ack = red_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ack + 1);
  float* rowscale_s = reinterpret_cast<float*>(tmem_slot + 2);  // [mc] folded-RMSNorm factors of this CTA's activation rows

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = p.split > 1 ? cluster_ctarank() : 0u;   // cluster = (1, split, 1): the K slices of one weight tile
  const int n0 = blockIdx.x * kRowsW;
  // split is a power of two (host plan): shifts, not divisions -- a 64-bit division is ~100 instructions in front of the first weight request
  const int kb0 = (int)((rank * (uint32_t)p.num_kb) >> p.split_shift);
  const int kb1 = (int)(((rank + 1u) * (uint32_t)p.num_kb) >> p.split_shift);
  const int nkb = kb1 - kb0;

  pdl_launch_dependents();
  if (threadIdx.x == 32) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmW) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmX) : "memory");
  }
  if (threadIdx.x == 0) {
    if (p.trace) p.trace[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + 0] = sk_globaltimer();
    SK_STAMP(1);
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
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
  // phase A of the cluster barrier: "this CTA is running" (its shared memory may be written by peers once they passed wait A)
  if (p.split > 1) cluster_arrive_release();

  if (warp == 0) {
    {  // ---------------- TMA producer: warp-uniform loop, one elected lane issues (tc_ptx.cuh elect_one)
      const bool lead = elect_one();
      const int pre = nkb < p.stages ? nkb : p.stages;
      if (lead) {
        for (int i = 0; i < pre; ++i) {  // weights do not depend on the predecessor kernel
          mbar_expect_tx(&full[i], (uint32_t)(kWBytes + x_bytes));
          tma_load_2d(sW + (size_t)i * kWBytes, &tmW, &full[i], (kb0 + i) * kBlockK, n0);
        }
        // the k-blocks beyond the ring depth cannot be requested before a stage frees (after the dependency): prefetch their weight
        // tiles into L2 now, so that request is an L2 hit instead of a DRAM round trip on the critical path
        for (int i = pre; i < nkb; ++i) tma_prefetch_2d(&tmW, (kb0 + i) * kBlockK, n0);
      }
      pdl_wait();
      int s = 0;
      uint32_t ph = 0;  // ring position as wrapping counters: no integer division per k-block in the issuing threads
      for (int i = 0; i < nkb; ++i) {
        if (i >= pre) mbar_wait(&empty[s], ph ^ 1u);
        if (lead) {
          if (i >= pre) {
            mbar_expect_tx(&full[s], (uint32_t)(kWBytes + x_bytes));
            tma_load_2d(sW + (size_t)s * kWBytes, &tmW, &full[s], (kb0 + i) * kBlockK, n0);
          }
          tma_load_2d(sX + (size_t)s * x_bytes, &tmX, &full[s], (kb0 + i) * kBlockK, 0);
        }
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    {  // ---------------- MMA issuer: D[128 weight rows, m_pad activation rows] (+)= W_tile . X^T.  The whole warp walks the loop
       // (uniform registers), one elected lane issues (tc_ptx.cuh elect_one)
      const bool lead = elect_one();
      const uint32_t idesc = (1u << 4) | ((uint32_t)(p.m_pad >> 3) << 17) | ((uint32_t)(kRowsW >> 4) << 24);
      int s = 0;
      uint32_t ph = 0;
      for (int i = 0; i < nkb; ++i) {
        mbar_wait(&full[s], ph);
        tc_fence_after();
        if (lead && i == 0) SK_STAMP(3);
        const uint64_t ad = umma_desc(smem_u32(sW + (size_t)s * kWBytes));
        const uint64_t bd = umma_desc(smem_u32(sX + (size_t)s * x_bytes));
        if (lead) {
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k)
            umma_f16(tmem_base, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (i | k) != 0 ? 1u : 0u);
          umma_commit(&empty[s]);
        }
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
      if (lead) umma_commit(tmem_full);
    }
    __syncwarp();
  } else {
    // ---------------- epilogue warps: warp w may touch TMEM lanes [32*(w%4), +32); thread = one weight row
    pdl_wait();  // residual rows were written by earlier kernels
    if (p.rms_x) sk_row_factors(p, rowscale_s, rank);  // while the operands stream in
    if (p.split > 1) cluster_wait_acquire();  // A: every peer CTA is resident, its mbarriers initialised (long complete by now)
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    if (threadIdx.x == 64) SK_STAMP(4);
    // TMEM -> local staging (it aliases the operand ring: every MMA of this CTA has completed) -> DSMEM exchange -> epilogue
    sk_reduce_epilogue<ACT, SWIGLU>(p, reinterpret_cast<float*>(smem), red, red_full, ack, rowscale_s, tmem_base, rank, n0);
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

constexpr int kSmemKB = 108;  // operand ring + reduction buffer

struct SkPlan {
  int m_pad, split, stages, num_kb, tiles;
  size_t smem;
};

SkPlan plan(const TcGemm& g) {
  SkPlan s{};
  const int M = g.Bt * g.T;
  s.m_pad = M <= 32 ? 32 : (M <= 64 ? 64 : 128);
  s.tiles = (g.N + kRowsW - 1) / kRowsW;
  s.num_kb = (g.cin + kBlockK - 1) / kBlockK;
  s.split = k_split(s.tiles, s.num_kb, s.m_pad);
  const int stage_bytes = kWBytes + s.m_pad * kBlockK * 2;
  const int red_bytes = kRowsW * s.m_pad * 4;
  const int nkb_max = (s.num_kb + s.split - 1) / s.split;
  s.stages = std::max(2, (kSmemKB * 1024 - red_bytes) / stage_bytes);
  s.stages = std::max(1, std::min(s.stages, nkb_max));
  // the ring doubles as the outgoing staging buffer [owner][128][mc] fp32 (= red_bytes) once the MMAs are done
  while (s.stages * stage_bytes < red_bytes) ++s.stages;
  s.smem = (size_t)s.stages * stage_bytes + red_bytes + 1024 + (2 * s.stages + 4) * 8 + 16 + 128 * 4;
  return s;
}

}  // namespace

bool tc_skinny_supported(const TcGemm& g) {
  const long long M = (long long)g.Bt * g.T;
  return g.allow_skinny && !g.res16 && !g.outr16 && g.ntap == 1 && M >= 1 && M <= 128 && !g.snake_ea && !g.pcm && !(g.swiglu && g.act != TC_ACT_NONE) && tc_gemm_supported(g);
}

using SkKernel = void (*)(const CUtensorMap, const CUtensorMap, const SkParams);
static SkKernel pick_kernel(int act, int swiglu) {
  if (swiglu) return tc_skinny_kernel<TC_ACT_NONE, true>;
  if (act == TC_ACT_GELU) return tc_skinny_kernel<TC_ACT_GELU, false>;
  if (act == TC_ACT_SILU) return tc_skinny_kernel<TC_ACT_SILU, false>;
  return tc_skinny_kernel<TC_ACT_NONE, false>;
}

void init_tc_skinny() {
  tc_resolve_encode();
  for (SkKernel k : {pick_kernel(0, 1), pick_kernel(TC_ACT_GELU, 0), pick_kernel(TC_ACT_SILU, 0), pick_kernel(0, 0)})
    Q3_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  for (SkKernel k : {pick_kernel(0, 1), pick_kernel(TC_ACT_GELU, 0), pick_kernel(TC_ACT_SILU, 0), pick_kernel(0, 0)})
    Q3_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  init_tc_skinny_q();
}

unsigned long long* g_sk_trace = nullptr;  // set by tc_skinny_trace around its launches

void tc_skinny_set_trace(unsigned long long* dev_buf) { g_sk_trace = dev_buf; }
unsigned long long* tc_skinny_trace_buf() { return g_sk_trace; }
void tc_skinny_grid(const TcGemm& g, int* tiles, int* split, int* stages) {
  const SkPlan s = plan(g);
  *tiles = s.tiles; *split = s.split; *stages = s.stages;
}

void launch_tc_skinny(const LaunchCtx& c, const TcGemm& g) {
  if (tc_skinny_q_supported(g)) return launch_tc_skinny_q(c, g);  // packed 4/8-bit weights: dequantised inside the kernel
  Q3_CHECK(tc_skinny_supported(g), Q3TTS_ERR_INVALID_ARG, "tc_skinny: unsupported shape (rows %d, cin %d, N %d)", g.Bt * g.T, g.cin, g.N);
  tc_resolve_encode();
  const SkPlan s = plan(g);
  SkParams p{};
  p.M = g.Bt * g.T; p.N = g.N; p.K = g.cin;
  p.m_pad = s.m_pad; p.split = s.split; p.mc = s.m_pad / s.split; p.stages = s.stages; p.num_kb = s.num_kb;
  p.mc_shift = 0;
  while ((1 << p.mc_shift) < p.mc) ++p.mc_shift;
  p.split_shift = 0;
  while ((1 << p.split_shift) < p.split) ++p.split_shift;
  p.tmem_cols = std::max(32, s.m_pad);
  p.bias = g.bias; p.res = g.res; p.ld_res = g.ld_res; p.scale = g.scale; p.act = g.act; p.swiglu = g.swiglu;
  p.out32 = g.out32; p.ld32 = g.ld32; p.out16 = g.out16; p.ld16 = g.ld16;
  p.out16_scale = g.out16_scale;
  p.rms_x = g.rms_in ? g.a : nullptr;
  p.rms_a = 1.0f / (g.in_scale * g.in_scale * (float)g.cin); p.rms_eps = g.rms_eps; p.rms_mult = 1.0f / g.in_scale;
  Q3_CHECK(!g.row_scale, Q3TTS_ERR_INVALID_ARG, "tc_skinny: pass rms_in instead of precomputed row factors");
  p.trace = g_sk_trace;

  const uint64_t wdims[2] = {(uint64_t)g.cin, (uint64_t)g.N};
  const uint64_t wstr[1] = {(uint64_t)g.cin * 2};
  const uint32_t wbox[2] = {(uint32_t)kBlockK, (uint32_t)kRowsW};
  const CUtensorMap mw = tc_make_map(g.w, 2, wdims, wstr, wbox);
  const uint64_t xdims[2] = {(uint64_t)g.cin, (uint64_t)p.M};
  const uint64_t xstr[1] = {(uint64_t)g.cin * 2};
  const uint32_t xbox[2] = {(uint32_t)kBlockK, (uint32_t)s.m_pad};
  const CUtensorMap mx = tc_make_map(g.a, 2, xdims, xstr, xbox);

  Q3_CHECK(s.smem <= 220 * 1024, Q3TTS_ERR_CAPACITY, "tc_skinny: shared memory request %zu too large", s.smem);
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
  Q3_CUDA(cudaLaunchKernelEx(&cfg, pick_kernel(g.act, g.swiglu), mw, mx, p));
  c.tick();
}

}  // namespace q3
