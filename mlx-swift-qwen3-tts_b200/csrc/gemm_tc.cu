// tcgen05 + TMEM + TMA implicit GEMM (sm_100a).  One CTA = one 128 x BN output tile:
//   warp 0   : TMA producer   (cp.async.bulk.tensor into a ring of 128B-swizzled smem stages, mbarrier complete_tx)
//   warp 1   : TMEM allocator + single-thread tcgen05.mma issuer (UMMA 128 x BN x 16, fp16 in, fp32 accumulate in TMEM)
//   warps 2-5: epilogue       (tcgen05.ld 32x32b -> registers -> bias / activation / SwiGLU / residual+scale / fused
//                              SnakeBeta of the next layer -> fp32 and/or fp16 stores)
// Causal convolutions are K-loops over (tap, channel block): the A box of a tap is the same [128 time steps x 64 channels]
// tile shifted back in time; negative time coordinates are zero-filled by the TMA unit, which IS the causal left padding.
#include <cuda.h>
#include <cudaTypedefs.h>

#include <mutex>

#include "gemm_tc.h"
#include "epi_io.cuh"
#include "tc_ptx.cuh"

namespace q3 {

namespace {

using namespace tcptx;

constexpr int kTileM = 128;
constexpr int kBlockK = 64;                       // fp16 elements per k-block = one 128-byte swizzle row
constexpr int kABytes = kTileM * kBlockK * 2;     // 16 KB per stage
constexpr int kMaxEpiSets = 3;                            // sets of 4 epilogue warps (persistent schedule)
constexpr int kMaxThreads = 64 + 128 * kMaxEpiSets;       // warps 0-1 + the epilogue sets
constexpr int kPersistMinTiles = 4;                       // tiles per resident CTA from which the schedule is persistent

// Ring position as counters that wrap (stage, parity of the round) instead of `it % stages` / `(it / stages) & 1`: a runtime integer
// division is ~35 dependent instructions, and one or two per k-block in the single MMA-issuing (or TMA-issuing) thread cost more than
// the four MMAs of the k-block (measured in codec_unit.cu: the issuing thread, not memory or the tensor pipe, set the stage time).
__device__ __forceinline__ int fast_div(int x, unsigned mul, unsigned shift) {
  return (int)((__umulhi((unsigned)x, mul) + (unsigned)x) >> shift);
}

struct TcRing {
  int s = 0, n;
  uint32_t ph = 0;
  bool wrapped = false;
  __device__ explicit TcRing(int stages) : n(stages) {}
  __device__ void next() { if (++s == n) { s = 0; ph ^= 1u; wrapped = true; } }
};

struct TcParams {
  int Bt, T, cin, N, ntap, dil;
  int bn, stages, tiles_per_batch, kb_per_tap, tmem_cols;
  const float* bias;
  const float* res;
  int ld_res;
  const float* scale;
  int act, swiglu;
  float* out32;
  int ld32;
  __half* out16;
  int ld16;
  const float* snake_ea;
  const float* snake_ieb;
  int snake_ch;
  float* pcm;
  const float* row_scale;
  int k_rotate;
  // tile schedule: a CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ... of the (tiles_m x tiles_n) grid, n fastest.  One tile
  // per CTA (gridDim.x == tiles) is the classic launch; with fewer CTAs than tiles the kernel is PERSISTENT: the TMA ring runs on
  // across tile boundaries and two TMEM accumulators (n_acc = 2) let the epilogue of tile i overlap the MMAs of tile i + 1.
  int tiles_m, tiles_n, n_acc, acc_cols;
  // division by tiles_n / tiles_per_batch without the ~35-instruction software divide (every epilogue thread decomposes its tile index
  // once per tile: 5.8 % of a thin vocoder launch's instructions): q = (umulhi(x, mul) + x) >> shift, exact for x < 2^31
  unsigned div_n_mul, div_n_shift, div_b_mul, div_b_shift;
  const __half* res16;
  __half* outr16;
  int epi_sets;  // sets of 4 epilogue warps; set e handles the 32-column chunks e, e + epi_sets, ... of every tile
  // residual ring (fp16 residual stream, classic schedule): the [128 rows x bn] residual tile of a tile is fetched by the TMA producer
  // res_stages tiles ahead of the epilogue that adds it.  Per-thread residual loads kept ONE 2 KB batch per epilogue warp in flight
  // (12 warps x 2 KB / ~1.2 us of DRAM latency = 20 GB/s per SM -- exactly what the 1x1 convolutions of the vocoder ran at, 30-45 %
  // of their HBM roofline); through the ring the bytes in flight are res_stages whole tiles.
  int res_stages, res_bytes;
  // fp16 rows (res16 / outr16 / out16) move 8 rows x 64 B per warp instruction through a warp-private shared-memory patch (epi_io.cuh)
  // instead of one row per lane: the thin vocoder stages were bound by the load/store unit's line visits, not by HBM
  int tio;
  int w_reps;
};

__device__ __forceinline__ float gelu_erf(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }
__device__ __forceinline__ float silu(float v) { return v / (1.0f + expf(-v)); }

__global__ void __launch_bounds__(kMaxThreads, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmR, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);  // SWIZZLE_128B: 1024-B aligned
  const int b_bytes = p.bn * kBlockK * 2;
  uint8_t* sA = smem;
  uint8_t* sB = smem + (size_t)p.stages * kABytes;
  // full[s] / empty[s] guard stage s of both rings
  uint8_t* sR = sB + (size_t)p.stages * b_bytes;   // [res_stages][128 rows][bn] fp16 residual tiles (dense rows, no swizzle)
  uint64_t* full = reinterpret_cast<uint64_t*>(sR + (size_t)p.res_stages * p.res_bytes);
  uint64_t* empty = full + p.stages;
  uint64_t* tmem_full = empty + p.stages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;     // [2]
  uint64_t* rfull = tmem_empty + 2;         // [res_stages]
  uint64_t* rempty = rfull + p.res_stages;  // [res_stages]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rempty + p.res_stages);
  uint8_t* patches = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 127) & ~(uintptr_t)127);  // tio: [epilogue warps][2 KB]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kb = p.ntap * p.kb_per_tap;
  const int total_tiles = p.tiles_m * p.tiles_n;

  // Per-column epilogue constants (bias, the consumer's SnakeBeta pair) of this CTA's columns in shared memory: every epilogue
  // thread needs the same 32 values per chunk -- as global loads they were 24 of the 32 load instructions of a chunk.  One
  // column tile per kernel (tiles_n == 1: every thin vocoder layer) so the table is filled once; static parameters, no
  // dependency on the predecessor kernel.
  // Round 2b: the table holds ALL N columns (index = absolute column) when N <= 768, so layers of several column tiles (the 1x1 and
  // transposed convolutions at N = 288 / 384 / 768) use it too -- on the global-load path their epilogues stalled on the constants in
  // front of every sine (ncu source view: 18 % of the stall samples on that line, another 10 % of the instructions in modulo / index code).
  constexpr int kTabMax = 768;  // 9 KB static: two 100-KB-ring CTAs still share an SM
  __shared__ __align__(16) float s_bias[kTabMax], s_ea[kTabMax], s_ieb[kTabMax];
  const bool tab = p.tiles_n * p.bn <= kTabMax && !p.swiglu;
  if (tab) {
    for (int cidx = threadIdx.x; cidx < p.tiles_n * p.bn; cidx += blockDim.x) {
      const bool in = cidx < p.N;
      s_bias[cidx] = (p.bias && in) ? p.bias[cidx] : 0.f;
      if (p.snake_ea) {
        const int ch = cidx % p.snake_ch;
        s_ea[cidx] = p.snake_ea[ch];
        s_ieb[cidx] = p.snake_ieb[ch];
      }
    }
  }
  pdl_launch_dependents();  // the next kernel of the stream may start its prologue / weight prefetch now
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(&tmem_full[0], 1); mbar_init(&tmem_full[1], 1);
    mbar_init(&tmem_empty[0], 4 * p.epi_sets); mbar_init(&tmem_empty[1], 4 * p.epi_sets);  // one arrival per epilogue warp
    for (int s = 0; s < p.res_stages; ++s) { mbar_init(&rfull[s], 1); mbar_init(&rempty[s], 4 * p.epi_sets); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {  // one warp allocates TMEM columns for the fp32 accumulator tile(s) and later frees them
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    {  // ---------------- TMA producer: warp-uniform loop, one elected lane issues (tc_ptx.cuh elect_one)
      const bool lead = elect_one();
      const int w_rep = (int)(blockIdx.x % (unsigned)p.w_reps);  // this CTA's copy of the weights (TcGemm::w_reps)
      // Weights never depend on the previous kernel: the first ring-full of B tiles is requested BEFORE the programmatic
      // dependency is resolved, so the weight stream overlaps the predecessor's tail; activations (A) follow the wait.
      // Every CTA of a column of the grid reads the SAME activation tiles: walking K from a per-CTA offset keeps the CTAs
      // off each other's L2 lines (same-address storms serialise in one L2 slice and multiply the TMA latency).
      TcRing rg(p.stages);  // the ring does not care about tile boundaries
      int rt = 0;  // residual tiles issued so far (tile sequence numbers of this CTA)
      // residual tiles of this CTA's tiles [rt, upto].  blocking: wait for a stage's previous tenant to be consumed (only ever for the
      // tile the CTA is about to work on: its predecessors' loads are all issued, so their epilogues will run); otherwise stop at the
      // first stage that is still occupied -- the look-ahead must never stall the operand stream
      auto issue_residuals = [&](int upto, bool blocking) {
        for (; rt <= upto; ++rt) {
          const long long tl = (long long)blockIdx.x + (long long)rt * gridDim.x;
          if (tl >= total_tiles) { rt = 1 << 30; break; }
          const int mt = (int)(tl / p.tiles_n), nt = (int)(tl - (long long)mt * p.tiles_n);
          const int bi = mt / p.tiles_per_batch, tt0 = (mt - bi * p.tiles_per_batch) * kTileM;
          const int rs = rt % p.res_stages;
          if (rt >= p.res_stages) {
            const uint32_t par = (uint32_t)(((rt / p.res_stages) - 1) & 1);
            if (blocking) mbar_wait(&rempty[rs], par);
            else if (__shfl_sync(0xffffffffu, (int)mbar_try_wait(&rempty[rs], par), 0) == 0) break;  // one lane's answer for the whole warp
          }
          if (lead) {
            mbar_expect_tx(&rfull[rs], (uint32_t)p.res_bytes);
            tma_load_3d(sR + (size_t)rs * p.res_bytes, &tmR, &rfull[rs], nt * p.bn, tt0, bi);
          }
        }
      };
      for (int tile = blockIdx.x, ti = 0; tile < total_tiles; tile += gridDim.x, ++ti) {
        const int m_tile = fast_div(tile, p.div_n_mul, p.div_n_shift), n_tile = tile - m_tile * p.tiles_n;
        const int bidx = fast_div(m_tile, p.div_b_mul, p.div_b_shift), t0 = (m_tile - bidx * p.tiles_per_batch) * kTileM, n0 = n_tile * p.bn;
        const int rot = p.k_rotate ? (int)(((unsigned)n_tile * 5u + (unsigned)m_tile * 3u) % (unsigned)num_kb) : 0;
        if (p.res_stages && ti > 0 && rt < (1 << 30)) {
          issue_residuals(ti, true);
          if (rt < (1 << 30)) issue_residuals(ti + p.res_stages - 1, false);
        }
        int pre = 0;
        if (ti == 0) {
          pre = num_kb < p.stages ? num_kb : p.stages;
          int tp = rot / p.kb_per_tap, kc = rot - tp * p.kb_per_tap;  // (tap, channel block) of k-block `rot`, then counted up
          for (int kb = 0; kb < pre; ++kb) {
            if (lead) {
              mbar_expect_tx(&full[kb], (uint32_t)(kABytes + b_bytes));
              tma_load_3d(sB + (size_t)kb * b_bytes, &tmB, &full[kb], kc * kBlockK, tp * p.N + n0, w_rep);
            }
            if (++kc == p.kb_per_tap) { kc = 0; if (++tp == p.ntap) tp = 0; }
          }
          pdl_wait();
          if (p.res_stages) issue_residuals(p.res_stages - 1, true);  // the residual stream was written by the predecessor: after the wait
        }
        int tap = rot / p.kb_per_tap, kcb = rot - tap * p.kb_per_tap;
        for (int kb = 0; kb < num_kb; ++kb) {
          const int s = rg.s, c0 = kcb * kBlockK;
          const int shift = (p.ntap - 1 - tap) * p.dil;
          if (kb >= pre && rg.wrapped) mbar_wait(&empty[s], rg.ph ^ 1u);
          if (lead) {
            if (kb >= pre) {
              mbar_expect_tx(&full[s], (uint32_t)(kABytes + b_bytes));
              tma_load_3d(sB + (size_t)s * b_bytes, &tmB, &full[s], c0, tap * p.N + n0, w_rep);
            }
            tma_load_3d(sA + (size_t)s * kABytes, &tmA, &full[s], c0, t0 - shift, bidx);
          }
          rg.next();
          if (++kcb == p.kb_per_tap) { kcb = 0; if (++tap == p.ntap) tap = 0; }
        }
      }
    }
  } else if (warp == 1) {
    {  // ---------------- MMA issuer: the whole warp walks the loop (uniform registers), one elected lane issues (tc_ptx.cuh elect_one)
      const bool lead = elect_one();
      // instruction descriptor (cute::UMMA::InstrDescriptor): c = F32 (bit 4), a = b = F16 (0), K-major both, N>>3 at bit 17, M>>4 at bit 24
      const uint32_t idesc = (1u << 4) | ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
      TcRing rg(p.stages);
      const uint32_t sA0 = smem_u32(sA), sB0 = smem_u32(sB);
      for (int tile = blockIdx.x, ti = 0; tile < total_tiles; tile += gridDim.x, ++ti) {
        const int a = p.n_acc == 2 ? (ti & 1) : 0, use = p.n_acc == 2 ? (ti >> 1) : ti;
        if (use > 0) {  // the epilogue must have drained this accumulator's previous tile
          mbar_wait(&tmem_empty[a], (uint32_t)((use - 1) & 1));
          tc_fence_after();
        }
        const uint32_t acc = tmem_base + (uint32_t)(a * p.acc_cols);
        for (int kb = 0; kb < num_kb; ++kb) {
          const int s = rg.s;
          mbar_wait(&full[s], rg.ph);
          tc_fence_after();
          const uint64_t ad = umma_desc(sA0 + (uint32_t)s * (uint32_t)kABytes);
          const uint64_t bd = umma_desc(sB0 + (uint32_t)s * (uint32_t)b_bytes);
          if (lead) {
#pragma unroll
            for (int k = 0; k < kBlockK / 16; ++k)  // +32 bytes along K inside the swizzle atom = +2 in the (addr >> 4) field
              umma_f16(acc, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit(&empty[s]);  // frees the smem stage when these MMAs have read it
          }
          rg.next();
        }
        if (lead) umma_commit(&tmem_full[a]);  // accumulator complete
      }
    }
  } else {
    // ---------------- epilogue: warp w may touch TMEM lanes [32*(w%4), +32)
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t patch = smem_u32(patches + (size_t)(warp - 2) * epiio::kPatchBytes);
    pdl_wait();  // residual / bias-free inputs of the epilogue were written by earlier kernels
    for (int tile = blockIdx.x, ti = 0; tile < total_tiles; tile += gridDim.x, ++ti) {
    const int m_tile = fast_div(tile, p.div_n_mul, p.div_n_shift), n_tile = tile - m_tile * p.tiles_n;
    const int bidx = fast_div(m_tile, p.div_b_mul, p.div_b_shift), t0 = (m_tile - bidx * p.tiles_per_batch) * kTileM, n0 = n_tile * p.bn;
    const int acc_i = p.n_acc == 2 ? (ti & 1) : 0, use = p.n_acc == 2 ? (ti >> 1) : ti;
    const uint32_t acc = tmem_base + (uint32_t)(acc_i * p.acc_cols);
    const int t = t0 + row;
    const bool row_ok = t < p.T;
    const size_t m = (size_t)bidx * p.T + t;
    const size_t wrow0 = (size_t)bidx * p.T + (size_t)(t0 + q * 32);   // tio: this warp's first row and how many of its 32 exist
    const int wvalid = min(32, max(0, p.T - (t0 + q * 32)));
    const int rs = p.res_stages ? ti % p.res_stages : 0;
    if (p.res_stages) mbar_wait(&rfull[rs], (uint32_t)((ti / p.res_stages) & 1));  // this tile's residual rows are in shared memory
    mbar_wait(&tmem_full[acc_i], (uint32_t)(use & 1));
    tc_fence_after();
    for (int c = ((warp - 2) >> 2) * 32; c < p.bn; c += 32 * p.epi_sets) {
      uint32_t raw[32];
      tmem_ld32_issue(acc + ((uint32_t)(q * 32) << 16) + (uint32_t)c, raw);
      const int nb = n0 + c;
      const bool col_ok = nb < p.N;
      const bool live = row_ok && col_ok;
      // the residual row segment is requested while the TMEM load is in flight (the epilogue is latency bound: ncu showed its
      // warps waiting on exactly these global loads)
      const int width0 = p.swiglu ? 16 : 32, ob0 = p.swiglu ? (nb >> 1) : nb;
      float4 rres[8];
      if (p.res && live) {
        const float* rp = p.res + m * p.ld_res + ob0;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (4 * j < width0) rres[j] = *reinterpret_cast<const float4*>(rp + 4 * j);
      } else if (p.res_stages && live) {  // residual ring: row `row` of the staged [128][bn] tile, columns c .. c + 31
        const uint4* rp = reinterpret_cast<const uint4*>(sR + (size_t)rs * p.res_bytes + ((size_t)row * p.bn + (size_t)c) * 2);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (8 * j < width0) reinterpret_cast<uint4*>(rres)[j] = rp[j];
      } else if (p.res16 && p.tio && col_ok) {  // all lanes: four lanes fetch 64 contiguous bytes of one row, 8 rows per instruction
        uint4 tmp[4];
        epiio::warp_load_64B_rows_issue(reinterpret_cast<const uint8_t*>(p.res16), wrow0, (size_t)p.ld_res * 2, ob0 * 2, tmp, lane, wvalid);
#pragma unroll
        for (int j = 0; j < 4; ++j) reinterpret_cast<uint4*>(rres)[j] = tmp[j];
      } else if (p.res16 && live) {  // fp16 residual stream: 8 halves per 16-byte load, widened once they have arrived
        const uint4* rp = reinterpret_cast<const uint4*>(p.res16 + m * p.ld_res + ob0);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (8 * j < width0) reinterpret_cast<uint4*>(rres)[j] = rp[j];
      }
      tmem_ld_wait32(raw);
      if (p.tio ? !col_ok : !live) continue;
      if (p.tio && p.res16 && !p.res_stages) {  // hand every lane the 64 bytes of ITS row
        uint4 tmp[4], mine[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) tmp[j] = reinterpret_cast<uint4*>(rres)[j];
        epiio::warp_load_64B_rows_complete(tmp, mine, patch, lane);
#pragma unroll
        for (int j = 0; j < 4; ++j) reinterpret_cast<uint4*>(rres)[j] = mine[j];
      }
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(raw[j]);
      if (p.row_scale) {  // folded RMSNorm of the input row (TcGemm::row_scale)
        const float rs = row_ok ? p.row_scale[m] : 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] *= rs;
      }
      if (p.bias) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b4 = tab ? *reinterpret_cast<const float4*>(s_bias + nb + j) : *reinterpret_cast<const float4*>(p.bias + nb + j);
          v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
        }
      }
      if (p.act == TC_ACT_GELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
      } else if (p.act == TC_ACT_SILU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = silu(v[j]);
      }
      int width = 32, ob = nb;
      if (p.swiglu) {  // (gate, up) interleaved along n
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = silu(v[2 * j]) * v[2 * j + 1];
        width = 16;
        ob = nb >> 1;
      }
      if (p.res16) {  // widen in place, back to front (rres[j] takes halves 4j..4j+3 = the low/high half of 16-byte word j/2)
#pragma unroll
        for (int j = 7; j >= 0; --j) {
          if (4 * j < width) {
            const uint4 w16 = reinterpret_cast<const uint4*>(rres)[j >> 1];
            const uint32_t lo = (j & 1) ? w16.z : w16.x, hi = (j & 1) ? w16.w : w16.y;
            const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&lo)), f1 = __half22float2(*reinterpret_cast<const __half2*>(&hi));
            rres[j] = make_float4(f0.x, f0.y, f1.x, f1.y);
          }
        }
      }
      if (p.res || p.res16) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          if (j < width) {
            const float4 r4 = rres[j >> 2];
            float s0 = 1.f, s1 = 1.f, s2 = 1.f, s3 = 1.f;
            if (p.scale) { const float4 s4 = *reinterpret_cast<const float4*>(p.scale + ob + j); s0 = s4.x; s1 = s4.y; s2 = s4.z; s3 = s4.w; }
            v[j] = r4.x + s0 * v[j]; v[j + 1] = r4.y + s1 * v[j + 1]; v[j + 2] = r4.z + s2 * v[j + 2]; v[j + 3] = r4.w + s3 * v[j + 3];
          }
        }
      }
      if (p.pcm) {  // DecoderOutputConv: the tile's other 31 columns are zero padding of the 1-channel weight
        if (nb == 0) p.pcm[m] = (v[0] != v[0]) ? 0.0f : fminf(1.0f, fmaxf(-1.0f, v[0]));
        continue;
      }
      if (p.outr16 && p.tio) {
        uint4 o4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          __half2 h0 = __floats2half2_rn(v[8 * j], v[8 * j + 1]), h1 = __floats2half2_rn(v[8 * j + 2], v[8 * j + 3]);
          __half2 h2 = __floats2half2_rn(v[8 * j + 4], v[8 * j + 5]), h3 = __floats2half2_rn(v[8 * j + 6], v[8 * j + 7]);
          o4[j] = make_uint4(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1), *reinterpret_cast<uint32_t*>(&h2), *reinterpret_cast<uint32_t*>(&h3));
        }
        epiio::warp_store_64B_rows(reinterpret_cast<uint8_t*>(p.outr16), wrow0, (size_t)p.ld32 * 2, ob * 2, o4, patch, lane, wvalid);
      } else if (p.outr16) {
        __half* hp = p.outr16 + m * p.ld32 + ob;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          if (j < width) {
            __half2 h0 = __floats2half2_rn(v[j], v[j + 1]), h1 = __floats2half2_rn(v[j + 2], v[j + 3]);
            __half2 h2 = __floats2half2_rn(v[j + 4], v[j + 5]), h3 = __floats2half2_rn(v[j + 6], v[j + 7]);
            uint4 pk;
            pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
            pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
            *reinterpret_cast<uint4*>(hp + j) = pk;
          }
        }
      }
      if (p.out32) {
        float* op = p.out32 + m * p.ld32 + ob;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          if (j < width) *reinterpret_cast<float4*>(op + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      }
      if (p.out16) {
        if (p.snake_ea) {  // SnakeBeta of the consumer layer, applied to the fp16 operand copy only
          // One modulo per 32-column chunk (not per element), per-channel constants as float4, and the SFU sine: the result
          // is rounded to fp16 (2^-11) right after, MUFU.SIN's ~2^-21 absolute error is invisible behind it.  The precise
          // sinf + per-element modulo cost ~50 instructions per output value and made the thin-channel vocoder stages
          // epilogue-issue bound.
          const int ch0 = tab ? 0 : ob % p.snake_ch;
          const bool vec = (p.snake_ch & 3) == 0 && (ch0 & 3) == 0;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (j < width) {
              int c = ch0 + j;
              while (!tab && c >= p.snake_ch) c -= p.snake_ch;
              float ea[4], ib[4];
              if (tab) {  // absolute column ob + j: shared-memory table
                const float4 a4 = *reinterpret_cast<const float4*>(s_ea + ob + j), b4 = *reinterpret_cast<const float4*>(s_ieb + ob + j);
                ea[0] = a4.x; ea[1] = a4.y; ea[2] = a4.z; ea[3] = a4.w;
                ib[0] = b4.x; ib[1] = b4.y; ib[2] = b4.z; ib[3] = b4.w;
              } else if (vec) {
                const float4 a4 = __ldg(reinterpret_cast<const float4*>(p.snake_ea + c)), b4 = __ldg(reinterpret_cast<const float4*>(p.snake_ieb + c));
                ea[0] = a4.x; ea[1] = a4.y; ea[2] = a4.z; ea[3] = a4.w;
                ib[0] = b4.x; ib[1] = b4.y; ib[2] = b4.z; ib[3] = b4.w;
              } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  int ci = c + i;
                  while (ci >= p.snake_ch) ci -= p.snake_ch;
                  ea[i] = p.snake_ea[ci]; ib[i] = p.snake_ieb[ci];
                }
              }
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float sn = __sinf(v[j + i] * ea[i]);
                v[j + i] = v[j + i] + ib[i] * (sn * sn);
              }
            }
          }
        }
        __half* hp = p.out16 + m * p.ld16 + ob;
        if (p.tio) {
          uint4 o4[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            __half2 h0 = __floats2half2_rn(v[8 * j], v[8 * j + 1]), h1 = __floats2half2_rn(v[8 * j + 2], v[8 * j + 3]);
            __half2 h2 = __floats2half2_rn(v[8 * j + 4], v[8 * j + 5]), h3 = __floats2half2_rn(v[8 * j + 6], v[8 * j + 7]);
            o4[j] = make_uint4(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1), *reinterpret_cast<uint32_t*>(&h2), *reinterpret_cast<uint32_t*>(&h3));
          }
          epiio::warp_store_64B_rows(reinterpret_cast<uint8_t*>(p.out16), wrow0, (size_t)p.ld16 * 2, ob * 2, o4, patch, lane, wvalid);
        } else
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          if (j < width) {
            __half2 h0 = __floats2half2_rn(v[j], v[j + 1]), h1 = __floats2half2_rn(v[j + 2], v[j + 3]);
            __half2 h2 = __floats2half2_rn(v[j + 4], v[j + 5]), h3 = __floats2half2_rn(v[j + 6], v[j + 7]);
            uint4 pk;
            pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
            pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
            *reinterpret_cast<uint4*>(hp + j) = pk;
          }
        }
      }
    }
    // this warp has read its quarter of the accumulator: hand it back to the MMA issuer
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&tmem_empty[acc_i]);
    if (p.res_stages && lane == 0) mbar_arrive(&rempty[rs]);  // ... and its rows of the residual tile
    }  // tile loop
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

// Tile width: the largest multiple of 32 (<= 256) dividing N that still yields >= one CTA per SM; small-M problems (batched
// decode) fall through to narrow tiles so the weight stream is spread over many SMs.
int pick_bn(int N, int tiles_m) {
  int best = 0, smallest = 0;
  for (int bn = 256; bn >= 32; bn -= 32) {
    if (N % bn != 0) continue;
    smallest = bn;
    if (best == 0 && (long long)tiles_m * (N / bn) >= 148) best = bn;
  }
  if (best) return best;
  if (smallest) return smallest;
  return N <= 256 ? N : 256;
}

}  // namespace

namespace {
PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
std::once_flag g_encode_once;
}  // namespace

void tc_resolve_encode() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  });
  Q3_CHECK(g_encode != nullptr, Q3TTS_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
}

TcEncodeFn tc_encode_fn() {
  tc_resolve_encode();
  return reinterpret_cast<TcEncodeFn>(g_encode);
}

CUtensorMap tc_make_map(const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box) {
  CUtensorMap m;
  const uint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  Q3_CHECK(r == CUDA_SUCCESS, Q3TTS_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu x %llu)", (int)r, rank,
           (unsigned long long)dims[0], (unsigned long long)dims[1]);
  return m;
}

bool tc_gemm_supported(const TcGemm& g) {
  const int n_out = g.swiglu ? g.N / 2 : g.N;
  return g.cin % 8 == 0 && g.N % 32 == 0 && g.N >= 32 && g.T >= 1 && g.Bt >= 1 && (reinterpret_cast<uintptr_t>(g.a) & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(g.w) & 15) == 0 && (!g.out32 || (g.ld32 % 4 == 0)) && (!g.out16 || (g.ld16 % 8 == 0)) &&
         (!g.res || g.ld_res % 4 == 0) && n_out % 16 == 0;
}

void init_tc_gemm() {
  tc_resolve_encode();
  Q3_CUDA(cudaFuncSetAttribute(tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 212 * 1024));  // + 9 KB static (epilogue tables) + 1 KB reserved <= 227 KB
  init_tc_skinny();
}

void launch_tc_gemm(const LaunchCtx& c, const TcGemm& g) {
  if (tc_skinny_supported(g)) return launch_tc_skinny(c, g);  // <= 128 rows: split-K cluster kernel (gemm_skinny.cu)
  Q3_CHECK(tc_gemm_supported(g), Q3TTS_ERR_INVALID_ARG, "tc_gemm: unsupported shape (cin %d, N %d)", g.cin, g.N);
  Q3_CHECK(!g.rms_in && g.out16_scale == 1.0f, Q3TTS_ERR_INVALID_ARG, "tc_gemm: rms_in / out16_scale are features of the <= 128-row kernel (use row_scale)");
  tc_resolve_encode();
  TcParams p{};
  p.Bt = g.Bt; p.T = g.T; p.cin = g.cin; p.N = g.N; p.ntap = g.ntap; p.dil = g.dil;
  p.kb_per_tap = (g.cin + kBlockK - 1) / kBlockK;
  p.tiles_per_batch = (g.T + kTileM - 1) / kTileM;
  p.bn = pick_bn(g.N, g.Bt * p.tiles_per_batch);
  const int stage_bytes = kABytes + p.bn * kBlockK * 2;
  p.tiles_m = g.Bt * p.tiles_per_batch;
  p.tiles_n = (g.N + p.bn - 1) / p.bn;
  auto magic = [](unsigned d, unsigned& mul, unsigned& shift) {  // d >= 1
    unsigned l = 0;
    while ((1ull << l) < d) ++l;
    mul = (unsigned)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
    shift = l;
  };
  magic((unsigned)p.tiles_n, p.div_n_mul, p.div_n_shift);
  magic((unsigned)p.tiles_per_batch, p.div_b_mul, p.div_b_shift);
  const long long tiles = (long long)p.tiles_m * p.tiles_n;
  int cols = 32;
  while (cols < p.bn) cols <<= 1;
  p.acc_cols = cols;
  // Persistent schedule for grids of many tiles (the codec's thin-channel stages launch up to 25 000): per-CTA set-up / tear-down
  // and the exposed epilogue of a one-tile CTA (a 128 x 96 tile lived ~14 us for ~2 us of MMA) are paid once per SM instead of
  // once per tile.
  // A persistent grid is one CTA per SM with up to kMaxEpiSets sets of epilogue warps.
  const long long resident = 148;
  const bool persistent = tiles >= kPersistMinTiles * resident;
  p.n_acc = persistent ? 2 : 1;
  p.tmem_cols = cols * p.n_acc;
  // The epilogue (TMEM -> registers -> bias / activation / SnakeBeta / residual -> global) is the latency-bound pipe of the thin
  // stages (ncu: 3 active warps per scheduler, 0.25 eligible): a persistent CTA gets up to three sets of epilogue warps, each
  // taking every third 32-column chunk of a tile.
  p.epi_sets = persistent ? std::max(1, std::min(kMaxEpiSets, p.bn / 32)) : 1;
  // Bytes in flight per SM bound a latency-limited K loop: big one-tile-per-CTA grids run 2 CTAs/SM with ~100 KB rings each, small
  // grids and persistent ones (one CTA per SM at most) take the whole shared memory for one deep ring.
  p.tio = (g.out16 || g.outr16) && !g.swiglu && !g.res && !g.out32 && !g.pcm && g.N % 32 == 0 && g.ld16 % 8 == 0 && (!g.outr16 || g.ld32 % 8 == 0) &&
          (!g.res16 || g.ld_res % 8 == 0);
  const int tio_bytes = p.tio ? 256 + 4 * p.epi_sets * epiio::kPatchBytes : 0;
  const int ring_budget = ((!persistent && tiles > 148) ? 100 * 1024 : 200 * 1024) - tio_bytes;
  p.stages = std::max(2, std::min(12, ring_budget / stage_bytes));
  if (!persistent) p.stages = std::min(p.stages, std::max(2, g.ntap * p.kb_per_tap));
  int ring_bytes = p.stages * stage_bytes;
  p.bias = g.bias; p.res = g.res; p.ld_res = g.ld_res; p.scale = g.scale; p.act = g.act; p.swiglu = g.swiglu;
  p.out32 = g.out32; p.ld32 = g.ld32; p.out16 = g.out16; p.ld16 = g.ld16;
  p.snake_ea = g.snake_ea; p.snake_ieb = g.snake_ieb; p.snake_ch = g.snake_ch > 0 ? g.snake_ch : 1;
  p.pcm = g.pcm;
  p.row_scale = g.row_scale;
  p.k_rotate = g.k_rotate;
  p.res16 = g.res16; p.outr16 = g.outr16;
  // residual ring: persistent classic schedule, fp16 residual stream, no SwiGLU column pairing
  p.res_stages = 0; p.res_bytes = kTileM * p.bn * 2;
  if (!p.tio && g.res16 && persistent && !g.swiglu && p.bn % 8 == 0 && g.N % p.bn == 0) {
    int rs = std::max(1, std::min(4, (ring_budget / 2) / p.res_bytes));
    int st = (ring_budget - rs * p.res_bytes) / stage_bytes;
    if (st >= 2) { p.res_stages = rs; p.stages = std::min(p.stages, st); ring_bytes = p.stages * stage_bytes; }
  }
  Q3_CHECK(!(g.res && g.res16) && !(g.res16 && g.ld_res % 8) && !(g.outr16 && g.ld32 % 8), Q3TTS_ERR_INVALID_ARG, "tc_gemm: bad fp16 residual arguments");

  const uint64_t adims[3] = {(uint64_t)g.cin, (uint64_t)g.T, (uint64_t)g.Bt};
  const uint64_t astr[2] = {(uint64_t)g.cin * 2, (uint64_t)g.T * g.cin * 2};
  const uint32_t abox[3] = {(uint32_t)kBlockK, (uint32_t)kTileM, 1};
  const CUtensorMap ma = tc_make_map(g.a, 3, adims, astr, abox);
  p.w_reps = std::max(1, g.w_reps);
  const uint64_t bdims[3] = {(uint64_t)g.cin, (uint64_t)g.ntap * g.N, (uint64_t)p.w_reps};
  const uint64_t bstr[2] = {(uint64_t)g.cin * 2, p.w_reps > 1 ? (uint64_t)g.w_rep_stride * 2 : (uint64_t)g.ntap * g.N * g.cin * 2};
  const uint32_t bbox[3] = {(uint32_t)kBlockK, (uint32_t)p.bn, 1};
  const CUtensorMap mb = tc_make_map(g.w, 3, bdims, bstr, bbox);

  CUtensorMap mr = mb;  // unused unless the residual ring is on
  if (p.res_stages) {
    const uint64_t rdims[3] = {(uint64_t)g.ld_res, (uint64_t)g.T, (uint64_t)g.Bt};
    const uint64_t rstr[2] = {(uint64_t)g.ld_res * 2, (uint64_t)g.T * g.ld_res * 2};
    const uint32_t rbox[3] = {(uint32_t)p.bn, (uint32_t)kTileM, 1};
    const uint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode(&mr, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<__half*>(g.res16), rdims, rstr, rbox, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    Q3_CHECK(r == CUDA_SUCCESS, Q3TTS_ERR_CUDA, "cuTensorMapEncodeTiled (residual tiles) failed with CUresult %d", (int)r);
  }
  const size_t smem = (size_t)ring_bytes + (size_t)p.res_stages * p.res_bytes + 1024 + 64 * 8 + (size_t)tio_bytes;
  Q3_CHECK(smem <= 212 * 1024, Q3TTS_ERR_CAPACITY, "tc_gemm: shared memory request %zu too large", smem);
  Q3_CHECK(2 * p.stages + 5 + 2 * p.res_stages <= 64, Q3TTS_ERR_CAPACITY, "tc_gemm: too many ring stages");
  dim3 grid((unsigned)(persistent ? std::min<long long>(tiles, resident) : tiles));
  launch_kernel_pdl(tc_gemm_kernel, grid, dim3(64 + 128 * p.epi_sets), smem, c.stream, pdl_enabled(), ma, mb, mr, p);
  c.tick();
}

// ---------------------------------------------------------------------------------------------- small fp16 producers
__global__ void f32_to_f16_kernel(const float* __restrict__ x, size_t n4, __half* __restrict__ y) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&a); pk.y = *reinterpret_cast<uint32_t*>(&b);
    reinterpret_cast<uint2*>(y)[i] = pk;
  }
}
void launch_f32_to_f16(const LaunchCtx& c, const float* x, size_t n, __half* y) {
  if (n == 0) return;
  Q3_CHECK(n % 4 == 0, Q3TTS_ERR_INVALID_ARG, "f32_to_f16: length must be a multiple of 4");
  const size_t n4 = n / 4;
  const int blocks = (int)std::min<size_t>((n4 + 255) / 256, 148 * 32);
  launch_kernel_pdl(f32_to_f16_kernel, dim3(blocks), dim3(256), 0, c.stream, pdl_enabled(), x, n4, y);
  c.tick();
}

__global__ void __launch_bounds__(256) rmsnorm_f16_kernel(const float* __restrict__ x, int ldx, int dim, const float* __restrict__ w, float eps,
                                                          __half* __restrict__ y, int ldy) {
  __shared__ float red[8];
  pdl_launch_dependents();
  pdl_wait();
  const float* xr = x + (size_t)blockIdx.x * ldx;
  float ss = 0.f;
  for (int i = threadIdx.x; i < dim; i += 256) { const float v = xr[i]; ss += v * v; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) tot += red[i];
  const float inv = rsqrtf(tot / (float)dim + eps);
  __half* yr = y + (size_t)blockIdx.x * ldy;
  for (int i = threadIdx.x; i < dim; i += 256) yr[i] = __float2half_rn(w ? xr[i] * inv * w[i] : xr[i] * inv);
}
void launch_rmsnorm_f16(const LaunchCtx& c, const float* x, int ldx, int m, int dim, const float* w, float eps, __half* y, int ldy) {
  if (m <= 0) return;
  launch_kernel_pdl(rmsnorm_f16_kernel, dim3(m), dim3(256), 0, c.stream, pdl_enabled(), x, ldx, dim, w, eps, y, ldy);
  c.tick();
}

__global__ void scale_to_f16_kernel(const float* __restrict__ x, size_t n4, float scale, __half* __restrict__ y) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    __half2 a = __floats2half2_rn(v.x * scale, v.y * scale), b = __floats2half2_rn(v.z * scale, v.w * scale);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&a); pk.y = *reinterpret_cast<uint32_t*>(&b);
    reinterpret_cast<uint2*>(y)[i] = pk;
  }
}
void launch_scale_to_f16(const LaunchCtx& c, const float* x, size_t n, float scale, __half* y) {
  if (n == 0) return;
  Q3_CHECK(n % 4 == 0, Q3TTS_ERR_INVALID_ARG, "scale_to_f16: length must be a multiple of 4");
  const size_t n4 = n / 4;
  const int blocks = (int)std::min<size_t>((n4 + 255) / 256, 148 * 32);
  launch_kernel_pdl(scale_to_f16_kernel, dim3(blocks), dim3(256), 0, c.stream, pdl_enabled(), x, n4, scale, y);
  c.tick();
}

// one 8-lane group per row (tc_row_sumsq_f16 order: bit-identical to the factors the skinny kernel derives for itself)
__global__ void __launch_bounds__(128) row_scale_kernel(const __half* __restrict__ a, int m, int dim, float rms_a, float eps, float mult,
                                                        float* __restrict__ rs) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x * 16 + (threadIdx.x >> 3), j = threadIdx.x & 7;
  float ss = row < m ? tc_row_sumsq_f16(a + (size_t)row * dim, dim, j) : 0.f;
  ss = tc_group8_sum(ss);
  if (j == 0 && row < m) rs[row] = mult * rsqrtf(ss * rms_a + eps);
}
void launch_row_scale(const LaunchCtx& c, const __half* a, int m, int dim, float in_scale, float eps, float* rs) {
  if (m <= 0) return;
  Q3_CHECK(dim % 8 == 0, Q3TTS_ERR_INVALID_ARG, "row_scale: row length must be a multiple of 8");
  launch_kernel_pdl(row_scale_kernel, dim3((m + 15) / 16), dim3(128), 0, c.stream, pdl_enabled(), a, m, dim, 1.0f / (in_scale * in_scale * (float)dim),
                    eps, 1.0f / in_scale, rs);
  c.tick();
}

}  // namespace q3
