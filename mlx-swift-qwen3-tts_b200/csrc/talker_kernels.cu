// Hand-written sm_100a kernels for the Qwen3-TTS talker / code-predictor decode path.
//
// Everything here is HBM/L2-bandwidth or latency bound (batch-1..8 GEMV, norms, RoPE, window attention, sampling),
// so the design rules are: 128-bit coalesced loads of the packed weights, activations staged once per CTA in shared
// memory in a lane-major layout (bank-conflict free float4 reads), warp-shuffle reductions, no integer->float
// conversion instructions on the dequant path (magic-number bit tricks), and fusion of the RMSNorm prologue and the
// bias / residual / SiLU / SwiGLU epilogues into the GEMV so a decoder layer is 6 launches.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "kernels.h"
#include "device_utils.cuh"
#include "sampler.cuh"

namespace q3 {

// ------------------------------------------------------------------------------------------------ dequantize
// deq32 = fp32(scale) * q (rounded) + fp32(bias) (rounded) — __fmul_rn/__fadd_rn forbid FMA contraction so the
// result is bit-identical to the two-rounding contract of the oracle.
__global__ void dequantize_kernel(const uint32_t* __restrict__ qw, const void* __restrict__ scales,
                                  const void* __restrict__ biases, int sdt, int out, int in, int group, int bits,
                                  int out_dt, void* __restrict__ dst) {
  const int per = 32 / bits;
  const size_t words = (size_t)out * (in / per);
  const uint32_t mask = (1u << bits) - 1u;
  for (size_t wi = (size_t)blockIdx.x * blockDim.x + threadIdx.x; wi < words; wi += (size_t)gridDim.x * blockDim.x) {
    const size_t row = wi / (in / per);
    const int col0 = (int)(wi % (in / per)) * per;
    const uint32_t w = qw[wi];
    const size_t gi = row * (in / group) + col0 / group;  // `per` divides group: one scale per word
    const float s = load_as_f32(scales, gi, sdt), b = load_as_f32(biases, gi, sdt);
    for (int j = 0; j < per; ++j) {
      const float q = (float)((w >> (j * bits)) & mask);
      const float v = __fadd_rn(__fmul_rn(s, q), b);
      const size_t o = row * in + col0 + j;
      if (out_dt == Q3TTS_F32) reinterpret_cast<float*>(dst)[o] = v;
      else if (out_dt == Q3TTS_F16) reinterpret_cast<__half*>(dst)[o] = __float2half_rn(v);
      else reinterpret_cast<__nv_bfloat16*>(dst)[o] = __float2bfloat16_rn(v);
    }
  }
}

void launch_dequantize(const LaunchCtx& c, const uint32_t* qw, const void* scales, const void* biases, int sdt, int out,
                       int in, int group, int bits, int out_dt, void* dst) {
  const size_t words = (size_t)out * in * bits / 32;
  int blocks = (int)std::min<size_t>((words + 255) / 256, 148 * 16);
  if (blocks < 1) blocks = 1;
  dequantize_kernel<<<blocks, 256, 0, c.stream>>>(qw, scales, biases, sdt, out, in, group, bits, out_dt, dst);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ b-bit rows -> 4/8-bit container
// MLX stores a row of b-bit codes as one little-endian, LSB-first bit stream: code j at bits [j*b, (j+1)*b) of the row.  One thread
// builds one container word (8 codes of 4 bits or 4 codes of 8 bits); their source bits span at most 24 bits starting anywhere in a
// word, so two consecutive source words always hold them.  The second word is read only while it is inside the row, so the last word
// of the last row never reads past the allocation.
__global__ void widen_bits_kernel(const uint32_t* __restrict__ src, size_t rows, int in, int bits, int cbits, uint32_t* __restrict__ dst) {
  const int per = 32 / cbits;
  const int src_words = in / 32 * bits, dst_words = in / per;
  const uint32_t mask = (1u << bits) - 1u;
  const size_t total = rows * (size_t)dst_words;
  for (size_t wi = (size_t)blockIdx.x * blockDim.x + threadIdx.x; wi < total; wi += (size_t)gridDim.x * blockDim.x) {
    const size_t row = wi / dst_words;
    const int col0 = (int)(wi - row * dst_words) * per;
    const uint32_t* s = src + row * src_words;
    const int bit0 = col0 * bits, w0 = bit0 >> 5;
    uint64_t v = s[w0];
    if (w0 + 1 < src_words) v |= (uint64_t)s[w0 + 1] << 32;
    v >>= bit0 & 31;
    uint32_t out = 0;
    for (int j = 0; j < per; ++j) out |= (uint32_t)((v >> (j * bits)) & mask) << (j * cbits);
    dst[wi] = out;
  }
}

void launch_widen_bits(const LaunchCtx& c, const uint32_t* src, int rows, int in, int bits, uint32_t* dst) {
  const int cbits = container_bits(bits);
  Q3_CHECK((bits == 2 || bits == 3 || bits == 5 || bits == 6) && in > 0 && in % 32 == 0 && rows > 0, Q3TTS_ERR_INVALID_ARG,
           "widen_bits: bits %d / in %d unsupported (bits 2, 3, 5 or 6, in a multiple of 32)", bits, in);
  const size_t words = (size_t)rows * in * cbits / 32;
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((words + 255) / 256, 148 * 16));
  widen_bits_kernel<<<blocks, 256, 0, c.stream>>>(src, (size_t)rows, in, bits, cbits, dst);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ mxfp4 -> exact 8-bit affine container
// One thread builds one 8-bit container word: 4 E2M1 codes, the low or high half of one source word.  Rows are whole groups of 32
// (in % 32 == 0), so the flat indices line up across rows: container word wi takes source word wi / 2 and lies in group wi / 8, and the
// first thread of each group writes its scale and bias.  The loop never indexes past rows * in / 4 words.  Scale and bias are built
// from bit patterns: 2^(e - 128) is a bf16 subnormal for e < 2 (0x20 << e) and normal otherwise (exponent field e - 1);
// -12 * 2^(e - 128) = -1.5 * 2^(e - 125) has exponent field e + 2 and mantissa 0x40.
__global__ void mxfp4_to_affine_kernel(const uint32_t* __restrict__ packed, const uint8_t* __restrict__ scale_bytes, size_t words,
                                       uint32_t* __restrict__ codes8, uint16_t* __restrict__ scales, uint16_t* __restrict__ biases) {
  // q = 2 * lut[c] + 12 by code c, one byte each: codes 0..7 {12,13,14,15,16,18,20,24}, codes 8..15 {12,11,10,9,8,6,4,0}
  constexpr uint64_t kLo = 0x181412100F0E0D0Cull, kHi = 0x00040608090A0B0Cull;
  for (size_t wi = (size_t)blockIdx.x * blockDim.x + threadIdx.x; wi < words; wi += (size_t)gridDim.x * blockDim.x) {
    const uint32_t src = packed[wi >> 1] >> ((wi & 1) * 16);
    uint32_t out = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t code = (src >> (4 * j)) & 0xFu;
      out |= (uint32_t)(((code < 8 ? kLo : kHi) >> (8 * (code & 7))) & 0xFFu) << (8 * j);
    }
    codes8[wi] = out;
    if ((wi & 7) == 0) {
      const uint32_t e = scale_bytes[wi >> 3];
      scales[wi >> 3] = (uint16_t)(e < 2 ? 0x20u << e : (e - 1) << 7);
      biases[wi >> 3] = (uint16_t)(0x8000u | ((e + 2) << 7) | 0x40u);
    }
  }
}

void launch_mxfp4_to_affine(const LaunchCtx& c, const uint32_t* packed, const uint8_t* scale_bytes, int rows, int in, uint32_t* codes8_out,
                            uint16_t* scales_out, uint16_t* biases_out) {
  Q3_CHECK(rows > 0 && in > 0 && in % 32 == 0, Q3TTS_ERR_INVALID_ARG, "mxfp4_to_affine: %d x %d unsupported (in a multiple of 32)", rows, in);
  const size_t words = (size_t)rows * in / 4;
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((words + 255) / 256, 148 * 16));
  mxfp4_to_affine_kernel<<<blocks, 256, 0, c.stream>>>(packed, scale_bytes, words, codes8_out, scales_out, biases_out);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ runtime quantisation
// MLX `quantize(w, group_size: 64, bits)` (affine), one thread per group of 64 weights, restated operation for operation from
// oracle/mlx_quant.py:quantize (every fp32 step rounded on its own: no FMA contraction, IEEE division, round-half-even):
//     s = max((max - min) / (2^bits - 1), 1e-7), sign by the larger-magnitude edge; q0 = rint(edge / s); s = edge / q0 if q0 != 0;
//     b = q0 == 0 ? 0 : edge; s, b rounded to the weight dtype; q = clip(rint((w - b) / s), 0, 2^bits - 1)
// The codes go into an 8-BIT container whatever `bits` is (4 or 6: Qwen3TTSPipeline.applyMixedQuantization, :961-980), so every 8-bit
// kernel of the engine runs them; `fake` (optional) receives dequantised values in the weight dtype (quantised embeddings).
__global__ void mlx_quantize_kernel(const void* __restrict__ w, int wdt, size_t groups, int in, int bits, uint32_t* __restrict__ qw8,
                                    void* __restrict__ scales, void* __restrict__ biases, void* __restrict__ fake) {
  const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= groups) return;
  const int gpr = in / 64;
  const size_t row = g / gpr;
  const size_t e0 = row * (size_t)in + (size_t)(g - row * gpr) * 64;
  float v[64];
  float mx = -INFINITY, mn = INFINITY;
#pragma unroll 8
  for (int j = 0; j < 64; ++j) {
    v[j] = load_as_f32(w, e0 + j, wdt);
    mx = fmaxf(mx, v[j]);
    mn = fminf(mn, v[j]);
  }
  const float n_bins = (float)((1 << bits) - 1);
  const bool side = fabsf(mn) > fabsf(mx);
  float s = fmaxf(__fdiv_rn(__fsub_rn(mx, mn), n_bins), 1e-7f);
  s = side ? s : -s;
  const float edge = side ? mn : mx;
  const float q0 = rintf(__fdiv_rn(edge, s));
  if (q0 != 0.f) s = __fdiv_rn(edge, q0);
  float b = q0 == 0.f ? 0.f : edge;
  // round to the weight dtype (MLX returns scales / biases in the dtype of w)
  if (wdt == Q3TTS_BF16) { s = __bfloat162float(__float2bfloat16_rn(s)); b = __bfloat162float(__float2bfloat16_rn(b)); }
  else if (wdt == Q3TTS_F16) { s = __half2float(__float2half_rn(s)); b = __half2float(__float2half_rn(b)); }
  const float s_safe = s == 0.f ? 1e-7f : s;
  if (wdt == Q3TTS_F32) { reinterpret_cast<float*>(scales)[g] = s; reinterpret_cast<float*>(biases)[g] = b; }
  else if (wdt == Q3TTS_F16) { reinterpret_cast<__half*>(scales)[g] = __float2half_rn(s); reinterpret_cast<__half*>(biases)[g] = __float2half_rn(b); }
  else { reinterpret_cast<__nv_bfloat16*>(scales)[g] = __float2bfloat16_rn(s); reinterpret_cast<__nv_bfloat16*>(biases)[g] = __float2bfloat16_rn(b); }
#pragma unroll 4
  for (int j = 0; j < 64; j += 4) {
    uint32_t word = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float q = fminf(fmaxf(rintf(__fdiv_rn(__fsub_rn(v[j + u], b), s_safe)), 0.f), n_bins);
      word |= (uint32_t)q << (8 * u);
      if (fake) {
        const float d = __fadd_rn(__fmul_rn(s, q), b);  // the q3tts_dequantize contract
        const size_t o = e0 + j + u;
        if (wdt == Q3TTS_F32) reinterpret_cast<float*>(fake)[o] = d;
        else if (wdt == Q3TTS_F16) reinterpret_cast<__half*>(fake)[o] = __float2half_rn(d);
        else reinterpret_cast<__nv_bfloat16*>(fake)[o] = __float2bfloat16_rn(d);
      }
    }
    if (qw8) qw8[(e0 + j) >> 2] = word;
  }
}

void launch_mlx_quantize(const LaunchCtx& c, const void* w, int wdt, int out, int in, int bits, uint32_t* qw8, void* scales, void* biases,
                         void* fake) {
  Q3_CHECK(in % 64 == 0 && (bits == 4 || bits == 6 || bits == 8), Q3TTS_ERR_INVALID_ARG, "mlx_quantize: in %d / bits %d unsupported", in, bits);
  const size_t groups = (size_t)out * (in / 64);
  mlx_quantize_kernel<<<(unsigned)((groups + 127) / 128), 128, 0, c.stream>>>(w, wdt, groups, in, bits, qw8, scales, biases, fake);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ GEMV / small-M linear
struct LinearKArgs {
  const void* w;        // packed or dense weights, row-major
  const void* scales;   // quantised only
  const void* biases;
  const float* bias;    // [out] or null
  const float* x;
  float* y;
  const float* norm_w;  // fused RMSNorm weight or null
  float eps;
  int out, in, group, sdt, m, ldx, ldy, epi;
};

// Shared-memory layout per CTA:  xs[MT][nchunk*KC/4] float4 in lane-major order,  xsum[MT][nchunk*32] (quantised formats).
// Lane-major: element e of a K-chunk (KC = 32*VPL values) lives at float4 index ((e%VPL)/4)*32 + e/VPL, so the 32
// lanes of a warp read 32 consecutive float4 — conflict free — while each lane's weights stay one contiguous
// 16-byte global load.
//
// Latency structure (batch-1 decode is latency bound, ~2 MB of weights per launch): the weight / scale loads of the warp's
// first row do not depend on the activations, so they are issued FIRST and fly while the CTA stages x; staging is a single
// pass (RMSNorm statistics, per-lane activation sums for the group-bias term and the smem fill together) behind ONE
// __syncthreads; the RMS scale is applied to the finished dot product (it is a per-row scalar).
template <int FMT, int MT>
__global__ void __launch_bounds__(256, (MT <= 2 ? 3 : 1)) linear_kernel(const LinearKArgs a) {
  constexpr int VPL = FmtTraits<FMT>::VPL;
  constexpr int KC = 32 * VPL;
  constexpr bool QUANT = (FMT == W_Q4 || FMT == W_Q8);
  constexpr int LPG = VPL / 4;  // staging threads (one float4 each) per weight lane
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nchunk = (a.in + KC - 1) / KC;   // the last chunk may be partial (in must be a multiple of VPL)
  const int xstride = nchunk * (KC / 4);     // float4 per activation row in shared memory (chunk-padded)
  float4* xs = reinterpret_cast<float4*>(smem_raw);
  float* xsum = reinterpret_cast<float*>(smem_raw + (size_t)MT * xstride * sizeof(float4));
  __shared__ float red[MT][8];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int m0 = blockIdx.y * MT;
  const int in4 = a.in >> 2;
  const int out_eff = (a.epi == EPI_SWIGLU) ? (a.out >> 1) : a.out;
  const int nsub = (a.epi == EPI_SWIGLU) ? 2 : 1;
  const size_t row_bytes = QUANT ? (size_t)a.in * (FMT == W_Q4 ? 4 : 8) / 8 : (size_t)a.in * (FMT == W_F32 ? 4 : 2);
  const int ngroups = QUANT ? a.in / a.group : 0;
  const int r_first = blockIdx.x * 8 + warp;

  // ---- (0) L2 prefetch of the warp's first row(s): weights do not depend on x, so their HBM->L2 trip overlaps the staging ----
  if (r_first < out_eff) {
    for (int s = 0; s < nsub; ++s) {
      const int row = r_first + s * out_eff;
      const unsigned char* wr = reinterpret_cast<const unsigned char*>(a.w) + (size_t)row * row_bytes;
      for (size_t off = (size_t)lane * 128; off < row_bytes; off += 32 * 128) prefetch_l2(wr + off);
      if constexpr (QUANT) {
        if (lane == 0) prefetch_l2(reinterpret_cast<const unsigned char*>(a.scales) + (size_t)row * ngroups * (a.sdt == Q3TTS_F32 ? 4 : 2));
        if (lane == 1) prefetch_l2(reinterpret_cast<const unsigned char*>(a.biases) + (size_t)row * ngroups * (a.sdt == Q3TTS_F32 ? 4 : 2));
      }
    }
  }

  // ---- (1) stage activations: one pass, one barrier ----
  const int iters = (in4 + 255) / 256;
#pragma unroll
  for (int mi = 0; mi < MT; ++mi) {
    const bool valid = (m0 + mi) < a.m;
    const float4* xr = reinterpret_cast<const float4*>(a.x + (size_t)(valid ? m0 + mi : 0) * a.ldx);
    float ss = 0.f;
    for (int it = 0; it < iters; ++it) {
      const int f = tid + it * 256;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid && f < in4) v = xr[f];
      ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
      if (a.norm_w != nullptr && f < in4) {
        const float4 nw = reinterpret_cast<const float4*>(a.norm_w)[f];
        v.x *= nw.x; v.y *= nw.y; v.z *= nw.z; v.w *= nw.w;
      }
      const int e = f << 2;
      const int ch = e / KC, ec = e - ch * KC;
      const int l = ec / VPL, j = (ec - l * VPL) >> 2;
      if (f < in4) xs[(size_t)mi * xstride + ch * (KC / 4) + j * 32 + l] = v;
      if constexpr (QUANT) {  // sum over the LPG consecutive float4 that belong to one weight lane (all lanes participate)
        float s4 = (v.x + v.y) + (v.z + v.w);
#pragma unroll
        for (int o = 1; o < LPG; o <<= 1) s4 += __shfl_xor_sync(0xffffffffu, s4, o);
        if ((tid & (LPG - 1)) == 0 && f < in4) xsum[mi * (nchunk * 32) + ch * 32 + l] = s4;
      }
    }
    if (a.norm_w != nullptr) {
      ss = warp_sum(ss);
      if (lane == 0) red[mi][warp] = ss;
    }
  }
  __syncthreads();
  float inv_rms[MT];
#pragma unroll
  for (int mi = 0; mi < MT; ++mi) {
    inv_rms[mi] = 1.0f;
    if (a.norm_w != nullptr) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += red[mi][w];
      inv_rms[mi] = rsqrtf(s / (float)a.in + a.eps);
    }
  }

  // ---- (2) stream weight rows: one warp per output row (pair of rows for SwiGLU) ----
  for (int r = r_first; r < out_eff; r += gridDim.x * 8) {
    float yold[MT];
#pragma unroll
    for (int mi = 0; mi < MT; ++mi) yold[mi] = (a.epi == EPI_ADD && lane == 0 && m0 + mi < a.m) ? a.y[(size_t)(m0 + mi) * a.ldy + r] : 0.f;
    float res[2][MT];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
#pragma unroll
      for (int mi = 0; mi < MT; ++mi) res[s][mi] = 0.f;
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      if (s >= nsub) break;
      const int row = r + s * out_eff;
      const uint4* wr = reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(a.w) + (size_t)row * row_bytes);
      float acc[MT];
#pragma unroll
      for (int mi = 0; mi < MT; ++mi) acc[mi] = 0.f;
      for (int c0 = 0; c0 < nchunk; c0 += 4) {
        uint4 wv[4];
        float scv[4], biv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if ((c0 + u) * KC + lane * VPL < a.in) {
            wv[u] = ldg_stream(wr + (size_t)(c0 + u) * 32 + lane);
            if constexpr (QUANT) {
              const size_t gi = (size_t)row * ngroups + ((c0 + u) * KC + lane * VPL) / a.group;
              scv[u] = load_as_f32(a.scales, gi, a.sdt);
              biv[u] = load_as_f32(a.biases, gi, a.sdt);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if ((c0 + u) * KC + lane * VPL < a.in) {
            const int ch = c0 + u;
            float wf[VPL];
            lane_expand<FMT>(wv[u], wf);
#pragma unroll
            for (int mi = 0; mi < MT; ++mi) {
              const float d = lane_dot<FMT>(wf, xs + (size_t)mi * xstride + ch * (KC / 4) + lane);
              if constexpr (QUANT) acc[mi] += scv[u] * d + biv[u] * xsum[mi * (nchunk * 32) + ch * 32 + lane];
              else acc[mi] += d;
            }
          }
        }
      }
#pragma unroll
      for (int mi = 0; mi < MT; ++mi) res[s][mi] = warp_sum(acc[mi]) * inv_rms[mi];
    }
    if (lane == 0) {
#pragma unroll
      for (int mi = 0; mi < MT; ++mi) {
        if (m0 + mi >= a.m) break;
        float v = res[0][mi];
        float* yp = a.y + (size_t)(m0 + mi) * a.ldy + r;
        if (a.epi == EPI_SWIGLU) {
          float g = v, u = res[1][mi];
          if (a.bias) { g += a.bias[r]; u += a.bias[r + out_eff]; }
          *yp = silu_f(g) * u;
        } else {
          if (a.bias) v += a.bias[r];
          if (a.epi == EPI_SILU) v = silu_f(v);
          if (a.epi == EPI_ADD) v += yold[mi];
          *yp = v;
        }
      }
    }
  }
}

template <int FMT, int MT>
static void launch_linear_t(const LaunchCtx& c, const LinearKArgs& a, int num_sms) {
  constexpr int VPL = FmtTraits<FMT>::VPL;
  constexpr bool QUANT = (FMT == W_Q4 || FMT == W_Q8);
  constexpr int KC = 32 * VPL;
  const int nchunk = (a.in + KC - 1) / KC;
  size_t smem = (size_t)MT * nchunk * KC * sizeof(float) + (QUANT ? (size_t)MT * nchunk * 32 * sizeof(float) : 0);
  const int out_eff = (a.epi == EPI_SWIGLU) ? a.out / 2 : a.out;
  int bx = (out_eff + 7) / 8;
  const int cap = num_sms * 8;
  if (bx > cap) bx = cap;
  dim3 grid(bx, (a.m + MT - 1) / MT);
  linear_kernel<FMT, MT><<<grid, 256, smem, c.stream>>>(a);
  c.tick();
}

template <int FMT>
static void launch_linear_f(const LaunchCtx& c, LinearKArgs a) {
  // M-tile: largest of {8,4,2,1} not above m whose activation stage fits ~96 KB of shared memory
  int mt = 8;
  while (mt > 1 && (mt > a.m * 2 - 1 || (size_t)mt * a.in * 5 > 96 * 1024)) mt >>= 1;
  if (a.m == 1) mt = 1;
  switch (mt) {
    case 8: launch_linear_t<FMT, 8>(c, a, 148); break;
    case 4: launch_linear_t<FMT, 4>(c, a, 148); break;
    case 2: launch_linear_t<FMT, 2>(c, a, 148); break;
    default: launch_linear_t<FMT, 1>(c, a, 148); break;
  }
}

void launch_linear(const LaunchCtx& c, const Linear& L, const float* x, int ldx, int m, float* y, int ldy,
                   const float* norm_w, float eps, int epilogue) {
  if (m <= 0) return;
  LinearKArgs a;
  a.w = L.bits ? (const void*)L.qw : L.w;
  a.scales = L.scales; a.biases = L.biases; a.bias = L.bias;
  a.x = x; a.y = y; a.norm_w = norm_w; a.eps = eps;
  a.out = L.out; a.in = L.in; a.group = L.group; a.sdt = L.sdt; a.m = m; a.ldx = ldx; a.ldy = ldy; a.epi = epilogue;
  Q3_CHECK((ldx % 4) == 0, Q3TTS_ERR_INVALID_ARG, "linear: activation stride %d not 16-byte aligned", ldx);
  if (L.bits == 4) {
    Q3_CHECK(L.in % 32 == 0 && L.group % 32 == 0, Q3TTS_ERR_BAD_CONFIG, "4-bit linear needs in %% 32 == 0 and group %% 32 == 0 (in=%d, group=%d)", L.in, L.group);
    launch_linear_f<W_Q4>(c, a);
  } else if (L.bits == 8) {
    Q3_CHECK(L.in % 16 == 0 && L.group % 16 == 0, Q3TTS_ERR_BAD_CONFIG, "8-bit linear needs in %% 16 == 0 (in=%d)", L.in);
    launch_linear_f<W_Q8>(c, a);
  } else if (L.bits == 0) {
    if (L.sdt == Q3TTS_BF16) { Q3_CHECK(L.in % 8 == 0, Q3TTS_ERR_BAD_CONFIG, "bf16 linear needs in %% 8 == 0 (in=%d)", L.in); launch_linear_f<W_BF16>(c, a); }
    else if (L.sdt == Q3TTS_F16) { Q3_CHECK(L.in % 8 == 0, Q3TTS_ERR_BAD_CONFIG, "f16 linear needs in %% 8 == 0 (in=%d)", L.in); launch_linear_f<W_F16>(c, a); }
    else { Q3_CHECK(L.in % 4 == 0, Q3TTS_ERR_BAD_CONFIG, "f32 linear needs in %% 4 == 0 (in=%d)", L.in); launch_linear_f<W_F32>(c, a); }
  } else {
    fail(Q3TTS_ERR_BAD_CONFIG, "unsupported quantisation bits %d (4 and 8 are in scope; 6-bit runtime quantisation is not)", L.bits);
  }
}

// ------------------------------------------------------------------------------------------------ RMSNorm
__global__ void __launch_bounds__(256) rmsnorm_kernel(const float* __restrict__ x, int ldx, int dim, const float* __restrict__ w,
                                                      float eps, float* __restrict__ y, int ldy) {
  __shared__ float red[8];
  const float* xr = x + (size_t)blockIdx.x * ldx;
  float ss = 0.f;
  for (int i = threadIdx.x; i < dim; i += 256) { const float v = xr[i]; ss += v * v; }
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) tot += red[i];
  const float inv = rsqrtf(tot / (float)dim + eps);
  float* yr = y + (size_t)blockIdx.x * ldy;
  for (int i = threadIdx.x; i < dim; i += 256) yr[i] = xr[i] * inv * w[i];
}
void launch_rmsnorm(const LaunchCtx& c, const float* x, int ldx, int m, int dim, const float* w, float eps, float* y, int ldy) {
  if (m <= 0) return;
  rmsnorm_kernel<<<m, 256, 0, c.stream>>>(x, ldx, dim, w, eps, y, ldy);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ q/k norm + RoPE + KV append
// One warp per (row, head).  head < heads: q;  < heads+kv: k;  else v.  head_dim == 128: lane l owns dims l, l+32 and
// their rotate-half partners l+64, l+96.
// KV cache element access: fp32 rings, or fp16 rings on batched handles (half the bytes of the window walk; K and V are rounded
// once when they are appended, everything downstream stays fp32)
__device__ __forceinline__ float4 kv_ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 kv_ld4(const __half* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float kv_ld(const float* p) { return *p; }
__device__ __forceinline__ float kv_ld(const __half* p) { return __half2float(*p); }
__device__ __forceinline__ void kv_st(float* p, float v) { *p = v; }
__device__ __forceinline__ void kv_st(__half* p, float v) { *p = __float2half_rn(v); }
template <typename KvT>
__global__ void __launch_bounds__(128) qk_norm_rope_append_kernel(float* __restrict__ qkv, int ld, int m, int heads, int kv_heads,
                                                                  const float* __restrict__ q_norm, const float* __restrict__ k_norm,
                                                                  float eps, const float* __restrict__ inv_freq,
                                                                  const int* __restrict__ row_slot, const int* __restrict__ row_pos,
                                                                  KVLayout kv) {
  const int total_heads = heads + 2 * kv_heads;
  const int gw = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (gw >= m * total_heads) return;
  const int row = gw / total_heads, head = gw - row * total_heads;
  const int lane = threadIdx.x & 31;
  float* p = qkv + (size_t)row * ld + (size_t)head * 128;
  const int slot = row_slot[row], pos = row_pos[row];
  const int ring = pos % kv.capacity;
  if (head >= heads + kv_heads) {  // v: plain append
    KvT* dst = static_cast<KvT*>(kv.v) + (size_t)slot * kv.slot_stride + ((size_t)(head - heads - kv_heads) * kv.capacity + ring) * 128;
    const float4 v4 = reinterpret_cast<const float4*>(p)[lane];
    kv_st(dst + 4 * lane, v4.x); kv_st(dst + 4 * lane + 1, v4.y); kv_st(dst + 4 * lane + 2, v4.z); kv_st(dst + 4 * lane + 3, v4.w);
    return;
  }
  const float a0 = p[lane], a1 = p[lane + 32], b0 = p[lane + 64], b1 = p[lane + 96];
  const float ss = warp_sum(a0 * a0 + a1 * a1 + b0 * b0 + b1 * b1);
  const float inv = rsqrtf(ss * (1.0f / 128.0f) + eps);
  const float* nw = head < heads ? q_norm : k_norm;
  const float x0 = a0 * inv * nw[lane], x1 = a1 * inv * nw[lane + 32];
  const float y0 = b0 * inv * nw[lane + 64], y1 = b1 * inv * nw[lane + 96];
  const float fp = (float)pos;
  float s0, c0, s1, c1;
  sincosf(fp * inv_freq[lane], &s0, &c0);
  sincosf(fp * inv_freq[lane + 32], &s1, &c1);
  // q*cos + rotate_half(q)*sin with rotate_half = [-x2, x1]  (Model/Qwen3Layers.swift:187-195)
  const float o0 = x0 * c0 - y0 * s0, o1 = x1 * c1 - y1 * s1;
  const float o2 = y0 * c0 + x0 * s0, o3 = y1 * c1 + x1 * s1;
  if (head >= heads) {
    KvT* dst = static_cast<KvT*>(kv.k) + (size_t)slot * kv.slot_stride + ((size_t)(head - heads) * kv.capacity + ring) * 128;
    kv_st(dst + lane, o0); kv_st(dst + lane + 32, o1); kv_st(dst + lane + 64, o2); kv_st(dst + lane + 96, o3);
  } else {
    p[lane] = o0; p[lane + 32] = o1; p[lane + 64] = o2; p[lane + 96] = o3;
  }
}
void launch_qk_norm_rope_append(const LaunchCtx& c, float* qkv, int ld, int m, int heads, int kv_heads, int head_dim,
                                const float* q_norm, const float* k_norm, float eps, const float* inv_freq,
                                const int* row_slot, const int* row_pos, const KVLayout& kv) {
  Q3_CHECK(head_dim == 128, Q3TTS_ERR_BAD_CONFIG, "talker kernels are specialised for head_dim 128 (got %d)", head_dim);
  const int warps = m * (heads + 2 * kv_heads);
  if (warps <= 0) return;
  if (kv.f16)
    qk_norm_rope_append_kernel<__half><<<(warps + 3) / 4, 128, 0, c.stream>>>(qkv, ld, m, heads, kv_heads, q_norm, k_norm, eps, inv_freq, row_slot, row_pos, kv);
  else
    qk_norm_rope_append_kernel<float><<<(warps + 3) / 4, 128, 0, c.stream>>>(qkv, ld, m, heads, kv_heads, q_norm, k_norm, eps, inv_freq, row_slot, row_pos, kv);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ window attention (decode + prefill)
// grid (row, kv_head), 128 threads.  Keys = absolute positions [win_start[slot], row_pos] of the row's slot, read
// through the ring.  G = heads / kv_heads query heads share the K/V reads (GQA, head h uses kv head h / G).
__device__ __forceinline__ void store_act(float* p, float v) { *p = v; }
__device__ __forceinline__ void store_act(__half* p, float v) { *p = __float2half_rn(v); }

template <int G, typename OutT, typename KvT>
__global__ void __launch_bounds__(128) attention_kernel(const float* __restrict__ qkv, int ld, int heads, int kv_heads,
                                                        const int* __restrict__ row_slot, const int* __restrict__ row_pos,
                                                        const int* __restrict__ win_start, KVLayout kv, OutT* __restrict__ out,
                                                        int ldo, float scale) {
  extern __shared__ __align__(16) float sm[];
  float* q = sm;                 // [G][128]
  float* sc = sm + G * 128;      // [G][S]
  __shared__ float red_max[G], red_sum[G];
  const int row = blockIdx.x, kvh = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slot = row_slot[row], pos = row_pos[row];
  const int w0 = win_start ? win_start[slot] : 0;
  const int S = pos - w0 + 1;
  const int cap = kv.capacity;
  const int r0 = w0 % cap;  // ring index of the window's first key: ONE division; key j sits at r0 + j (- cap), never a modulo per key
  const KvT* kb = static_cast<const KvT*>(kv.k) + (size_t)slot * kv.slot_stride + (size_t)kvh * cap * 128;
  const KvT* vb = static_cast<const KvT*>(kv.v) + (size_t)slot * kv.slot_stride + (size_t)kvh * cap * 128;
#pragma unroll
  for (int g = 0; g < G; ++g) q[g * 128 + tid] = qkv[(size_t)row * ld + (size_t)(kvh * G + g) * 128 + tid];
  __syncthreads();
  for (int j = tid; j < S; j += 128) {
    const int rj = r0 + j;
    const KvT* kr = kb + (size_t)(rj >= cap ? rj - cap : rj) * 128;
    float acc[G];
#pragma unroll
    for (int g = 0; g < G; ++g) acc[g] = 0.f;
#pragma unroll 8
    for (int d = 0; d < 32; ++d) {
      const float4 kk = kv_ld4(kr + 4 * d);
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const float4 qq = reinterpret_cast<const float4*>(q + g * 128)[d];
        acc[g] += kk.x * qq.x + kk.y * qq.y + kk.z * qq.z + kk.w * qq.w;
      }
    }
#pragma unroll
    for (int g = 0; g < G; ++g) sc[g * S + j] = acc[g] * scale;
  }
  __syncthreads();
  for (int g = warp; g < G; g += 4) {  // softmax per query head, one warp each
    float mx = -INFINITY;
    for (int j = lane; j < S; j += 32) mx = fmaxf(mx, sc[g * S + j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < S; j += 32) { const float e = expf(sc[g * S + j] - mx); sc[g * S + j] = e; sum += e; }
    sum = warp_sum(sum);
    if (lane == 0) { red_max[g] = mx; red_sum[g] = sum; }
  }
  __syncthreads();
  float o[G];
#pragma unroll
  for (int g = 0; g < G; ++g) o[g] = 0.f;
  for (int j = 0; j < S; ++j) {
    const int rj = r0 + j;
    const float vv = kv_ld(vb + (size_t)(rj >= cap ? rj - cap : rj) * 128 + tid);
#pragma unroll
    for (int g = 0; g < G; ++g) o[g] = fmaf(sc[g * S + j], vv, o[g]);
  }
#pragma unroll
  for (int g = 0; g < G; ++g) store_act(out + (size_t)row * ldo + (size_t)(kvh * G + g) * 128 + tid, o[g] / red_sum[g]);
}
// Decode-step fusion of q/k norm + RoPE + KV append + window attention (one launch instead of two, no q/k round trip through
// HBM).  Valid only when every slot contributes ONE row to the launch (talker step, code-predictor passes >= 1): the keys of
// positions < pos were written by earlier launches, the current position's k/v are appended here (same CTA: visible after the
// barrier).
// Single pass, flash-decoding style: the 128 threads form 16 groups of 8 lanes; a group owns keys j = group, group + 16, ...
// and each lane 16 of the 128 dims (4 x float4, so the 8 lanes of a group read one 512-byte K row and one V row fully
// coalesced).  Per key: 8 independent 128-bit loads per lane (two keys in flight), a 3-step shuffle reduce of the partial dot
// products, an online-softmax update of the lane's 16 output dims.  Groups are merged at the end (2 shuffle steps inside a
// warp, shared memory across the 4 warps).  The previous version (thread-per-key score loop with 8 loads in flight, three
// block barriers, 4 V loads in flight) spent ~11 us per launch on dependent round trips even for 2-17 keys.
template <int G, typename OutT, typename KvT>
__global__ void __launch_bounds__(128, 4) rope_attention_kernel(const float* __restrict__ qkv, int ld, int heads, int kv_heads,
                                                             const float* __restrict__ q_norm, const float* __restrict__ k_norm, float eps,
                                                             const float* __restrict__ inv_freq, const int* __restrict__ row_slot,
                                                             const int* __restrict__ row_pos, const int* __restrict__ win_start, KVLayout kv,
                                                             OutT* __restrict__ out, int ldo, float scale) {
  __shared__ __align__(16) float q[G * 128];
  __shared__ __align__(16) float part_o[4][G][128];
  __shared__ float part_m[4][G], part_l[4][G];
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x, kvh = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slot = row_slot[row], pos = row_pos[row];
  const int w0 = win_start ? win_start[slot] : 0;
  const int S = pos - w0 + 1;
  const int cap = kv.capacity;
  const int r0 = w0 % cap;  // see attention_kernel: key j of the window sits at ring index r0 + j (- cap)
  const int ring = (r0 + S - 1 >= cap) ? r0 + S - 1 - cap : r0 + S - 1;  // == pos % cap (S <= cap)
  KvT* kb = static_cast<KvT*>(kv.k) + (size_t)slot * kv.slot_stride + (size_t)kvh * cap * 128;
  KvT* vb = static_cast<KvT*>(kv.v) + (size_t)slot * kv.slot_stride + (size_t)kvh * cap * 128;
  const float* rowp = qkv + (size_t)row * ld;
  // phase 0: per-head RMSNorm + rotate-half RoPE (Model/Qwen3Layers.swift:174-195); warp hh < G -> q head, hh == G -> k head
  for (int hh = warp; hh <= G; hh += 4) {
    const float* src = rowp + (size_t)(hh < G ? (kvh * G + hh) : (heads + kvh)) * 128;
    const float a0 = src[lane], a1 = src[lane + 32], b0 = src[lane + 64], b1 = src[lane + 96];
    const float ss = warp_sum(a0 * a0 + a1 * a1 + b0 * b0 + b1 * b1);
    const float inv = rsqrtf(ss * (1.0f / 128.0f) + eps);
    const float* nw = hh < G ? q_norm : k_norm;
    const float x0 = a0 * inv * nw[lane], x1 = a1 * inv * nw[lane + 32], y0 = b0 * inv * nw[lane + 64], y1 = b1 * inv * nw[lane + 96];
    float s0, c0, s1, c1;
    sincosf((float)pos * inv_freq[lane], &s0, &c0);
    sincosf((float)pos * inv_freq[lane + 32], &s1, &c1);
    const float o0 = x0 * c0 - y0 * s0, o1 = x1 * c1 - y1 * s1, o2 = y0 * c0 + x0 * s0, o3 = y1 * c1 + x1 * s1;
    if (hh < G) {
      float* dst = q + hh * 128;
      dst[lane] = o0; dst[lane + 32] = o1; dst[lane + 64] = o2; dst[lane + 96] = o3;
    } else {  // k is appended to the ring (:197-201)
      KvT* dst = kb + (size_t)ring * 128;
      kv_st(dst + lane, o0); kv_st(dst + lane + 32, o1); kv_st(dst + lane + 64, o2); kv_st(dst + lane + 96, o3);
    }
  }
  kv_st(vb + (size_t)ring * 128 + tid, rowp[(size_t)(heads + kv_heads + kvh) * 128 + tid]);
  __syncthreads();
  // phase 1: one pass over the window
  const int seg = lane & 7, grp = warp * 4 + (lane >> 3);
  float qf[G][16];
#pragma unroll
  for (int g = 0; g < G; ++g)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 t = *reinterpret_cast<const float4*>(q + g * 128 + i * 32 + seg * 4);
      qf[g][4 * i] = t.x * scale; qf[g][4 * i + 1] = t.y * scale; qf[g][4 * i + 2] = t.z * scale; qf[g][4 * i + 3] = t.w * scale;
    }
  float mx[G], l[G], o[G][16];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    mx[g] = -INFINITY; l[g] = 0.f;
#pragma unroll
    for (int d = 0; d < 16; ++d) o[g][d] = 0.f;
  }
  for (int jb = 0; jb < S; jb += 32) {  // keys jb + grp and jb + grp + 16 of this group: 16 independent 128-bit loads in flight
    const int j0 = jb + grp;              // (the trip count is the same for every lane: the shuffles below stay convergent)
    float4 kk[2][4], vv[2][4];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int j = j0 + 16 * u;
      const int rj = r0 + (j < S ? j : 0);
      const size_t base = (size_t)(rj >= cap ? rj - cap : rj) * 128 + seg * 4;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        kk[u][i] = kv_ld4(kb + base + i * 32);
        vv[u][i] = kv_ld4(vb + base + i * 32);
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const bool valid = j0 + 16 * u < S;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        float sdot = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          sdot += kk[u][i].x * qf[g][4 * i] + kk[u][i].y * qf[g][4 * i + 1] + kk[u][i].z * qf[g][4 * i + 2] + kk[u][i].w * qf[g][4 * i + 3];
        sdot += __shfl_xor_sync(0xffffffffu, sdot, 1);
        sdot += __shfl_xor_sync(0xffffffffu, sdot, 2);
        sdot += __shfl_xor_sync(0xffffffffu, sdot, 4);
        if (!valid) sdot = -INFINITY;
        const float mn = fmaxf(mx[g], sdot);
        const bool none = mn == -INFINITY;  // no key seen yet and this one is out of range
        const float corr = none ? 1.f : expf(mx[g] - mn), pr = none ? 0.f : expf(sdot - mn);
        mx[g] = mn;
        l[g] = l[g] * corr + pr;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          o[g][4 * i] = o[g][4 * i] * corr + pr * vv[u][i].x;
          o[g][4 * i + 1] = o[g][4 * i + 1] * corr + pr * vv[u][i].y;
          o[g][4 * i + 2] = o[g][4 * i + 2] * corr + pr * vv[u][i].z;
          o[g][4 * i + 3] = o[g][4 * i + 3] * corr + pr * vv[u][i].w;
        }
      }
    }
  }
  // merge the 4 groups of a warp, then the 4 warps
#pragma unroll
  for (int g = 0; g < G; ++g) {
    float m_all = fmaxf(mx[g], __shfl_xor_sync(0xffffffffu, mx[g], 8));
    m_all = fmaxf(m_all, __shfl_xor_sync(0xffffffffu, m_all, 16));
    const float f = (mx[g] == -INFINITY) ? 0.f : expf(mx[g] - m_all);  // a warp with no key at all keeps m_all = -inf
    float lw = l[g] * f;
    lw += __shfl_xor_sync(0xffffffffu, lw, 8);
    lw += __shfl_xor_sync(0xffffffffu, lw, 16);
#pragma unroll
    for (int d = 0; d < 16; ++d) {
      float t = o[g][d] * f;
      t += __shfl_xor_sync(0xffffffffu, t, 8);
      t += __shfl_xor_sync(0xffffffffu, t, 16);
      o[g][d] = t;
    }
    if (lane < 8) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(&part_o[warp][g][i * 32 + seg * 4]) = make_float4(o[g][4 * i], o[g][4 * i + 1], o[g][4 * i + 2], o[g][4 * i + 3]);
      if (lane == 0) { part_m[warp][g] = m_all; part_l[warp][g] = lw; }
    }
  }
  __syncthreads();
#pragma unroll
  for (int g = 0; g < G; ++g) {
    float m_all = fmaxf(fmaxf(part_m[0][g], part_m[1][g]), fmaxf(part_m[2][g], part_m[3][g]));
    float num = 0.f, den = 0.f;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const float f = (part_m[w][g] == -INFINITY) ? 0.f : expf(part_m[w][g] - m_all);
      num += part_o[w][g][tid] * f;
      den += part_l[w][g] * f;
    }
    store_act(out + (size_t)row * ldo + (size_t)(kvh * G + g) * 128 + tid, num / den);
  }
}
// Code-predictor pass 0 (Qwen3CodePredictor.swift:183-212 with L = 2): rows (2s, 2s+1) of slot s sit at positions 0 and 1 of a
// cache that is reset every frame, so norm + RoPE + append + causal attention of BOTH rows is one small CTA per (slot, kv head):
// position 0 attends to itself (output = v0), position 1 to keys {0, 1}.  Replaces qk_norm_rope_append + attention_kernel
// (two launches, ~28 us under ncu) on the decode path.
template <int G>
__global__ void __launch_bounds__(128) cp_pass0_attention_kernel(const float* __restrict__ qkv, int ld, int heads, int kv_heads,
                                                                 const float* __restrict__ q_norm, const float* __restrict__ k_norm, float eps,
                                                                 const float* __restrict__ inv_freq, KVLayout kv, __half* __restrict__ out,
                                                                 int ldo, float scale) {
  __shared__ __align__(16) float q1[G * 128];   // roped query heads of position 1
  __shared__ __align__(16) float kk[2][128];    // roped keys of positions 0 and 1
  __shared__ __align__(16) float vv[2][128];
  __shared__ float w0[G], w1[G];                // softmax weights of position 1 over keys {0, 1}
  pdl_launch_dependents();
  pdl_wait();
  const int slot = blockIdx.x, kvh = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* kb = static_cast<float*>(kv.k) + (size_t)slot * kv.slot_stride + (size_t)kvh * kv.capacity * 128;  // the code predictor's cache is fp32
  float* vb = static_cast<float*>(kv.v) + (size_t)slot * kv.slot_stride + (size_t)kvh * kv.capacity * 128;
  // work items: (pos, head) with head in {q heads of pos 1 (G), k of pos 0, k of pos 1}; the q heads of position 0 are not needed
  // (a single key: its softmax weight is 1 whatever the score)
  for (int item = warp; item < G + 2; item += 4) {
    const int pos = item < G ? 1 : item - G;
    const float* rowp = qkv + (size_t)(2 * slot + pos) * ld;
    const float* src = rowp + (size_t)(item < G ? (kvh * G + item) : (heads + kvh)) * 128;
    const float a0 = src[lane], a1 = src[lane + 32], b0 = src[lane + 64], b1 = src[lane + 96];
    const float ss = warp_sum(a0 * a0 + a1 * a1 + b0 * b0 + b1 * b1);
    const float inv = rsqrtf(ss * (1.0f / 128.0f) + eps);
    const float* nw = item < G ? q_norm : k_norm;
    const float x0 = a0 * inv * nw[lane], x1 = a1 * inv * nw[lane + 32], y0 = b0 * inv * nw[lane + 64], y1 = b1 * inv * nw[lane + 96];
    float s0 = 0.f, c0 = 1.f, s1 = 0.f, c1 = 1.f;   // position 0: identity rotation (sincosf(0) is exactly (0, 1))
    if (pos == 1) {
      sincosf(inv_freq[lane], &s0, &c0);
      sincosf(inv_freq[lane + 32], &s1, &c1);
    }
    const float o0 = x0 * c0 - y0 * s0, o1 = x1 * c1 - y1 * s1, o2 = y0 * c0 + x0 * s0, o3 = y1 * c1 + x1 * s1;
    float* dst = item < G ? q1 + item * 128 : kk[pos];
    dst[lane] = o0; dst[lane + 32] = o1; dst[lane + 64] = o2; dst[lane + 96] = o3;
    if (item >= G) {  // append k to the cache (ring index == position: the cache holds 17 positions at most)
      float* kd = kb + (size_t)pos * 128;
      kd[lane] = o0; kd[lane + 32] = o1; kd[lane + 64] = o2; kd[lane + 96] = o3;
    }
  }
#pragma unroll
  for (int pos = 0; pos < 2; ++pos) {
    const float v = qkv[(size_t)(2 * slot + pos) * ld + (size_t)(heads + kv_heads + kvh) * 128 + tid];
    vv[pos][tid] = v;
    vb[(size_t)pos * 128 + tid] = v;
  }
  __syncthreads();
  for (int g = warp; g < G; g += 4) {
    float d0 = 0.f, d1 = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float qv = q1[g * 128 + lane + 32 * i];
      d0 = fmaf(qv, kk[0][lane + 32 * i], d0);
      d1 = fmaf(qv, kk[1][lane + 32 * i], d1);
    }
    d0 = warp_sum(d0) * scale;
    d1 = warp_sum(d1) * scale;
    const float mx = fmaxf(d0, d1);
    const float e0 = expf(d0 - mx), e1 = expf(d1 - mx);
    if (lane == 0) { w0[g] = e0 / (e0 + e1); w1[g] = e1 / (e0 + e1); }
  }
  __syncthreads();
#pragma unroll
  for (int g = 0; g < G; ++g) {
    out[(size_t)(2 * slot) * ldo + (size_t)(kvh * G + g) * 128 + tid] = __float2half_rn(vv[0][tid]);
    out[(size_t)(2 * slot + 1) * ldo + (size_t)(kvh * G + g) * 128 + tid] = __float2half_rn(w0[g] * vv[0][tid] + w1[g] * vv[1][tid]);
  }
}
void launch_cp_pass0_attention_f16(const LaunchCtx& c, const float* qkv, int ld, int n_slots, int heads, int kv_heads, const float* q_norm,
                                   const float* k_norm, float eps, const float* inv_freq, const KVLayout& kv, __half* out, int ldo) {
  if (n_slots <= 0) return;
  const int G = heads / kv_heads;
  const float scale = 1.0f / sqrtf(128.0f);
  dim3 grid(n_slots, kv_heads);
  const bool pdl = pdl_enabled();
  Q3_CHECK(G == 1 || G == 2 || G == 4, Q3TTS_ERR_BAD_CONFIG, "unsupported GQA group size %d", G);
  if (G == 1) launch_kernel_pdl(cp_pass0_attention_kernel<1>, grid, dim3(128), 0, c.stream, pdl, qkv, ld, heads, kv_heads, q_norm, k_norm, eps, inv_freq, kv, out, ldo, scale);
  else if (G == 2) launch_kernel_pdl(cp_pass0_attention_kernel<2>, grid, dim3(128), 0, c.stream, pdl, qkv, ld, heads, kv_heads, q_norm, k_norm, eps, inv_freq, kv, out, ldo, scale);
  else launch_kernel_pdl(cp_pass0_attention_kernel<4>, grid, dim3(128), 0, c.stream, pdl, qkv, ld, heads, kv_heads, q_norm, k_norm, eps, inv_freq, kv, out, ldo, scale);
  c.tick();
}

template <typename OutT>
static void launch_rope_attention_t(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, const float* q_norm,
                                    const float* k_norm, float eps, const float* inv_freq, const int* row_slot, const int* row_pos,
                                    const int* win_start, const KVLayout& kv, OutT* out, int ldo) {
  if (m <= 0) return;
  const int G = heads / kv_heads;
  const float scale = 1.0f / sqrtf(128.0f);
  const size_t smem = 0;
  dim3 grid(m, kv_heads);
  const bool pdl = pdl_enabled();
  Q3_CHECK(G == 1 || G == 2 || G == 4, Q3TTS_ERR_BAD_CONFIG, "unsupported GQA group size %d", G);
#define RA_LAUNCH(GV)                                                                                                                              \
  {                                                                                                                                                \
    if (kv.f16) launch_kernel_pdl(rope_attention_kernel<GV, OutT, __half>, grid, dim3(128), smem, c.stream, pdl, qkv, ld, heads, kv_heads, q_norm, k_norm, eps, \
                                  inv_freq, row_slot, row_pos, win_start, kv, out, ldo, scale);                                                    \
    else launch_kernel_pdl(rope_attention_kernel<GV, OutT, float>, grid, dim3(128), smem, c.stream, pdl, qkv, ld, heads, kv_heads, q_norm, k_norm, eps,         \
                           inv_freq, row_slot, row_pos, win_start, kv, out, ldo, scale);                                                           \
  }
  if (G == 1) RA_LAUNCH(1)
  else if (G == 2) RA_LAUNCH(2)
  else RA_LAUNCH(4)
#undef RA_LAUNCH
  c.tick();
}
void launch_rope_attention(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, const float* q_norm,
                           const float* k_norm, float eps, const float* inv_freq, const int* row_slot, const int* row_pos,
                           const int* win_start, const KVLayout& kv, float* out, int ldo) {
  launch_rope_attention_t<float>(c, qkv, ld, m, heads, kv_heads, q_norm, k_norm, eps, inv_freq, row_slot, row_pos, win_start, kv, out, ldo);
}
void launch_rope_attention_f16(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, const float* q_norm,
                               const float* k_norm, float eps, const float* inv_freq, const int* row_slot, const int* row_pos,
                               const int* win_start, const KVLayout& kv, __half* out, int ldo) {
  launch_rope_attention_t<__half>(c, qkv, ld, m, heads, kv_heads, q_norm, k_norm, eps, inv_freq, row_slot, row_pos, win_start, kv, out, ldo);
}

template <typename OutT>
static void launch_attention_t(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, int head_dim,
                               const int* row_slot, const int* row_pos, const int* win_start, const KVLayout& kv, OutT* out, int ldo) {
  Q3_CHECK(head_dim == 128, Q3TTS_ERR_BAD_CONFIG, "talker kernels are specialised for head_dim 128 (got %d)", head_dim);
  if (m <= 0) return;
  const int G = heads / kv_heads;
  const float scale = 1.0f / sqrtf((float)head_dim);
  const size_t smem = (size_t)G * (128 + kv.capacity) * sizeof(float);
  dim3 grid(m, kv_heads);
#define Q3_ATT(GV)                                                                                                     \
  {                                                                                                                    \
    if (kv.f16) attention_kernel<GV, OutT, __half><<<grid, 128, smem, c.stream>>>(qkv, ld, heads, kv_heads, row_slot, row_pos, win_start, kv, out, ldo, scale); \
    else attention_kernel<GV, OutT, float><<<grid, 128, smem, c.stream>>>(qkv, ld, heads, kv_heads, row_slot, row_pos, win_start, kv, out, ldo, scale); \
  }
  Q3_CHECK(smem <= 160 * 1024, Q3TTS_ERR_CAPACITY, "kv_capacity %d too large for the attention kernel", kv.capacity);
  if (G == 1) Q3_ATT(1) else if (G == 2) Q3_ATT(2) else if (G == 4) Q3_ATT(4)
  else fail(Q3TTS_ERR_BAD_CONFIG, "unsupported GQA group size %d", G);
#undef Q3_ATT
  c.tick();
}
void launch_attention(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, int head_dim,
                      const int* row_slot, const int* row_pos, const int* win_start, const KVLayout& kv, float* out, int ldo) {
  launch_attention_t<float>(c, qkv, ld, m, heads, kv_heads, head_dim, row_slot, row_pos, win_start, kv, out, ldo);
}
void launch_attention_f16(const LaunchCtx& c, const float* qkv, int ld, int m, int heads, int kv_heads, int head_dim,
                          const int* row_slot, const int* row_pos, const int* win_start, const KVLayout& kv, __half* out, int ldo) {
  launch_attention_t<__half>(c, qkv, ld, m, heads, kv_heads, head_dim, row_slot, row_pos, win_start, kv, out, ldo);
}

__global__ void weight_to_f16_kernel(const void* __restrict__ w, int dt, int rows, int cols, int interleave, const float* __restrict__ col_scale,
                                     __half* __restrict__ dst) {
  const size_t total = (size_t)rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), cidx = (int)(i - (size_t)r * cols);
    int dr = r;
    if (interleave) dr = r < rows / 2 ? 2 * r : 2 * (r - rows / 2) + 1;
    const float v = load_as_f32(w, i, dt);
    dst[(size_t)dr * cols + cidx] = __float2half_rn(col_scale ? v * col_scale[cidx] : v);
  }
}
void launch_weight_to_f16(const LaunchCtx& c, const void* w, int dt, int rows, int cols, bool interleave_halves, __half* dst,
                          const float* col_scale) {
  const size_t total = (size_t)rows * cols;
  if (total == 0) return;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 32);
  weight_to_f16_kernel<<<blocks, 256, 0, c.stream>>>(w, dt, rows, cols, interleave_halves ? 1 : 0, col_scale, dst);
  c.tick();
}

__global__ void gather_rows_f16_kernel(Embedding e, const int* __restrict__ ids, __half* __restrict__ y, int ldy) {
  const int row = blockIdx.x;
  const int id = ids[row];
  for (int d = threadIdx.x; d < e.dim; d += blockDim.x)
    y[(size_t)row * ldy + d] = (id >= 0 && id < e.rows) ? __float2half_rn(load_as_f32(e.w, (size_t)id * e.dim + d, e.dt)) : __float2half_rn(0.f);
}
void launch_gather_rows_f16(const LaunchCtx& c, const Embedding& e, const int* ids, int n, __half* y, int ldy) {
  if (n <= 0) return;
  gather_rows_f16_kernel<<<n, 256, 0, c.stream>>>(e, ids, y, ldy);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ embeddings / prompt assembly
__global__ void gather_rows_kernel(Embedding e, const int* __restrict__ ids, int n, float* __restrict__ y, int ldy, int accumulate) {
  const int row = blockIdx.x;
  const int id = ids[row];
  if (id < 0 || id >= e.rows) return;
  for (int d = threadIdx.x; d < e.dim; d += blockDim.x) {
    const float v = load_as_f32(e.w, (size_t)id * e.dim + d, e.dt);
    float* p = y + (size_t)row * ldy + d;
    *p = accumulate ? (*p + v) : v;
  }
}
void launch_gather_rows(const LaunchCtx& c, const Embedding& e, const int* ids, int n, float* y, int ldy, bool accumulate) {
  if (n <= 0) return;
  gather_rows_kernel<<<n, 256, 0, c.stream>>>(e, ids, n, y, ldy, accumulate ? 1 : 0);
  c.tick();
}

__global__ void assemble_rows_kernel(const float* __restrict__ tp_rows, int H, Embedding codec, const float* __restrict__ spk,
                                     const int* __restrict__ desc, float* __restrict__ y) {
  const int row = blockIdx.x;
  const int tp = desc[row * 3 + 0], cd = desc[row * 3 + 1], sp = desc[row * 3 + 2];
  for (int d = threadIdx.x; d < H; d += blockDim.x) {
    float v = 0.f;
    if (tp >= 0) v += tp_rows[(size_t)tp * H + d];
    if (cd >= 0) v += load_as_f32(codec.w, (size_t)cd * H + d, codec.dt);
    if (sp > 0) v += spk[(size_t)(sp - 1) * H + d];  // sp = 1 + index of the utterance's raw speaker embedding
    y[(size_t)row * H + d] = v;
  }
}
void launch_assemble_rows(const LaunchCtx& c, const float* tp_rows, int H, const Embedding& codec, const float* spk,
                          const int* desc, int n, float* y) {
  if (n <= 0) return;
  assemble_rows_kernel<<<n, 256, 0, c.stream>>>(tp_rows, H, codec, spk, desc, y);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ voice prefix <-> KV rings
// grid (x: 16-byte vectors of one run, y: run = (K|V, layer, kv head), z: table entry).  A run is n_pos consecutive ring rows of one
// (layer, kv head) and the matching contiguous block of the compact buffer; the copy is a bit copy whatever the element type.
__global__ void __launch_bounds__(256) kv_prefix_copy_kernel(const KvPrefixEntry* __restrict__ table, char* k, char* v, size_t slot_bytes,
                                                             size_t layer_bytes, size_t head_bytes, int layers, int kv_heads, int row_bytes,
                                                             int to_ring) {
  const KvPrefixEntry e = table[blockIdx.z];
  const int run = blockIdx.y, per_kind = layers * kv_heads;
  const int kind = run / per_kind, layer = (run - kind * per_kind) / kv_heads, head = run - kind * per_kind - layer * kv_heads;
  uint4* ring = reinterpret_cast<uint4*>((kind ? v : k) + (size_t)e.slot * slot_bytes + (size_t)layer * layer_bytes + (size_t)head * head_bytes);
  uint4* comp = reinterpret_cast<uint4*>(static_cast<char*>(e.compact) + (size_t)run * e.n_pos * row_bytes);
  const int n_vec = e.n_pos * (row_bytes / 16);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += gridDim.x * blockDim.x) {
    if (to_ring) ring[i] = comp[i];
    else comp[i] = ring[i];
  }
}

void launch_kv_prefix_copy(const LaunchCtx& c, const KvPrefixEntry* table, int n_entries, int max_pos, void* k, void* v, size_t slot_stride,
                           size_t layer_stride, int layers, int kv_heads, int capacity, int elem_bytes, bool to_ring) {
  if (n_entries <= 0 || max_pos <= 0) return;
  Q3_CHECK(elem_bytes == 2 || elem_bytes == 4, Q3TTS_ERR_INVALID_ARG, "kv prefix copy: element size %d", elem_bytes);
  Q3_CHECK(max_pos <= capacity && n_entries <= 65535 && 2 * layers * kv_heads <= 65535, Q3TTS_ERR_INVALID_ARG, "kv prefix copy: bad shape");
  const int row_bytes = 128 * elem_bytes;
  const int n_vec = max_pos * (row_bytes / 16);
  dim3 grid((n_vec + 255) / 256, 2 * layers * kv_heads, n_entries);
  kv_prefix_copy_kernel<<<grid, 256, 0, c.stream>>>(table, static_cast<char*>(k), static_cast<char*>(v), slot_stride * elem_bytes,
                                                    layer_stride * elem_bytes, (size_t)capacity * row_bytes, layers, kv_heads, row_bytes,
                                                    to_ring ? 1 : 0);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ sampler
// (device code in sampler.cuh, shared with the frame megakernel)
// After the group's token is known the same CTA writes the code predictor's NEXT input rows (Qwen3Talker.swift:501-523:
// pass 0 = [last hidden, codec_embedding(code0)], pass g = cp.codec_embedding[g-1](code_g)) -- fp32, and optionally the fp16
// operand copy the tensor-core stack reads -- so a frame has no separate input-row or conversion launches.
__global__ void __launch_bounds__(kSampleThreads) sample_kernel(const float* __restrict__ logits, int ld, SlotState* __restrict__ st,
                                                               SamplerParams p, unsigned* __restrict__ token_sets,
                                                               int* __restrict__ cur_codes, const int* __restrict__ forced,
                                                               int max_frames, float* __restrict__ dump, int dump_stride_frame,
                                                               int dump_offset, int dump_slot, NextInput ni) {
  __shared__ float sl[kMaxVocab];
  __shared__ BlockRed br;
  sample_slot<0, kSampleThreads>(blockIdx.x, logits, ld, st, p, token_sets, cur_codes, forced, max_frames, dump, dump_stride_frame, dump_offset, dump_slot, sl, br);
  if (ni.mode == 0) return;
  __syncthreads();  // cur_codes[slot][group] written by thread 0 of this CTA
  const int slot = blockIdx.x, H = ni.H;
  const int code = cur_codes[slot * p.groups + p.group];
  if (ni.mode == 1) {  // -> pass 0
    const bool ok = code >= 0 && code < ni.codec.rows;
    for (int d = threadIdx.x; d < H; d += kSampleThreads) {
      const float a = ni.h_last[(size_t)slot * H + d];
      const float b = ok ? load_as_f32(ni.codec.w, (size_t)code * H + d, ni.codec.dt) : 0.f;
      ni.y32[(size_t)(2 * slot) * H + d] = a;
      ni.y32[(size_t)(2 * slot + 1) * H + d] = b;
      if (ni.y16) {
        ni.y16[(size_t)(2 * slot) * H + d] = __float2half_rn(a * ni.y16_scale);
        ni.y16[(size_t)(2 * slot + 1) * H + d] = __float2half_rn(b * ni.y16_scale);
      }
    }
  } else {             // -> pass p.group (>= 1)
    const Embedding e = ni.cp_emb[p.group - 1];
    const bool ok = code >= 0 && code < e.rows;
    for (int d = threadIdx.x; d < H; d += kSampleThreads) {
      const float v = ok ? load_as_f32(e.w, (size_t)code * H + d, e.dt) : 0.f;
      ni.y32[(size_t)slot * H + d] = v;
      if (ni.y16) ni.y16[(size_t)slot * H + d] = __float2half_rn(v * ni.y16_scale);
    }
  }
}
void launch_sample(const LaunchCtx& c, const float* logits, int ld, int n_slots, SlotState* st, const SamplerParams& p,
                   unsigned* token_sets, int* cur_codes, const int* forced, int max_frames, float* logits_dump,
                   int dump_stride_frame, int dump_offset, int dump_slot, const NextInput& ni) {
  Q3_CHECK(p.vocab <= kMaxVocab, Q3TTS_ERR_BAD_CONFIG, "sampler supports vocab <= %d (got %d)", kMaxVocab, p.vocab);
  sample_kernel<<<n_slots, kSampleThreads, 0, c.stream>>>(logits, ld, st, p, token_sets, cur_codes, forced, max_frames, logits_dump,
                                                          dump_stride_frame, dump_offset, dump_slot, ni);
  c.tick();
}

__global__ void __launch_bounds__(kSampleThreads) sample_probe_kernel(const float* __restrict__ logits, int V, int codec_vocab,
                                                                     float temperature, int top_k, float top_p, float rep_penalty,
                                                                     const unsigned* __restrict__ set_bitmap, unsigned long long seed,
                                                                     unsigned long long counter, int* __restrict__ id_out) {
  __shared__ float sl[kMaxVocab];
  __shared__ BlockRed br;
  for (int i = threadIdx.x; i < V; i += kSampleThreads) sl[i] = logits[i];
  __syncthreads();
  const int tok = sample_block<0, kSampleThreads>(sl, V, codec_vocab, temperature, top_k, top_p, rep_penalty, set_bitmap, seed, counter, br);
  if (threadIdx.x == 0) *id_out = tok;
}
void launch_sample_probe(const LaunchCtx& c, const float* logits, int vocab, int codec_vocab, float temperature, int top_k,
                         float top_p, float rep_penalty, const unsigned* set_bitmap, unsigned long long seed,
                         unsigned long long counter, int* id_out) {
  Q3_CHECK(vocab <= kMaxVocab, Q3TTS_ERR_INVALID_ARG, "sampler supports vocab <= %d (got %d)", kMaxVocab, vocab);
  sample_probe_kernel<<<1, kSampleThreads, 0, c.stream>>>(logits, vocab, codec_vocab, temperature, top_k, top_p, rep_penalty,
                                                          set_bitmap, seed, counter, id_out);
  c.tick();
}

// q3tts_sampler_probe / q3tts_sampler_slot_probe.  FORM 0 runs the sampler as sample_kernel does (__syncthreads over 512
// threads), FORM 1 as frame_megakernel does: named barrier 1 over warps 0-14 of a 512-thread CTA, warp 15 idle.
template <int FORM>
constexpr int probe_threads() { return FORM == 0 ? kSampleThreads : kFrameSampleThreads; }

template <int FORM, bool DUMP>
__global__ void __launch_bounds__(kSampleThreads) sampler_probe_kernel(const float* __restrict__ logits, int ld, int V, int codec_vocab,
                                                                      SamplerProbeRows rows, int* __restrict__ ids,
                                                                      float* __restrict__ processed) {
  constexpr int NT = probe_threads<FORM>();
  __shared__ float sl[kMaxVocab];
  __shared__ BlockRed br;
  if (threadIdx.x >= NT) return;
  const int r = blockIdx.x;
  for (int i = threadIdx.x; i < V; i += NT) sl[i] = logits[(size_t)r * ld + i];
  block_sync<FORM, NT>();
  const int tok = sample_block<FORM, NT, DUMP>(sl, V, codec_vocab, rows.temperature[r], rows.top_k[r], rows.top_p[r], rows.rep_penalty[r],
                                               rows.sets ? rows.sets + (size_t)r * (kMaxVocab / 32) : nullptr, rows.seed[r], rows.counter[r],
                                               br, DUMP ? processed + (size_t)r * V : nullptr);
  if (threadIdx.x == 0) ids[r] = tok;
}
void launch_sampler_probe(const LaunchCtx& c, int form, const float* logits, int ld, int n_rows, int V, int codec_vocab,
                          const SamplerProbeRows& rows, int* ids, float* processed) {
  Q3_CHECK(V >= 1 && V <= kMaxVocab && n_rows >= 1 && (form == 0 || form == 1), Q3TTS_ERR_INVALID_ARG, "sampler probe: bad V %d / rows %d / form %d",
           V, n_rows, form);
  auto k = form == 0 ? (processed ? sampler_probe_kernel<0, true> : sampler_probe_kernel<0, false>)
                     : (processed ? sampler_probe_kernel<1, true> : sampler_probe_kernel<1, false>);
  k<<<n_rows, kSampleThreads, 0, c.stream>>>(logits, ld, V, codec_vocab, rows, ids, processed);
  c.tick();
}

__global__ void __launch_bounds__(kSampleThreads) sample_slot_frame_form_kernel(const float* __restrict__ logits, int ld, SlotState* __restrict__ st,
                                                                               SamplerParams p, unsigned* __restrict__ token_sets,
                                                                               int* __restrict__ cur_codes, const int* __restrict__ forced,
                                                                               int max_frames, float* __restrict__ dump, int dump_stride_frame,
                                                                               int dump_offset, int dump_slot) {
  __shared__ float sl[kMaxVocab];
  __shared__ BlockRed br;
  if (threadIdx.x >= kFrameSampleThreads) return;
  sample_slot<1, kFrameSampleThreads>(blockIdx.x, logits, ld, st, p, token_sets, cur_codes, forced, max_frames, dump, dump_stride_frame,
                                      dump_offset, dump_slot, sl, br);
}
void launch_sample_frame_form(const LaunchCtx& c, const float* logits, int ld, int n_slots, SlotState* st, const SamplerParams& p,
                              unsigned* token_sets, int* cur_codes, const int* forced, int max_frames, float* logits_dump,
                              int dump_stride_frame, int dump_offset, int dump_slot) {
  Q3_CHECK(p.vocab <= kMaxVocab, Q3TTS_ERR_BAD_CONFIG, "sampler supports vocab <= %d (got %d)", kMaxVocab, p.vocab);
  sample_slot_frame_form_kernel<<<n_slots, kSampleThreads, 0, c.stream>>>(logits, ld, st, p, token_sets, cur_codes, forced, max_frames,
                                                                          logits_dump, dump_stride_frame, dump_offset, dump_slot);
  c.tick();
}

// ------------------------------------------------------------------------------------------------ frame plumbing
__global__ void cp_input_kernel(int pass, const float* __restrict__ h_last, int H, Embedding codec, const Embedding* __restrict__ cp_emb,
                                const int* __restrict__ cur_codes, float* __restrict__ y, int groups) {
  const int slot = blockIdx.x;
  if (pass == 0) {
    const int code0 = cur_codes[slot * groups];
    const bool ok = code0 >= 0 && code0 < codec.rows;
    for (int d = threadIdx.x; d < H; d += blockDim.x) {
      y[(size_t)(2 * slot) * H + d] = h_last[(size_t)slot * H + d];
      y[(size_t)(2 * slot + 1) * H + d] = ok ? load_as_f32(codec.w, (size_t)code0 * H + d, codec.dt) : 0.f;
    }
  } else {
    const Embedding e = cp_emb[pass - 1];
    const int code = cur_codes[slot * groups + pass];
    const bool ok = code >= 0 && code < e.rows;
    for (int d = threadIdx.x; d < H; d += blockDim.x)
      y[(size_t)slot * H + d] = ok ? load_as_f32(e.w, (size_t)code * H + d, e.dt) : 0.f;
  }
}
void launch_cp_input(const LaunchCtx& c, int pass, int n_slots, const float* h_last, int H, const Embedding& codec,
                     const Embedding* cp_emb_dev, const int* cur_codes, float* y) {
  cp_input_kernel<<<n_slots, 256, 0, c.stream>>>(pass, h_last, H, codec, cp_emb_dev, cur_codes, y, 16);
  c.tick();
}

__global__ void frame_finalize_kernel(SlotState* __restrict__ st, const int* __restrict__ cur_codes, int* __restrict__ frames_out,
                                      int max_frames, unsigned* __restrict__ token_sets, int set_words,
                                      const float* __restrict__ trailing, int max_trailing, const float* __restrict__ tts_pad,
                                      Embedding codec, const Embedding* __restrict__ cp_emb, int H, float* __restrict__ x_next,
                                      __half* __restrict__ x16_next, float x16_scale) {
  const int slot = blockIdx.x;
  SlotState& s = st[slot];
  if (!s.frame_alive) return;
  constexpr int G = 16;
  __shared__ int codes[G];
  __shared__ const void* rowp[G];  // embedding row of each group's code (null: out of range), resolved once per CTA
  __shared__ int rowdt[G];
  if (threadIdx.x < G) {
    const int g = threadIdx.x, code = cur_codes[slot * G + g];
    codes[g] = code;
    const Embedding e = g == 0 ? codec : cp_emb[g - 1];
    const bool ok = code >= 0 && code < e.rows;
    rowp[g] = ok ? static_cast<const char*>(e.w) + (size_t)code * H * (e.dt == Q3TTS_F32 ? 4 : 2) : nullptr;
    rowdt[g] = e.dt;
  }
  __syncthreads();
  const int ti = s.trailing_idx;
  const float* text = (ti < s.total_text) ? trailing + ((size_t)slot * max_trailing + ti) * H : tts_pad;
  for (int d = threadIdx.x; d < H; d += blockDim.x) {
    // codecEmbedSum = codec_embedding(code0) + sum_i cp.codec_embedding[i](code_{i+1}); input = text + sum (:531-548)
    float v[G];
#pragma unroll
    for (int g = 0; g < G; ++g) v[g] = rowp[g] ? load_as_f32(rowp[g], (size_t)d, rowdt[g]) : 0.f;  // 16 independent loads
    float sum = v[0];
#pragma unroll
    for (int g = 1; g < G; ++g) sum += v[g];  // same order as before: code0, then groups 1..15
    const float x = text[d] + sum;
    x_next[(size_t)slot * H + d] = x;
    if (x16_next) x16_next[(size_t)slot * H + d] = __float2half_rn(x * x16_scale);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s.n_frames < max_frames) {
      for (int g = 0; g < G; ++g) frames_out[((size_t)slot * max_frames + s.n_frames) * G + g] = codes[g];
      s.n_frames += 1;
    }
    if (codes[0] >= 0 && codes[0] < set_words * 32) {
      unsigned* set0 = token_sets + (size_t)slot * G * set_words;
      set0[codes[0] >> 5] |= 1u << (codes[0] & 31);  // generatedCode0TokensSet.insert (:528)
    }
    if (ti < s.total_text) s.trailing_idx = ti + 1;
  }
}
void launch_frame_finalize(const LaunchCtx& c, int n_slots, SlotState* st, const int* cur_codes, int* frames_out,
                           int max_frames, unsigned* token_sets, int set_words, const float* trailing, int max_trailing,
                           const float* tts_pad, const Embedding& codec, const Embedding* cp_emb_dev, int H, float* x_next,
                           __half* x16_next, float x16_scale) {
  frame_finalize_kernel<<<n_slots, 256, 0, c.stream>>>(st, cur_codes, frames_out, max_frames, token_sets, set_words, trailing,
                                                       max_trailing, tts_pad, codec, cp_emb_dev, H, x_next, x16_next, x16_scale);
  c.tick();
}

__global__ void step_advance_kernel(int n_slots, SlotState* __restrict__ st, int window) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_slots) return;
  SlotState& s = st[slot];
  if (!s.frame_alive) return;
  s.pos += 1;
  s.step += 1;
  // trimKVCache every 15th step when longer than the window (Model/Qwen3Talker.swift:556-558; Qwen3Layers.swift:111-124)
  if (s.step % 15 == 0 && s.pos - s.win_start > window) s.win_start = s.pos - window;
  if (s.step >= s.max_tokens) s.finished = 1;
  s.frame_alive = 0;
}
void launch_step_advance(const LaunchCtx& c, int n_slots, SlotState* st, int window) {
  step_advance_kernel<<<(n_slots + 63) / 64, 64, 0, c.stream>>>(n_slots, st, window);
  c.tick();
}

__global__ void step_rows_kernel(int n_slots, const SlotState* __restrict__ st, int* __restrict__ row_slot, int* __restrict__ row_pos,
                                 int* __restrict__ win_start) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_slots) return;
  row_slot[slot] = slot;
  row_pos[slot] = st[slot].pos;
  win_start[slot] = st[slot].win_start;
}
void launch_step_rows(const LaunchCtx& c, int n_slots, const SlotState* st, int* row_slot, int* row_pos, int* win_start) {
  step_rows_kernel<<<(n_slots + 63) / 64, 64, 0, c.stream>>>(n_slots, st, row_slot, row_pos, win_start);
  c.tick();
}

// Opt-in dynamic shared memory above 48 KB, set once per device at handle creation (never during graph capture).
template <int FMT>
static void init_linear_fmt() {
  Q3_CUDA(cudaFuncSetAttribute(linear_kernel<FMT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  Q3_CUDA(cudaFuncSetAttribute(linear_kernel<FMT, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  Q3_CUDA(cudaFuncSetAttribute(linear_kernel<FMT, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  Q3_CUDA(cudaFuncSetAttribute(linear_kernel<FMT, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
}
void init_talker_kernels() {
  init_linear_fmt<W_Q4>();
  init_linear_fmt<W_Q8>();
  init_linear_fmt<W_BF16>();
  init_linear_fmt<W_F16>();
  init_linear_fmt<W_F32>();
  // rope_attention_kernel uses static shared memory only; attention_kernel keeps [G][128 + window] floats in dynamic shared memory
#define Q3_ATT_ATTR(GV, OT, KT) Q3_CUDA(cudaFuncSetAttribute(attention_kernel<GV, OT, KT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
#define Q3_ATT_ATTR_G(OT, KT) Q3_ATT_ATTR(1, OT, KT) Q3_ATT_ATTR(2, OT, KT) Q3_ATT_ATTR(4, OT, KT)
  Q3_ATT_ATTR_G(float, float) Q3_ATT_ATTR_G(float, __half) Q3_ATT_ATTR_G(__half, float) Q3_ATT_ATTR_G(__half, __half)
#undef Q3_ATT_ATTR_G
#undef Q3_ATT_ATTR
}

}  // namespace q3
