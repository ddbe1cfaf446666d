// Codec-decoder kernels, first correct (fp32 SIMT) generation.  Channels-last [B, T, C] activations.
// The dense contractions (causal convs, polyphase transposed convs, linears) all go through one implicit-GEMM
// formulation:  Y[m, n] = bias[n] + sum_tap X[m - shift(tap), :] . W[tap][n][:]   with m = b*T + t and rows whose source
// time is negative reading zeros (causal left padding, Vocoder/SpeechTokenizer.swift:160-169, 796-801).
#include "codec_kernels.h"

namespace q3 {

__device__ __forceinline__ float warp_sum_c(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max_c(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------------------------------------- implicit-GEMM conv (SIMT fp32)
constexpr int CB_M = 64, CB_N = 64, CB_K = 16;

__global__ void __launch_bounds__(256) conv_gemm_kernel(const float* __restrict__ x, ConvW w, float* y, const float* res,
                                                        const float* __restrict__ scale, int M, int T, int epi) {
  __shared__ float As[CB_K][CB_M + 4];
  __shared__ float Bs[CB_K][CB_N + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.x * CB_M, n0 = blockIdx.y * CB_N;  // M tiles on x: up to 2^31-1 blocks
  const int lrow = tid >> 2, kq = (tid & 3) * 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int am = m0 + lrow;
  const int at = am % T;
  const bool vec = (w.cin & 3) == 0;
  for (int tap = 0; tap < w.ntap; ++tap) {
    const int shift = (w.ntap - 1 - tap) * w.dil;
    const bool a_ok = am < M && (at - shift) >= 0;
    const float* xa = x + (size_t)(am - shift) * w.cin;
    const int bn = n0 + lrow;
    const bool b_ok = bn < w.n;
    const float* wb = w.w + ((size_t)tap * w.n + bn) * w.cin;
    for (int c0 = 0; c0 < w.cin; c0 += CB_K) {
      float av[4] = {0.f, 0.f, 0.f, 0.f}, bv[4] = {0.f, 0.f, 0.f, 0.f};
      const int c = c0 + kq;
      if (vec && c + 3 < w.cin) {
        if (a_ok) { const float4 t4 = *reinterpret_cast<const float4*>(xa + c); av[0] = t4.x; av[1] = t4.y; av[2] = t4.z; av[3] = t4.w; }
        if (b_ok) { const float4 t4 = *reinterpret_cast<const float4*>(wb + c); bv[0] = t4.x; bv[1] = t4.y; bv[2] = t4.z; bv[3] = t4.w; }
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (c + i < w.cin) {
            if (a_ok) av[i] = xa[c + i];
            if (b_ok) bv[i] = wb[c + i];
          }
        }
      }
      __syncthreads();
#pragma unroll
      for (int i = 0; i < 4; ++i) { As[kq + i][lrow] = av[i]; Bs[kq + i][lrow] = bv[i]; }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < CB_K; ++k) {
        const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
        const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
        const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= w.n) continue;
      float v = acc[i][j] + (w.bias ? w.bias[n] : 0.f);
      const size_t o = (size_t)m * w.n + n;
      if (epi == CE_GELU) v = 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f));  // exact erf GELU (:230)
      else if (epi == CE_RES_SCALE) v = res[o] + (scale ? scale[n] : 1.0f) * v;
      y[o] = v;
    }
  }
}

void launch_conv_gemm(const LaunchCtx& c, const float* x, const ConvW& w, float* y, const float* res, const float* scale, int M,
                      int T, int epi) {
  if (M <= 0) return;
  dim3 grid((M + CB_M - 1) / CB_M, (w.n + CB_N - 1) / CB_N);
  conv_gemm_kernel<<<grid, 256, 0, c.stream>>>(x, w, y, res, scale, M, T, epi);
  c.tick();
}

// ---------------------------------------------------------------------------------------------- elementwise / small ops
__global__ void snake_kernel(const float* __restrict__ x, const float* __restrict__ ea, const float* __restrict__ inv_eb, int C,
                             size_t total, float* __restrict__ y) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int ch = (int)(i % C);
    const float v = x[i];
    const float s = sinf(v * ea[ch]);
    y[i] = v + inv_eb[ch] * (s * s);  // x + sin^2(x e^alpha) / (e^beta + 1e-9)  (SpeechTokenizer.swift:105-109)
  }
}
void launch_snake(const LaunchCtx& c, const float* x, const SnakeW& s, size_t rows, float* y) {
  const size_t total = rows * s.ch;
  if (total == 0) return;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 32);
  snake_kernel<<<blocks, 256, 0, c.stream>>>(x, s.alpha, s.beta, s.ch, total, y);
  c.tick();
}

__global__ void dwconv7_kernel(const float* __restrict__ x, const float* __restrict__ w /*[7][C]*/, const float* __restrict__ b,
                               int C, int T, size_t total, float* __restrict__ y) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int ch = (int)(i % C);
    const size_t m = i / C;
    const int t = (int)(m % T);
    float acc = b[ch];
#pragma unroll
    for (int k = 0; k < 7; ++k) {
      const int sh = 6 - k;
      if (t - sh >= 0) acc = fmaf(x[i - (size_t)sh * C], w[k * C + ch], acc);
    }
    y[i] = acc;
  }
}
void launch_dwconv7(const LaunchCtx& c, const float* x, const float* w, const float* b, int C, int T, size_t rows, float* y) {
  const size_t total = rows * C;
  if (total == 0) return;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 32);
  dwconv7_kernel<<<blocks, 256, 0, c.stream>>>(x, w, b, C, T, total, y);
  c.tick();
}

__device__ __forceinline__ void store_out(float* p, float v) { *p = v; }
__device__ __forceinline__ void store_out(__half* p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ float load_in(const float* p) { return *p; }
__device__ __forceinline__ float load_in(const __half* p) { return __half2float(*p); }

template <typename OutT>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, int C, const float* __restrict__ w,
                                                        const float* __restrict__ b, float eps, OutT* __restrict__ y) {
  __shared__ float red[8], red2[8];
  const float* xr = x + (size_t)blockIdx.x * C;
  float s = 0.f;
  for (int i = threadIdx.x; i < C; i += 256) s += xr[i];
  s = warp_sum_c(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  float mean = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) mean += red[i];
  mean /= (float)C;
  float v = 0.f;
  for (int i = threadIdx.x; i < C; i += 256) { const float d = xr[i] - mean; v += d * d; }
  v = warp_sum_c(v);
  if ((threadIdx.x & 31) == 0) red2[threadIdx.x >> 5] = v;
  __syncthreads();
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) var += red2[i];
  const float inv = rsqrtf(var / (float)C + eps);
  OutT* yr = y + (size_t)blockIdx.x * C;
  for (int i = threadIdx.x; i < C; i += 256) store_out(yr + i, (xr[i] - mean) * inv * w[i] + b[i]);
}
void launch_layernorm(const LaunchCtx& c, const float* x, int rows, int C, const float* w, const float* b, float eps, float* y) {
  if (rows <= 0) return;
  layernorm_kernel<float><<<rows, 256, 0, c.stream>>>(x, C, w, b, eps, y);
  c.tick();
}
void launch_layernorm_f16(const LaunchCtx& c, const float* x, int rows, int C, const float* w, const float* b, float eps, __half* y) {
  if (rows <= 0) return;
  layernorm_kernel<__half><<<rows, 256, 0, c.stream>>>(x, C, w, b, eps, y);
  c.tick();
}

__global__ void silu_mul_kernel(const float* __restrict__ gu, int I, size_t total, float* __restrict__ y) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t m = i / I;
    const int j = (int)(i % I);
    const float g = gu[m * 2 * I + j], u = gu[m * 2 * I + I + j];
    y[i] = (g / (1.0f + expf(-g))) * u;
  }
}
void launch_silu_mul(const LaunchCtx& c, const float* gu, size_t rows, int I, float* y) {
  const size_t total = rows * I;
  if (total == 0) return;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 32);
  silu_mul_kernel<<<blocks, 256, 0, c.stream>>>(gu, I, total, y);
  c.tick();
}

// RoPE of the codec transformer: head_dim 64, positions restart at 0 in every window (SpeechTokenizer.swift:469-472, 304-317)
__global__ void codec_rope_kernel(float* __restrict__ qkv, int ld, int M, int T, int n_rot_heads, const float* __restrict__ inv_freq) {
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (gw >= M * n_rot_heads) return;
  const int m = gw / n_rot_heads, h = gw - m * n_rot_heads, lane = threadIdx.x & 31;
  float* p = qkv + (size_t)m * ld + (size_t)h * 64;
  const float ang = (float)(m % T) * inv_freq[lane];
  float s, co;
  sincosf(ang, &s, &co);
  const float a = p[lane], b = p[lane + 32];
  p[lane] = a * co - b * s;
  p[lane + 32] = b * co + a * s;
}
void launch_codec_rope(const LaunchCtx& c, float* qkv, int ld, int M, int T, int n_rot_heads, const float* inv_freq) {
  const int warps = M * n_rot_heads;
  if (warps <= 0) return;
  codec_rope_kernel<<<(warps + 3) / 4, 128, 0, c.stream>>>(qkv, ld, M, T, n_rot_heads, inv_freq);
  c.tick();
}

// Full-causal MHA, head_dim 64, online softmax; grid (q tiles of 16, heads, batch), 4 warps x 4 query rows.
template <typename OutT>
__global__ void __launch_bounds__(128) codec_attention_kernel(const float* __restrict__ qkv, int ld, int T, int nh, int nkv, float scale,
                                                              OutT* __restrict__ out, int ldo, int causal) {
  __shared__ float Ks[32][65];
  __shared__ float Vs[32][64];
  __shared__ float Qs[16][64];
  const int r0 = blockIdx.x * 16, h = blockIdx.y, b = blockIdx.z;
  const int kvh = h / (nh / nkv);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* base = qkv + (size_t)b * T * ld;
  for (int i = tid; i < 16 * 64; i += 128) {
    const int r = i >> 6, d = i & 63;
    Qs[r][d] = (r0 + r < T) ? base[(size_t)(r0 + r) * ld + h * 64 + d] : 0.f;
  }
  float mi[4], li[4], acc[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) { mi[i] = -INFINITY; li[i] = 0.f; acc[i][0] = acc[i][1] = 0.f; }
  const int koff = nh * 64 + kvh * 64, voff = nh * 64 + nkv * 64 + kvh * 64;
  const int last = causal ? min(T, r0 + 16) : T;  // causal = 0: the ICL encoder's bidirectional attention (Qwen3TTSAudioEncoder.swift:331)
  for (int kt = 0; kt < last; kt += 32) {
    __syncthreads();
    for (int i = tid; i < 32 * 64; i += 128) {
      const int r = i >> 6, d = i & 63;
      const bool ok = kt + r < T;
      Ks[r][d] = ok ? base[(size_t)(kt + r) * ld + koff + d] : 0.f;
      Vs[r][d] = ok ? base[(size_t)(kt + r) * ld + voff + d] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rl = warp * 4 + i, row = r0 + rl;
      if (row >= T) continue;
      float s = 0.f;
#pragma unroll 16
      for (int d = 0; d < 64; ++d) s = fmaf(Qs[rl][d], Ks[lane][d], s);
      const int j = kt + lane;
      s = ((j <= row || !causal) && j < T) ? s * scale : -INFINITY;
      const float mt = warp_max_c(s);
      const float mnew = fmaxf(mi[i], mt);
      if (mnew == -INFINITY) continue;  // whole tile masked for this row
      const float p = (s == -INFINITY) ? 0.f : expf(s - mnew);
      const float corr = (mi[i] == -INFINITY) ? 0.f : expf(mi[i] - mnew);
      li[i] = li[i] * corr + warp_sum_c(p);
      float a0 = acc[i][0] * corr, a1 = acc[i][1] * corr;
#pragma unroll 8
      for (int jj = 0; jj < 32; ++jj) {
        const float pj = __shfl_sync(0xffffffffu, p, jj);
        a0 = fmaf(pj, Vs[jj][lane], a0);
        a1 = fmaf(pj, Vs[jj][lane + 32], a1);
      }
      acc[i][0] = a0; acc[i][1] = a1;
      mi[i] = mnew;
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = r0 + warp * 4 + i;
    if (row >= T) continue;
    OutT* o = out + ((size_t)b * T + row) * ldo + h * 64;
    store_out(o + lane, acc[i][0] / li[i]);
    store_out(o + lane + 32, acc[i][1] / li[i]);
  }
}
void launch_codec_attention(const LaunchCtx& c, const float* qkv, int ld, int B, int T, int nh, int nkv, float* out, int ldo) {
  if (B <= 0 || T <= 0) return;
  dim3 grid((T + 15) / 16, nh, B);
  codec_attention_kernel<float><<<grid, 128, 0, c.stream>>>(qkv, ld, T, nh, nkv, 1.0f / sqrtf(64.0f), out, ldo, 1);
  c.tick();
}
void launch_codec_attention_bidir(const LaunchCtx& c, const float* qkv, int ld, int B, int T, int nh, int nkv, float* out, int ldo) {
  if (B <= 0 || T <= 0) return;
  dim3 grid((T + 15) / 16, nh, B);
  codec_attention_kernel<float><<<grid, 128, 0, c.stream>>>(qkv, ld, T, nh, nkv, 1.0f / sqrtf(64.0f), out, ldo, 0);
  c.tick();
}
// The same attention on tensor cores (mma.sync m16n8k16, fp16 operands, fp32 accumulate and softmax): the codec transformer's windows
// are 18-750 frames of 16 heads x 64 dims -- a tile problem far too small for tcgen05 (a 128-row UMMA tile would be 80 % padding at
// T = 26) but 3 000 shared-memory loads per CTA as a SIMT loop (52 us per layer at 64 x 26 frames, LDS-bound).  One warp owns 16 query
// rows: Q fragments live in registers, K and V^T tiles of 64 keys are staged in shared memory as fp16 (row pitch 72 halves: the
// fragment loads of the 8 x 4 lane grid hit 32 different banks), S = Q.K^T -> online softmax in registers -> the probabilities ARE the A
// fragments of P.V (accumulator layout of one m16n8 tile = half an A fragment of the next MMA).  Operands are rounded to fp16 once
// (q, k after RoPE, v, p): the same rounding every other contraction of this pipeline applies.
__device__ __forceinline__ uint32_t att_pack(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void att_mma(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__global__ void __launch_bounds__(128) codec_attention_mma_kernel(const float* __restrict__ qkv, int ld, int T, int nh, int nkv, float scale,
                                                                  __half* __restrict__ out, int ldo, int causal) {
  constexpr int KT = 64, PITCH = 72;
  __shared__ __align__(16) __half Ks[KT][PITCH];   // [key][dim]
  __shared__ __align__(16) __half Vt[64][PITCH];   // [dim][key]
  const int h = blockIdx.y, b = blockIdx.z, kvh = h / (nh / nkv);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int r0 = blockIdx.x * 64 + warp * 16;  // this warp's first query row
  const float* base = qkv + (size_t)b * T * ld;
  const int koff = nh * 64 + kvh * 64, voff = nh * 64 + nkv * 64 + kvh * 64;
  // Q fragments: rows r0 + g and r0 + g + 8, 4 k-steps of 16 dims
  uint32_t qa[4][4];
  {
    const int ra = r0 + g, rb = r0 + g + 8;
    const float* qra = base + (size_t)(ra < T ? ra : 0) * ld + h * 64;
    const float* qrb = base + (size_t)(rb < T ? rb : 0) * ld + h * 64;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const float2 a_lo = *reinterpret_cast<const float2*>(qra + ks * 16 + 2 * t), a_hi = *reinterpret_cast<const float2*>(qra + ks * 16 + 8 + 2 * t);
      const float2 b_lo = *reinterpret_cast<const float2*>(qrb + ks * 16 + 2 * t), b_hi = *reinterpret_cast<const float2*>(qrb + ks * 16 + 8 + 2 * t);
      qa[ks][0] = att_pack(a_lo.x, a_lo.y); qa[ks][1] = att_pack(b_lo.x, b_lo.y);
      qa[ks][2] = att_pack(a_hi.x, a_hi.y); qa[ks][3] = att_pack(b_hi.x, b_hi.y);
    }
  }
  float o[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
  float m_a = -INFINITY, m_b = -INFINITY, l_a = 0.f, l_b = 0.f;  // rows r0 + g / r0 + g + 8
  const int cta_last = causal ? min(T, (int)blockIdx.x * 64 + 64) : T;   // keys any warp of this CTA needs
  const int my_last = causal ? min(T, r0 + 16) : T;                      // keys THIS warp needs (uniform per warp)
  for (int kt = 0; kt < cta_last; kt += KT) {
    __syncthreads();
    for (int i = tid; i < KT * 16; i += 128) {  // 64 keys x 16 float4 of K and of V
      const int r = i >> 4, d = (i & 15) * 4;
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (kt + r < T) {
        kv = *reinterpret_cast<const float4*>(base + (size_t)(kt + r) * ld + koff + d);
        vv = *reinterpret_cast<const float4*>(base + (size_t)(kt + r) * ld + voff + d);
      }
      *reinterpret_cast<uint2*>(&Ks[r][d]) = make_uint2(att_pack(kv.x, kv.y), att_pack(kv.z, kv.w));
      Vt[d][r] = __float2half_rn(vv.x); Vt[d + 1][r] = __float2half_rn(vv.y); Vt[d + 2][r] = __float2half_rn(vv.z); Vt[d + 3][r] = __float2half_rn(vv.w);
    }
    __syncthreads();
    if (kt >= my_last || r0 >= T) continue;  // warp-uniform: nothing of this tile is visible to this warp's rows
    // S = Q . K^T for 64 keys: 8 n-tiles of 8 keys
    float sc[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      sc[n][0] = sc[n][1] = sc[n][2] = sc[n][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(&Ks[n * 8 + g][ks * 16 + 2 * t]);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(&Ks[n * 8 + g][ks * 16 + 8 + 2 * t]);
        att_mma(sc[n], qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3], b0, b1);
      }
    }
    // mask + scale; row maxima
    const int ra = r0 + g, rb = r0 + g + 8;
    float mx_a = -INFINITY, mx_b = -INFINITY;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int j = kt + n * 8 + 2 * t + e;
        const bool in = j < T;
        sc[n][e] = (in && (!causal || j <= ra)) ? sc[n][e] * scale : -INFINITY;
        sc[n][2 + e] = (in && (!causal || j <= rb)) ? sc[n][2 + e] * scale : -INFINITY;
        mx_a = fmaxf(mx_a, sc[n][e]); mx_b = fmaxf(mx_b, sc[n][2 + e]);
      }
    }
    mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 1)); mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 2));
    mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 1)); mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 2));
    const float mn_a = fmaxf(m_a, mx_a), mn_b = fmaxf(m_b, mx_b);
    // a row with nothing visible yet keeps m = -inf: use 0 as the reference so exp(-inf - 0) = 0 (no NaN)
    const float ref_a = mn_a == -INFINITY ? 0.f : mn_a, ref_b = mn_b == -INFINITY ? 0.f : mn_b;
    const float corr_a = m_a == -INFINITY ? 0.f : __expf(m_a - ref_a), corr_b = m_b == -INFINITY ? 0.f : __expf(m_b - ref_b);
    float sum_a = 0.f, sum_b = 0.f;
    uint32_t pa[4][4];  // P as A fragments: k-step kk = keys 16 kk .. 16 kk + 15 = n-tiles 2 kk, 2 kk + 1
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      const float p0 = __expf(sc[n][0] - ref_a), p1 = __expf(sc[n][1] - ref_a), p2 = __expf(sc[n][2] - ref_b), p3 = __expf(sc[n][3] - ref_b);
      sum_a += p0 + p1; sum_b += p2 + p3;
      pa[n >> 1][(n & 1) * 2] = att_pack(p0, p1);
      pa[n >> 1][(n & 1) * 2 + 1] = att_pack(p2, p3);
    }
    sum_a += __shfl_xor_sync(0xffffffffu, sum_a, 1); sum_a += __shfl_xor_sync(0xffffffffu, sum_a, 2);
    sum_b += __shfl_xor_sync(0xffffffffu, sum_b, 1); sum_b += __shfl_xor_sync(0xffffffffu, sum_b, 2);
    l_a = l_a * corr_a + sum_a; l_b = l_b * corr_b + sum_b;
    m_a = mn_a; m_b = mn_b;
    // O = O * corr + P . V: 8 n-tiles of 8 dims, 4 k-steps of 16 keys
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      o[n][0] *= corr_a; o[n][1] *= corr_a; o[n][2] *= corr_b; o[n][3] *= corr_b;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(&Vt[n * 8 + g][kk * 16 + 2 * t]);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(&Vt[n * 8 + g][kk * 16 + 8 + 2 * t]);
        att_mma(o[n], pa[kk][0], pa[kk][1], pa[kk][2], pa[kk][3], b0, b1);
      }
    }
  }
  const int ra = r0 + g, rb = r0 + g + 8;
  const float inv_a = l_a > 0.f ? 1.0f / l_a : 0.f, inv_b = l_b > 0.f ? 1.0f / l_b : 0.f;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    if (ra < T) *reinterpret_cast<uint32_t*>(out + ((size_t)b * T + ra) * ldo + h * 64 + n * 8 + 2 * t) = att_pack(o[n][0] * inv_a, o[n][1] * inv_a);
    if (rb < T) *reinterpret_cast<uint32_t*>(out + ((size_t)b * T + rb) * ldo + h * 64 + n * 8 + 2 * t) = att_pack(o[n][2] * inv_b, o[n][3] * inv_b);
  }
}

void launch_codec_attention_f16(const LaunchCtx& c, const float* qkv, int ld, int B, int T, int nh, int nkv, __half* out, int ldo, bool mma) {
  if (B <= 0 || T <= 0) return;
  if (mma && ld % 4 == 0 && ldo % 2 == 0) {
    dim3 grid((T + 63) / 64, nh, B);
    codec_attention_mma_kernel<<<grid, 128, 0, c.stream>>>(qkv, ld, T, nh, nkv, 1.0f / sqrtf(64.0f), out, ldo, 1);
  } else {
    dim3 grid((T + 15) / 16, nh, B);
    codec_attention_kernel<__half><<<grid, 128, 0, c.stream>>>(qkv, ld, T, nh, nkv, 1.0f / sqrtf(64.0f), out, ldo, 1);
  }
  c.tick();
}

// code -> embedding gather-sum in codebook order, fp32 adds (bit-exact contract).  emb [M][2*D] = [first | rest].
__global__ void rvq_embed_kernel(const int* __restrict__ codes, const float* const* __restrict__ codebooks, int Q, int n_sem, int D,
                                 int size, int M, float* __restrict__ emb) {
  const int m = blockIdx.x;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float first = 0.f, rest = 0.f;
    for (int q = 0; q < Q; ++q) {
      int code = codes[(size_t)m * Q + q];
      code = min(max(code, 0), size - 1);
      const float v = codebooks[q][(size_t)code * D + d];
      if (q < n_sem) first = __fadd_rn(first, v);
      else rest = __fadd_rn(rest, v);
    }
    emb[(size_t)m * 2 * D + d] = first;
    emb[(size_t)m * 2 * D + D + d] = rest;
  }
}
void launch_rvq_embed(const LaunchCtx& c, const int* codes, const float* const* codebooks, int Q, int n_sem, int D, int size, int M,
                      float* emb) {
  if (M <= 0) return;
  rvq_embed_kernel<<<M, 128, 0, c.stream>>>(codes, codebooks, Q, n_sem, D, size, M, emb);
  c.tick();
}

__global__ void rvq_embed_f16_kernel(const int* __restrict__ codes, const float* const* __restrict__ codebooks, int Q, int n_sem, int D,
                                     int size, int M, __half* __restrict__ emb) {
  const int m = blockIdx.x;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float first = 0.f, rest = 0.f;
    for (int q = 0; q < Q; ++q) {
      int code = codes[(size_t)m * Q + q];
      code = min(max(code, 0), size - 1);
      const float v = codebooks[q][(size_t)code * D + d];
      if (q < n_sem) first = __fadd_rn(first, v);
      else rest = __fadd_rn(rest, v);
    }
    emb[(size_t)m * 2 * D + d] = __float2half_rn(first);
    emb[(size_t)m * 2 * D + D + d] = __float2half_rn(rest);
  }
}
void launch_rvq_embed_f16(const LaunchCtx& c, const int* codes, const float* const* codebooks, int Q, int n_sem, int D, int size, int M,
                          __half* emb16) {
  if (M <= 0) return;
  rvq_embed_f16_kernel<<<M, 128, 0, c.stream>>>(codes, codebooks, Q, n_sem, D, size, M, emb16);
  c.tick();
}

// DecoderOutputConv (k = 7, C -> 1) + clip(-1, 1) + NaN scrub (SpeechTokenizer.swift:823-840, 951); x is already snake-activated.
template <typename InT>
__global__ void __launch_bounds__(128) out_conv_kernel(const InT* __restrict__ x, const float* __restrict__ w /*[7][C]*/,
                                                       const float* __restrict__ bias, int C, int T, float* __restrict__ y) {
  extern __shared__ float xs[];  // [(128 + 6)][C + 1]  (+1: consecutive threads read consecutive rows)
  const int b = blockIdx.y, t0 = blockIdx.x * 128;
  const InT* xb = x + (size_t)b * T * C;
  const int rows = 134, ldc = C + 1;
  for (int i = threadIdx.x; i < rows * C; i += 128) {
    const int r = i / C, ch = i - r * C;
    const int t = t0 - 6 + r;
    xs[r * ldc + ch] = (t >= 0 && t < T) ? load_in(xb + (size_t)t * C + ch) : 0.f;
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= T) return;
  float acc = bias[0];
  for (int k = 0; k < 7; ++k) {
    const float* xr = xs + (size_t)(threadIdx.x + k) * ldc;
    const float* wr = w + (size_t)k * C;
    for (int ch = 0; ch < C; ++ch) acc = fmaf(xr[ch], wr[ch], acc);
  }
  // clip(-1, 1); a NaN becomes 0 here so the host needs no scrub pass (Qwen3TTSPipeline.swift:565-570: NaN/Inf -> 0 after the clip)
  y[(size_t)b * T + t] = (acc != acc) ? 0.0f : fminf(1.0f, fmaxf(-1.0f, acc));
}
void launch_out_conv(const LaunchCtx& c, const float* x, const float* w, const float* bias, int C, int B, int T, float* y) {
  if (B <= 0 || T <= 0) return;
  dim3 grid((T + 127) / 128, B);
  out_conv_kernel<float><<<grid, 128, (size_t)134 * (C + 1) * sizeof(float), c.stream>>>(x, w, bias, C, T, y);
  c.tick();
}
void launch_out_conv_f16(const LaunchCtx& c, const __half* x, const float* w, const float* bias, int C, int B, int T, float* y) {
  if (B <= 0 || T <= 0) return;
  dim3 grid((T + 127) / 128, B);
  out_conv_kernel<__half><<<grid, 128, (size_t)134 * (C + 1) * sizeof(float), c.stream>>>(x, w, bias, C, T, y);
  c.tick();
}

// DecoderOutputConv as a STREAMING kernel (Vocoder/SpeechTokenizer.swift:823-840: causal 7-tap conv, C -> 1 channel, then the clip of
// decodeImpl :927).  HBM-bound: every activation byte is needed once (B*T*C fp16 in, B*T fp32 out; 672 MACs per output are nothing).
// A warp walks a strip of consecutive time steps; lane l holds the 7 x CPL weights of channels l, l + 32, ... in registers and a
// sliding window of 7 partial sums: input row r adds x[r] . w[6 - j] to output r + j, so each row is read exactly once -- straight
// from global memory, 64 contiguous bytes per load instruction, no shared memory -- and completes output r, which is reduced across
// the lanes by shuffles and stored 32 outputs at a time.  Through the tensor-core GEMM (31 of 32 output columns zero padding) the
// same conv ran at 17 % of the HBM roofline.
template <int CPL>
__global__ void __launch_bounds__(128) out_conv_stream_kernel(const __half* __restrict__ x, const float* __restrict__ w /*[7][C]*/,
                                                              const float* __restrict__ bias, int T, int strip, int strips_per_b, int n_warps,
                                                              float* __restrict__ y) {
  constexpr int C = CPL * 32;
  const int wid = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (wid >= n_warps) return;
  const int b = wid / strips_per_b, t0 = (wid - b * strips_per_b) * strip;
  const int t1 = t0 + strip < T ? t0 + strip : T;
  const __half* xb = x + (size_t)b * T * C;
  float wr[7][CPL];
#pragma unroll
  for (int k = 0; k < 7; ++k)
#pragma unroll
    for (int j = 0; j < CPL; ++j) wr[k][j] = w[k * C + j * 32 + lane];
  const float b0 = bias[0];
  float acc[7];
#pragma unroll
  for (int j = 0; j < 7; ++j) acc[j] = 0.f;
  float keep = 0.f;
  const int r0 = t0 - 6 > 0 ? t0 - 6 : 0;  // rows before 0 are the causal zero padding
  // rows in chunks of 7, the next chunk's loads issued before the current chunk's arithmetic: 14 rows x 64 B per load in flight per warp
  // (a row-at-a-time loop leaves one row in flight: the shuffles and the guarded store keep the compiler from hoisting the loads)
  constexpr int R = 7;  // = the window depth: after unrolling, the rotation of the 7 partial sums is a renaming, not 6 moves per row
  __half cur[R][CPL], nxt[R][CPL];
  auto fetch = [&](__half (&dst)[R][CPL], int r) {
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int rr = r + i < T ? r + i : T - 1;  // clamped: rows past the strip only feed outputs that are never stored
#pragma unroll
      for (int j = 0; j < CPL; ++j) dst[i][j] = xb[(size_t)rr * C + j * 32 + lane];
    }
  };
  fetch(cur, r0);
  for (int r = r0; r < t1; r += R) {
    if (r + R < t1) fetch(nxt, r + R);
#pragma unroll
    for (int i = 0; i < R; ++i) {
      float xv[CPL];
#pragma unroll
      for (int c = 0; c < CPL; ++c) xv[c] = __half2float(cur[i][c]);
#pragma unroll
      for (int j = 0; j < 7; ++j)
#pragma unroll
        for (int c = 0; c < CPL; ++c) acc[j] = fmaf(xv[c], wr[6 - j][c], acc[j]);
      float v = acc[0];  // output r + i is complete: rows r + i - 6 .. r + i have been added
#pragma unroll
      for (int j = 0; j < 6; ++j) acc[j] = acc[j + 1];
      acc[6] = 0.f;
      const int ro = r + i;
      if (ro >= t0 && ro < t1) {  // warp-uniform
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        v += b0;
        // clip(-1, 1); a NaN becomes 0 here so the host needs no scrub pass (Qwen3TTSPipeline.swift:565-570: NaN/Inf -> 0 after the clip)
        v = (v != v) ? 0.0f : fminf(1.0f, fmaxf(-1.0f, v));
        const int idx = ro - t0;
        if ((idx & 31) == lane) keep = v;
        if ((idx & 31) == 31 || ro == t1 - 1) {
          const int base = t0 + (idx & ~31);
          if (base + lane <= ro) y[(size_t)b * T + base + lane] = keep;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
      for (int j = 0; j < CPL; ++j) cur[i][j] = nxt[i][j];
  }
}
bool out_conv_stream_supported(int C) { return C == 32 || C == 64 || C == 96 || C == 128; }
void launch_out_conv_stream_f16(const LaunchCtx& c, const __half* x, const float* w, const float* bias, int C, int B, int T, float* y, int strip_rows) {
  if (B <= 0 || T <= 0) return;
  const int strip = strip_rows >= 32 ? (strip_rows & ~31) : 256;  // multiple of 32 (outputs are stored 32 at a time); ~3 waves of warps at B x T = 64 x 49 920
  const int strips = (T + strip - 1) / strip, n_warps = B * strips;
  const unsigned blocks = (unsigned)((n_warps + 3) / 4);
  switch (C / 32) {
    case 1: out_conv_stream_kernel<1><<<blocks, 128, 0, c.stream>>>(x, w, bias, T, strip, strips, n_warps, y); break;
    case 2: out_conv_stream_kernel<2><<<blocks, 128, 0, c.stream>>>(x, w, bias, T, strip, strips, n_warps, y); break;
    case 3: out_conv_stream_kernel<3><<<blocks, 128, 0, c.stream>>>(x, w, bias, T, strip, strips, n_warps, y); break;
    default: out_conv_stream_kernel<4><<<blocks, 128, 0, c.stream>>>(x, w, bias, T, strip, strips, n_warps, y); break;
  }
  c.tick();
}

void init_codec_kernels() {
  Q3_CUDA(cudaFuncSetAttribute(out_conv_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  Q3_CUDA(cudaFuncSetAttribute(out_conv_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
}

// ---------------------------------------------------------------------------------------------- ICL audio encoder pieces
// ELUActivation (Vocoder/Qwen3TTSAudioEncoder.swift:8-20): max(x, 0) + min(alpha * (exp(x) - 1), 0), alpha = 1
__global__ void elu_kernel(const float* __restrict__ x, size_t total, float* __restrict__ y) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    y[i] = fmaxf(v, 0.f) + fminf(expf(v) - 1.0f, 0.f);
  }
}
void launch_elu(const LaunchCtx& c, const float* x, size_t total, float* y) {
  if (total == 0) return;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 32);
  elu_kernel<<<blocks, 256, 0, c.stream>>>(x, total, y);
  c.tick();
}

// EncoderSplitResidualVectorQuantizer.encode (:424-460) for one frame per CTA: the semantic chain (layers [0, n_sem)) starts from
// lat_sem[t], the acoustic chain (layers [n_sem, n_out)) from lat_ac[t]; per layer the nearest codeword by
// (|x|^2 - 2 x.e) + |e|^2 (EuclideanCodebook.encode, Vocoder/SpeechTokenizer.swift:511-519; first index on ties), then
// residual -= e[idx] (:408-412).  A warp owns codewords w, w + 8, ...: lanes stride the D dims of a row (coalesced), shuffle reduce.
__global__ void __launch_bounds__(256) rvq_encode_kernel(const float* __restrict__ lat_sem, const float* __restrict__ lat_ac,
                                                         const float* const* __restrict__ books, const float* const* __restrict__ books_sq, int n_sem,
                                                         int n_out, int D, int size, int T, int* __restrict__ codes) {
  extern __shared__ float rvq_sm[];
  float* res = rvq_sm;  // [D]
  __shared__ float red[8];
  __shared__ float best_d[8];
  __shared__ int best_i[8];
  __shared__ int chosen;
  const int t = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int q = 0; q < n_out; ++q) {
    if (q == 0 || q == n_sem) {  // start of a chain: its own projection of the frame
      const float* src = (q < n_sem ? lat_sem : lat_ac) + (size_t)t * D;
      __syncthreads();
      for (int d = tid; d < D; d += 256) res[d] = src[d];
      __syncthreads();
    }
    float ss = 0.f;
    for (int d = tid; d < D; d += 256) ss = fmaf(res[d], res[d], ss);
    ss = warp_sum_c(ss);
    if (lane == 0) red[warp] = ss;
    __syncthreads();
    float xsq = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) xsq += red[w];
    const float* E = books[q];
    const float* Esq = books_sq[q];
    float bd = INFINITY;
    int bi = 0x7fffffff;
    for (int cidx = warp; cidx < size; cidx += 8) {
      const float* e = E + (size_t)cidx * D;
      float dot = 0.f;
      for (int d = lane; d < D; d += 32) dot = fmaf(res[d], e[d], dot);
      dot = warp_sum_c(dot);
      const float dist = (xsq - 2.0f * dot) + Esq[cidx];
      if (dist < bd) { bd = dist; bi = cidx; }  // ascending cidx inside a warp: strict < keeps the first minimum
    }
    if (lane == 0) { best_d[warp] = bd; best_i[warp] = bi; }
    __syncthreads();
    if (tid == 0) {
      float d0 = best_d[0];
      int i0 = best_i[0];
      for (int w = 1; w < 8; ++w)
        if (best_d[w] < d0 || (best_d[w] == d0 && best_i[w] < i0)) { d0 = best_d[w]; i0 = best_i[w]; }
      if (i0 < 0 || i0 >= size) i0 = 0;  // all-NaN distances: keep the walk in bounds
      chosen = i0;
      codes[(size_t)q * T + t] = i0;
    }
    __syncthreads();
    const float* e = E + (size_t)chosen * D;
    for (int d = tid; d < D; d += 256) res[d] -= e[d];
    __syncthreads();
  }
}
void launch_rvq_encode(const LaunchCtx& c, const float* lat_sem, const float* lat_ac, const float* const* books, const float* const* books_sq, int n_sem,
                       int n_out, int D, int size, int T, int* codes) {
  if (T <= 0) return;
  rvq_encode_kernel<<<T, 256, sizeof(float) * D, c.stream>>>(lat_sem, lat_ac, books, books_sq, n_sem, n_out, D, size, T, codes);
  c.tick();
}

}  // namespace q3
