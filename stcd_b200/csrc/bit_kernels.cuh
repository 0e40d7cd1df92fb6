// K12: BIT's token path (models/networks.py:359-394,414-428; blocks in models/help_funcs.py) on a 32-channel bf16 feature
// map [img][4][h*w][8], fp32 arithmetic.
//
//   bit_tokenizer_kernel   one CTA per image: tokens[l] = sum_n softmax_n(conv_a(x))[l, n] x[n]  (online softmax, one read)
//   bit_token_mixer_kernel one CTA per pair: + learned positions, the transformer encoder over the pair's 2L tokens
//   bit_coef_kernel        one CTA per (pair, decoder layer): the collapsed cross-attention matrices of both streams
//                            A[c][(h, j)]  = scale * sum_d Wq[h*dh + d][c] * k[j][h*dh + d]       k = Wk LN(m)
//                            Bm[(h, j)][c] =         sum_d Wout[c][h*dh + d] * v[j][h*dh + d]     v = Wv LN(m)   (Wout packed transposed)
//                          so that softmax_j(q_h . k_hj * scale) v_hj Wout^T == softmax_groups(LN(x) A) Bm.
//   bit_decoder_kernel     one thread per pixel, its 32 channels in registers through every decoder layer:
//                          x += softmax_groups(LN(x) A) Bm + bout;  x += W2 gelu(W1 LN(x) + b1) + b2
// C = 32 channels, L = 4 tokens, 8 heads (heads * L = 32 scores per pixel), mlp = 64: the only configuration the reference
// registers (models/networks.py:174-182); the host checks it.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "transformer_kernels.cuh"

namespace stcd {

constexpr int kBitC = 32, kBitL = 4, kBitHeads = 8, kBitMlp = 64, kBitHJ = kBitHeads * kBitL;
constexpr int kBitCoef = 2 * kBitC * kBitHJ;   // floats per (image, decoder layer): A | Bm

__host__ __device__ constexpr int bit_enc_size(int inner) {
  return 2 * kBitC + 3 * inner * kBitC + kBitC * inner + kBitC + 2 * kBitC + kBitMlp * kBitC + kBitMlp + kBitC * kBitMlp + kBitC;
}
__host__ __device__ constexpr int bit_dec_size(int inner) {
  return 2 * kBitC + 3 * inner * kBitC + kBitC * inner + kBitC + 2 * kBitC + kBitC * kBitMlp + kBitMlp + kBitMlp * kBitC + kBitC;
}
// offset of the per-pixel part of a decoder layer (bout | ln2_g | ln2_b | w1t | b1 | w2t | b2) and its length
__host__ __device__ constexpr int bit_dec_tail_off(int inner) { return 2 * kBitC + 3 * inner * kBitC + kBitC * inner; }
constexpr int kBitDecTail = kBitC + 2 * kBitC + kBitC * kBitMlp + kBitMlp + kBitMlp * kBitC + kBitC;

__device__ __forceinline__ float bit_gelu(float x) { return gelu_fast(x); }

// ------------------------------------------------------------------------------------------ tokenizer
// grid = images, 256 threads.  State per thread and token: running max m, sum s, weighted channel sums acc[32].
// SPLIT: src holds hi + lo planes (lo at src_c8/2 groups), read as hi + lo; the token path is fp32 either way.
template <bool SPLIT>
__global__ void __launch_bounds__(256) bit_tokenizer_kernel(const __nv_bfloat16* __restrict__ src, const float* __restrict__ conv_a,
                                                            float* __restrict__ tokens, int src_c8, int hw) {
  __shared__ float s_wa[kBitL * kBitC];
  __shared__ float s_m[8][kBitL], s_s[8][kBitL], s_acc[8][kBitL][kBitC];
  const int img = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < kBitL * kBitC) s_wa[threadIdx.x] = conv_a[threadIdx.x];
  __syncthreads();
  float m[kBitL], s[kBitL], acc[kBitL][kBitC];
#pragma unroll
  for (int l = 0; l < kBitL; ++l) {
    m[l] = -1e30f;
    s[l] = 0.f;
#pragma unroll
    for (int c = 0; c < kBitC; ++c) acc[l][c] = 0.f;
  }
  const __nv_bfloat16* base = src + static_cast<size_t>(img) * src_c8 * hw * 8;
  for (int n = threadIdx.x; n < hw; n += blockDim.x) {
    float x[kBitC];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if constexpr (SPLIT) load8_split(base + (static_cast<size_t>(g) * hw + n) * 8, static_cast<size_t>(src_c8 >> 1) * hw * 8, x + 8 * g);
      else unpack8(__ldg(reinterpret_cast<const uint4*>(base + (static_cast<size_t>(g) * hw + n) * 8)), x + 8 * g);
    }
#pragma unroll
    for (int l = 0; l < kBitL; ++l) {
      float a = 0.f;
#pragma unroll
      for (int c = 0; c < kBitC; ++c) a = fmaf(s_wa[l * kBitC + c], x[c], a);
      const float mn = fmaxf(m[l], a);
      const float r = expf(m[l] - mn), e = expf(a - mn);
      s[l] = s[l] * r + e;
#pragma unroll
      for (int c = 0; c < kBitC; ++c) acc[l][c] = fmaf(acc[l][c], r, e * x[c]);
      m[l] = mn;
    }
  }
  // butterfly over the warp (fixed order), then over the 8 warps through shared memory
#pragma unroll
  for (int l = 0; l < kBitL; ++l) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float mo = __shfl_xor_sync(0xffffffffu, m[l], o), so = __shfl_xor_sync(0xffffffffu, s[l], o);
      const float mn = fmaxf(m[l], mo);
      const float r = expf(m[l] - mn), ro = expf(mo - mn);
      s[l] = s[l] * r + so * ro;
#pragma unroll
      for (int c = 0; c < kBitC; ++c) acc[l][c] = acc[l][c] * r + __shfl_xor_sync(0xffffffffu, acc[l][c], o) * ro;
      m[l] = mn;
    }
    if (lane == 0) {
      s_m[warp][l] = m[l];
      s_s[warp][l] = s[l];
    }
#pragma unroll
    for (int c = 0; c < kBitC; ++c)
      if (lane == c) s_acc[warp][l][c] = acc[l][c];
  }
  __syncthreads();
  if (threadIdx.x < kBitL * kBitC) {
    const int l = threadIdx.x / kBitC, c = threadIdx.x % kBitC;
    float M = -1e30f;
    for (int w = 0; w < 8; ++w) M = fmaxf(M, s_m[w][l]);
    float S = 0.f, A = 0.f;
    for (int w = 0; w < 8; ++w) {
      const float r = expf(s_m[w][l] - M);
      S = fmaf(s_s[w][l], r, S);
      A = fmaf(s_acc[w][l][c], r, A);
    }
    tokens[(static_cast<size_t>(img) * kBitL + l) * kBitC + c] = A / S;
  }
}

// ------------------------------------------------------------------------------------------ token mixer
__device__ __forceinline__ void bit_ln_rows(const float* __restrict__ in, float* __restrict__ out, const float* __restrict__ g,
                                            const float* __restrict__ b, int rows) {
  // one warp per row, lane = channel (C = 32)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = warp; r < rows; r += 8) {
    const float v = in[r * kBitC + lane];
    float mean = v;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mean += __shfl_xor_sync(0xffffffffu, mean, o);
    mean *= (1.f / kBitC);
    const float d = v - mean;
    float var = d * d;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
    out[r * kBitC + lane] = d * rsqrtf(var * (1.f / kBitC) + 1e-5f) * __ldg(g + lane) + __ldg(b + lane);
  }
}

// grid = pairs (chunk), 256 threads; dynamic smem: big[8 * 3 * inner_max] floats
__global__ void __launch_bounds__(256) bit_token_mixer_kernel(const float* __restrict__ tokens, const float* __restrict__ pos,
                                                              const float* __restrict__ enc, float* __restrict__ tok_out, int chunk,
                                                              int n_enc, int inner_e, float scale) {
  extern __shared__ float s_big[];                 // qkv [8][3*inner_e]
  __shared__ float s_t[2 * kBitL * kBitC], s_y[2 * kBitL * kBitC], s_attn[kBitHeads][2 * kBitL][2 * kBitL], s_h[2 * kBitL * kBitMlp];
  const int pair = blockIdx.x, tid = threadIdx.x;
  constexpr int R = 2 * kBitL;                      // 8 token rows per pair
  {
    const int r = tid / kBitC, c = tid % kBitC;     // 256 threads == R * C
    const int img = (r < kBitL ? 0 : chunk) + pair;
    s_t[tid] = tokens[(static_cast<size_t>(img) * kBitL + (r % kBitL)) * kBitC + c] + __ldg(pos + tid);
  }
  __syncthreads();
  for (int l = 0; l < n_enc; ++l) {
    const float* P = enc + static_cast<size_t>(l) * bit_enc_size(inner_e);
    const float* ln1_g = P;
    const float* ln1_b = ln1_g + kBitC;
    const float* wqkv = ln1_b + kBitC;
    const float* wout = wqkv + 3 * inner_e * kBitC;
    const float* bout = wout + kBitC * inner_e;
    const float* ln2_g = bout + kBitC;
    const float* ln2_b = ln2_g + kBitC;
    const float* w1 = ln2_b + kBitC;
    const float* b1 = w1 + kBitMlp * kBitC;
    const float* w2 = b1 + kBitMlp;
    const float* b2 = w2 + kBitC * kBitMlp;
    bit_ln_rows(s_t, s_y, ln1_g, ln1_b, R);
    __syncthreads();
    for (int j = tid; j < 3 * inner_e; j += blockDim.x) {       // qkv[r][j] = y[r] . Wqkv[j]
      float w[kBitC];
#pragma unroll
      for (int q = 0; q < kBitC / 4; ++q) {
        const float4 t4 = __ldg(reinterpret_cast<const float4*>(wqkv + static_cast<size_t>(j) * kBitC) + q);
        w[4 * q] = t4.x, w[4 * q + 1] = t4.y, w[4 * q + 2] = t4.z, w[4 * q + 3] = t4.w;
      }
      for (int r = 0; r < R; ++r) {
        float a = 0.f;
#pragma unroll
        for (int c = 0; c < kBitC; ++c) a = fmaf(s_y[r * kBitC + c], w[c], a);
        s_big[r * 3 * inner_e + j] = a;
      }
    }
    __syncthreads();
    const int dh = inner_e / kBitHeads;
    if (tid < kBitHeads * R) {                                  // one (head, query) per thread: 8 scores, softmax
      const int h = tid / R, i = tid % R;
      float d[R], mx = -1e30f;
      for (int j = 0; j < R; ++j) {
        float a = 0.f;
        for (int e = 0; e < dh; ++e) a = fmaf(s_big[i * 3 * inner_e + h * dh + e], s_big[j * 3 * inner_e + inner_e + h * dh + e], a);
        d[j] = a * scale;
        mx = fmaxf(mx, d[j]);
      }
      float sum = 0.f;
      for (int j = 0; j < R; ++j) {
        d[j] = expf(d[j] - mx);
        sum += d[j];
      }
      for (int j = 0; j < R; ++j) s_attn[h][i][j] = d[j] / sum;
    }
    __syncthreads();
    // o[i][col] = sum_j attn[h(col)][i][j] v[j][col], written over q (each (i, col) is read by nobody else after the scores)
    for (int it = tid; it < R * inner_e; it += blockDim.x) {
      const int i = it / inner_e, col = it % inner_e, h = col / dh;
      float a = 0.f;
      for (int j = 0; j < R; ++j) a = fmaf(s_attn[h][i][j], s_big[j * 3 * inner_e + 2 * inner_e + col], a);
      s_big[i * 3 * inner_e + col] = a;
    }
    __syncthreads();
    for (int c = tid >> 5; c < kBitC; c += 8) {                 // warp per output channel: lanes stride over inner (coalesced rows)
      const int lane = tid & 31;
      float a[R];
#pragma unroll
      for (int r = 0; r < R; ++r) a[r] = 0.f;
      for (int j = lane; j < inner_e; j += 32) {
        const float wv_ = __ldg(wout + static_cast<size_t>(c) * inner_e + j);
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] = fmaf(s_big[r * 3 * inner_e + j], wv_, a[r]);
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a[r] += __shfl_xor_sync(0xffffffffu, a[r], o);
        if (lane == 0) s_t[r * kBitC + c] += a[r] + __ldg(bout + c);
      }
    }
    __syncthreads();
    bit_ln_rows(s_t, s_y, ln2_g, ln2_b, R);
    __syncthreads();
    for (int it = tid; it < R * kBitMlp; it += blockDim.x) {
      const int r = it / kBitMlp, k = it % kBitMlp;
      float a = __ldg(b1 + k);
#pragma unroll
      for (int c = 0; c < kBitC; ++c) a = fmaf(s_y[r * kBitC + c], __ldg(w1 + k * kBitC + c), a);
      s_h[it] = bit_gelu(a);
    }
    __syncthreads();
    {
      const int r = tid / kBitC, c = tid % kBitC;
      float a = __ldg(b2 + c);
#pragma unroll
      for (int k = 0; k < kBitMlp; ++k) a = fmaf(s_h[r * kBitMlp + k], __ldg(w2 + c * kBitMlp + k), a);
      s_t[tid] += a;
    }
    __syncthreads();
  }
  tok_out[static_cast<size_t>(pair) * R * kBitC + tid] = s_t[tid];
}

// grid (pairs, decoder layers), 256 threads; dynamic smem: k | v [2][8][inner_d] floats.  The encoder's tokens are the memory
// of every decoder layer (they never change), so the layers' collapsed matrices are independent of each other.
__global__ void __launch_bounds__(256) bit_coef_kernel(const float* __restrict__ tok, const float* __restrict__ dec, float* __restrict__ coef,
                                                       int chunk, int n_dec, int inner_d, float scale) {
  extern __shared__ float s_kv[];
  __shared__ float s_t[2 * kBitL * kBitC], s_y[2 * kBitL * kBitC];
  constexpr int R = 2 * kBitL;
  const int pair = blockIdx.x, l = blockIdx.y, tid = threadIdx.x;
  const int dh = inner_d / kBitHeads;
  s_t[tid] = tok[static_cast<size_t>(pair) * R * kBitC + tid];
  __syncthreads();
  const float* P = dec + static_cast<size_t>(l) * bit_dec_size(inner_d);
  const float* wq = P + 2 * kBitC;
  const float* wk = wq + inner_d * kBitC;
  const float* wv = wk + inner_d * kBitC;
  const float* woutt = wv + inner_d * kBitC;                    // [inner][c]
  bit_ln_rows(s_t, s_y, P, P + kBitC, R);                       // PreNorm2: the layer's norm on the memory too
  __syncthreads();
  float* s_k = s_kv;                                            // [R][inner_d]
  float* s_v = s_kv + R * inner_d;
  for (int j = tid; j < 2 * inner_d; j += blockDim.x) {
    const float* wrow = (j < inner_d ? wk + static_cast<size_t>(j) * kBitC : wv + static_cast<size_t>(j - inner_d) * kBitC);
    float w[kBitC];
#pragma unroll
    for (int q = 0; q < kBitC / 4; ++q) {
      const float4 t4 = __ldg(reinterpret_cast<const float4*>(wrow) + q);
      w[4 * q] = t4.x, w[4 * q + 1] = t4.y, w[4 * q + 2] = t4.z, w[4 * q + 3] = t4.w;
    }
    for (int r = 0; r < R; ++r) {
      float a = 0.f;
#pragma unroll
      for (int c = 0; c < kBitC; ++c) a = fmaf(s_y[r * kBitC + c], w[c], a);
      (j < inner_d ? s_k[r * inner_d + j] : s_v[r * inner_d + j - inner_d]) = a;
    }
  }
  __syncthreads();
  for (int it = tid; it < 2 * kBitC * kBitHJ; it += blockDim.x) {         // (stream, hj, c): lanes vary c, both weight reads coalesce
    const int s = it / (kBitC * kBitHJ), rem = it % (kBitC * kBitHJ);
    const int hj = rem / kBitC, c = rem % kBitC;
    const int h = hj / kBitL, j = hj % kBitL, row = s * kBitL + j;
    float a = 0.f, b = 0.f;
    for (int e = 0; e < dh; ++e) {
      a = fmaf(__ldg(wq + static_cast<size_t>(h * dh + e) * kBitC + c), s_k[row * inner_d + h * dh + e], a);
      b = fmaf(__ldg(woutt + static_cast<size_t>(h * dh + e) * kBitC + c), s_v[row * inner_d + h * dh + e], b);
    }
    float* o = coef + (static_cast<size_t>(s * chunk + pair) * n_dec + l) * kBitCoef;
    o[c * kBitHJ + hj] = a * scale;
    o[kBitC * kBitHJ + hj * kBitC + c] = b;
  }
}

// ------------------------------------------------------------------------------------------ decoder
// Two pixels per thread and packed fp32 FMAs (FFMA2): every broadcast LDS.128 of a weight row feeds 8 FMAs (4 FFMA2), which
// keeps the kernel on the FMA pipe instead of the shared-memory port.
struct BitPx {                     // one pixel's 32 channels as 16 packed pairs
  float2 v[kBitC / 2];
};

__device__ __forceinline__ void bit_ln32(const BitPx& x, float (&y)[kBitC], const float* __restrict__ g, const float* __restrict__ b) {
  float mean = 0.f;
#pragma unroll
  for (int c = 0; c < kBitC / 2; ++c) mean += x.v[c].x + x.v[c].y;
  mean *= (1.f / kBitC);
  float var = 0.f;
#pragma unroll
  for (int c = 0; c < kBitC / 2; ++c) {
    var = fmaf(x.v[c].x - mean, x.v[c].x - mean, var);
    var = fmaf(x.v[c].y - mean, x.v[c].y - mean, var);
  }
  const float rs = rsqrtf(var * (1.f / kBitC) + 1e-5f);
#pragma unroll
  for (int c = 0; c < kBitC / 2; ++c) {
    y[2 * c] = (x.v[c].x - mean) * rs * g[2 * c] + b[2 * c];
    y[2 * c + 1] = (x.v[c].y - mean) * rs * g[2 * c + 1] + b[2 * c + 1];
  }
}

// out{0,1}[32] += in{0,1}[K] . W[K][32 of a row of `stride` floats]  (rows in shared memory, broadcast float4 reads)
template <int K>
__device__ __forceinline__ void bit_matvec2(const float* __restrict__ in0, const float* __restrict__ in1, const float* __restrict__ W,
                                            int stride, BitPx& out0, BitPx& out1) {
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const float2 a0 = make_float2(in0[k], in0[k]), a1 = make_float2(in1[k], in1[k]);
#pragma unroll
    for (int n4 = 0; n4 < kBitC / 4; ++n4) {
      const float4 w = *reinterpret_cast<const float4*>(W + k * stride + 4 * n4);
      const float2 wlo = make_float2(w.x, w.y), whi = make_float2(w.z, w.w);
      out0.v[2 * n4] = __ffma2_rn(a0, wlo, out0.v[2 * n4]);
      out0.v[2 * n4 + 1] = __ffma2_rn(a0, whi, out0.v[2 * n4 + 1]);
      out1.v[2 * n4] = __ffma2_rn(a1, wlo, out1.v[2 * n4]);
      out1.v[2 * n4 + 1] = __ffma2_rn(a1, whi, out1.v[2 * n4 + 1]);
    }
  }
}

__device__ __forceinline__ void bit_softmax_groups(BitPx& d) {       // 8 heads x 4 keys: groups of two packed pairs
#pragma unroll
  for (int h = 0; h < kBitHeads; ++h) {
    float2& p = d.v[2 * h];
    float2& q = d.v[2 * h + 1];
    const float mx = fmaxf(fmaxf(p.x, p.y), fmaxf(q.x, q.y));
    p.x = __expf(p.x - mx), p.y = __expf(p.y - mx), q.x = __expf(q.x - mx), q.y = __expf(q.y - mx);
    const float inv = 1.f / (p.x + p.y + q.x + q.y);
    p.x *= inv, p.y *= inv, q.x *= inv, q.y *= inv;
  }
}

constexpr int kBitDecThreads = 128;

// grid (pixel blocks of 2 * kBitDecThreads, images)
// SPLIT: src and dst hold hi + lo planes (lo at half the stored channel groups): the map is read as hi + lo and written as
// hi = bf16(x), lo = bf16(x - hi).
template <bool SPLIT>
__global__ void __launch_bounds__(kBitDecThreads) bit_decoder_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                                     const float* __restrict__ dec, const float* __restrict__ coef,
                                                                     int src_c8, int dst_c8, int hw, int n_dec, int inner_d, int softmax) {
  __shared__ __align__(16) float s_ln1[2 * kBitC];
  __shared__ __align__(16) float s_coef[kBitCoef];
  __shared__ __align__(16) float s_tail[kBitDecTail];
  const int img = blockIdx.y;
  const int pix0 = blockIdx.x * (2 * kBitDecThreads) + threadIdx.x, pix1 = pix0 + kBitDecThreads;
  BitPx x0, x1;
  {
    const __nv_bfloat16* b = src + static_cast<size_t>(img) * src_c8 * hw * 8;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float t[8];
      if (pix0 < hw) {
        if constexpr (SPLIT) load8_split(b + (static_cast<size_t>(g) * hw + pix0) * 8, static_cast<size_t>(src_c8 >> 1) * hw * 8, t);
        else unpack8(__ldg(reinterpret_cast<const uint4*>(b + (static_cast<size_t>(g) * hw + pix0) * 8)), t);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) x0.v[4 * g + j] = make_float2(t[2 * j], t[2 * j + 1]);
      if (pix1 < hw) {
        if constexpr (SPLIT) load8_split(b + (static_cast<size_t>(g) * hw + pix1) * 8, static_cast<size_t>(src_c8 >> 1) * hw * 8, t);
        else unpack8(__ldg(reinterpret_cast<const uint4*>(b + (static_cast<size_t>(g) * hw + pix1) * 8)), t);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) x1.v[4 * g + j] = make_float2(t[2 * j], t[2 * j + 1]);
    }
  }
  for (int l = 0; l < n_dec; ++l) {
    const float* P = dec + static_cast<size_t>(l) * bit_dec_size(inner_d);
    const float* cf = coef + (static_cast<size_t>(img) * n_dec + l) * kBitCoef;
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * kBitC; i += blockDim.x) s_ln1[i] = __ldg(P + i);
    for (int i = threadIdx.x; i < kBitCoef / 4; i += blockDim.x)
      reinterpret_cast<float4*>(s_coef)[i] = __ldg(reinterpret_cast<const float4*>(cf) + i);
    for (int i = threadIdx.x; i < kBitDecTail / 4; i += blockDim.x)
      reinterpret_cast<float4*>(s_tail)[i] = __ldg(reinterpret_cast<const float4*>(P + bit_dec_tail_off(inner_d)) + i);
    __syncthreads();
    const float* bout = s_tail;
    const float* ln2_g = bout + kBitC;
    const float* ln2_b = ln2_g + kBitC;
    const float* w1t = ln2_b + kBitC;
    const float* b1 = w1t + kBitC * kBitMlp;
    const float* w2t = b1 + kBitMlp;
    const float* b2 = w2t + kBitMlp * kBitC;
    float y0[kBitC], y1[kBitC];
    bit_ln32(x0, y0, s_ln1, s_ln1 + kBitC);
    bit_ln32(x1, y1, s_ln1, s_ln1 + kBitC);
    {
      BitPx d0, d1;
#pragma unroll
      for (int i = 0; i < kBitC / 2; ++i) d0.v[i] = d1.v[i] = make_float2(0.f, 0.f);
      bit_matvec2<kBitC>(y0, y1, s_coef, kBitHJ, d0, d1);
      if (softmax) {
        bit_softmax_groups(d0);
        bit_softmax_groups(d1);
      }
#pragma unroll
      for (int c = 0; c < kBitC / 2; ++c) {
        const float2 bb = make_float2(bout[2 * c], bout[2 * c + 1]);
        x0.v[c].x += bb.x, x0.v[c].y += bb.y, x1.v[c].x += bb.x, x1.v[c].y += bb.y;
      }
      bit_matvec2<kBitHJ>(reinterpret_cast<const float*>(d0.v), reinterpret_cast<const float*>(d1.v), s_coef + kBitC * kBitHJ, kBitC, x0, x1);
    }
    bit_ln32(x0, y0, ln2_g, ln2_b);
    bit_ln32(x1, y1, ln2_g, ln2_b);
#pragma unroll
    for (int c = 0; c < kBitC / 2; ++c) {
      const float2 bb = make_float2(b2[2 * c], b2[2 * c + 1]);
      x0.v[c].x += bb.x, x0.v[c].y += bb.y, x1.v[c].x += bb.x, x1.v[c].y += bb.y;
    }
#pragma unroll 1
    for (int half = 0; half < kBitMlp / kBitC; ++half) {        // hidden units 32 at a time: bounds the live registers
      BitPx h0, h1;
#pragma unroll
      for (int k = 0; k < kBitC / 2; ++k) h0.v[k] = h1.v[k] = make_float2(b1[half * kBitC + 2 * k], b1[half * kBitC + 2 * k + 1]);
      bit_matvec2<kBitC>(y0, y1, w1t + half * kBitC, kBitMlp, h0, h1);
#pragma unroll
      for (int k = 0; k < kBitC / 2; ++k) {
        h0.v[k] = gelu_fast2(h0.v[k]);
        h1.v[k] = gelu_fast2(h1.v[k]);
      }
      bit_matvec2<kBitC>(reinterpret_cast<const float*>(h0.v), reinterpret_cast<const float*>(h1.v), w2t + half * kBitC * kBitC, kBitC, x0, x1);
    }
  }
  __nv_bfloat16* o = dst + static_cast<size_t>(img) * dst_c8 * hw * 8;
  if constexpr (SPLIT) {
    const size_t lo_off = static_cast<size_t>(dst_c8 >> 1) * hw * 8;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      uint4 qh, ql;
      if (pix0 < hw) {
        split8(reinterpret_cast<const float*>(x0.v + 4 * g), qh, ql);
        *reinterpret_cast<uint4*>(o + (static_cast<size_t>(g) * hw + pix0) * 8) = qh;
        *reinterpret_cast<uint4*>(o + (static_cast<size_t>(g) * hw + pix0) * 8 + lo_off) = ql;
      }
      if (pix1 < hw) {
        split8(reinterpret_cast<const float*>(x1.v + 4 * g), qh, ql);
        *reinterpret_cast<uint4*>(o + (static_cast<size_t>(g) * hw + pix1) * 8) = qh;
        *reinterpret_cast<uint4*>(o + (static_cast<size_t>(g) * hw + pix1) * 8 + lo_off) = ql;
      }
    }
    return;
  }
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    if (pix0 < hw) *reinterpret_cast<uint4*>(o + (static_cast<size_t>(g) * hw + pix0) * 8) = pack8(reinterpret_cast<const float*>(x0.v + 4 * g));
    if (pix1 < hw) *reinterpret_cast<uint4*>(o + (static_cast<size_t>(g) * hw + pix1) * 8) = pack8(reinterpret_cast<const float*>(x1.v + 4 * g));
  }
}

}  // namespace stcd
