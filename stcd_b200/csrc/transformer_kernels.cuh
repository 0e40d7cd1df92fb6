// MiT / ChangeFormer encoder ops that are not convolutions (models/ChangeFormer.py): LayerNorm over channels,
// spatial-reduction attention, depth-wise 3x3 + GELU.  All on bf16 [img][c/8][h*w][8] plan tensors, fp32 arithmetic.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

namespace stcd {

__device__ __forceinline__ void unpack8(uint4 q, float* v) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
    v[2 * j] = __low2float(h);
    v[2 * j + 1] = __high2float(h);
  }
}
__device__ __forceinline__ uint4 pack8(const float* v) {
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    w[j] = *reinterpret_cast<uint32_t*>(&h);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// Split precision (lowering.Program.precision "split"): a value is hi + lo, hi in channel groups [0, c8/2) of the tensor, lo in
// [c8/2, c8).  load8_split reads both planes as fp32 sums; split8 writes hi = bf16(v), lo = bf16(v - hi).
__device__ __forceinline__ void load8_split(const __nv_bfloat16* p, size_t lo_off, float* v) {
  float l[8];
  unpack8(__ldg(reinterpret_cast<const uint4*>(p)), v);
  unpack8(__ldg(reinterpret_cast<const uint4*>(p + lo_off)), l);
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] += l[j];
}
__device__ __forceinline__ void split8(const float* v, uint4& hi, uint4& lo) {
  float h[8], r[8];
  hi = pack8(v);
  unpack8(hi, h);
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = v[j] - h[j];
  lo = pack8(r);
}

// nn.LayerNorm(C, eps) per pixel: y = (x - mean) / sqrt(var + eps) * gamma + beta, biased variance, fp32 statistics
// (two passes over the pixel's C channels: mean, then centred sum of squares; the second and third reads hit L1/L2).
// A warp covers 8 consecutive pixels x 4 channel slices (lane = slice * 8 + pixel): every load is a 128-byte row of one channel
// group, a lane walks every fourth group and the four partial sums meet in two butterfly steps (fixed order).  One thread per pixel
// walked 64 groups three times at the coarse MiT stages (33 us for 8 MB); this is 4x shorter and has 4x the threads.
// Optionally also writes the space-to-depth copy dst2 ([h/2][w/2] pixels, channel block (y%2)*2 + x%2).
// HBM-bound: 2 B read + 2 (or 4) B written per element.
// SPLIT: src, dst and dst2 hold hi and lo planes (lowering.Program.precision); the statistics run over hi + lo and both planes are
// written (dst2's lo plane of class k, channel ch sits at channel 4C + k*C + ch).
template <bool SPLIT>
__global__ void __launch_bounds__(256) layernorm_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                        __nv_bfloat16* __restrict__ dst2, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, int B, int C, int src_c8, int dst_c8,
                                                        int dst2_c8, int h, int w, float eps) {
  const int hw = h * w, g8 = C >> 3;
  const size_t total = static_cast<size_t>(B) * hw;
  const int lane = threadIdx.x & 31, slice = lane >> 3;
  const size_t warps = (static_cast<size_t>(gridDim.x) * blockDim.x) >> 5;
  for (size_t wi = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5; wi * 8 < total; wi += warps) {
    const size_t i_raw = wi * 8 + (lane & 7);
    const bool live = i_raw < total;
    const size_t i = live ? i_raw : total - 1;             // clamped: idle lanes still take part in the shuffles
    const size_t b = i / hw;
    const int pix = static_cast<int>(i - b * hw);
    const __nv_bfloat16* s = src + (b * src_c8 * hw + pix) * 8;
    const size_t s_lo = static_cast<size_t>(src_c8 >> 1) * hw * 8;        // split: offset of the lo plane
    float sum = 0.f;
    for (int g = slice; g < g8; g += 4) {
      float v[8];
      if constexpr (SPLIT) load8_split(s + static_cast<size_t>(g) * hw * 8, s_lo, v);
      else unpack8(__ldg(reinterpret_cast<const uint4*>(s + static_cast<size_t>(g) * hw * 8)), v);
#pragma unroll
      for (int j = 0; j < 8; ++j) sum += v[j];
    }
    sum += __shfl_xor_sync(0xffffffffu, sum, 8);
    sum += __shfl_xor_sync(0xffffffffu, sum, 16);
    const float mean = sum / static_cast<float>(C);
    float sq = 0.f;
    for (int g = slice; g < g8; g += 4) {
      float v[8];
      if constexpr (SPLIT) load8_split(s + static_cast<size_t>(g) * hw * 8, s_lo, v);
      else unpack8(__ldg(reinterpret_cast<const uint4*>(s + static_cast<size_t>(g) * hw * 8)), v);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = v[j] - mean;
        sq = fmaf(d, d, sq);
      }
    }
    sq += __shfl_xor_sync(0xffffffffu, sq, 8);
    sq += __shfl_xor_sync(0xffffffffu, sq, 16);
    const float rstd = rsqrtf(sq / static_cast<float>(C) + eps);
    __nv_bfloat16* o = dst + (b * dst_c8 * hw + pix) * 8;
    __nv_bfloat16* o2 = nullptr;
    size_t hw2 = 0;
    if (dst2 != nullptr) {
      const int y = pix / w, x = pix - y * w;
      hw2 = static_cast<size_t>(hw >> 2);
      o2 = dst2 + ((b * dst2_c8 + static_cast<size_t>(((y & 1) * 2 + (x & 1)) * g8)) * hw2 + static_cast<size_t>(y >> 1) * (w >> 1) + (x >> 1)) * 8;
    }
    if (!live) continue;
    for (int g = slice; g < g8; g += 4) {
      float v[8];
      if constexpr (SPLIT) load8_split(s + static_cast<size_t>(g) * hw * 8, s_lo, v);
      else unpack8(__ldg(reinterpret_cast<const uint4*>(s + static_cast<size_t>(g) * hw * 8)), v);
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + g * 8)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + g * 8 + 4));
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + g * 8)), b1 = __ldg(reinterpret_cast<const float4*>(beta + g * 8 + 4));
      const float gm[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float bt[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf((v[j] - mean) * rstd, gm[j], bt[j]);
      if constexpr (SPLIT) {
        uint4 qh, ql;
        split8(v, qh, ql);
        *reinterpret_cast<uint4*>(o + static_cast<size_t>(g) * hw * 8) = qh;
        *reinterpret_cast<uint4*>(o + (static_cast<size_t>(g) + (dst_c8 >> 1)) * hw * 8) = ql;
        if (o2 != nullptr) {
          *reinterpret_cast<uint4*>(o2 + static_cast<size_t>(g) * hw2 * 8) = qh;
          *reinterpret_cast<uint4*>(o2 + (static_cast<size_t>(g) + (dst2_c8 >> 1)) * hw2 * 8) = ql;
        }
      } else {
        const uint4 q = pack8(v);
        *reinterpret_cast<uint4*>(o + static_cast<size_t>(g) * hw * 8) = q;
        if (o2 != nullptr) *reinterpret_cast<uint4*>(o2 + static_cast<size_t>(g) * hw2 * 8) = q;
      }
    }
  }
}

// Spatial-reduction attention (ChangeFormer.py:338-358): out[n] = softmax_j(q[n].k[j] * scale) v[j] per head, NK <= 64
// keys.  grid (ceil(N / 256), heads, B), 128 threads = 256 queries; the head's K and V (fp32, [NK][D]) sit in shared
// memory and every lane reads the same address (broadcast).  q streams through registers 8 channels at a time, the 64
// scores stay in registers; the [N, NK] score matrix never exists in memory.
constexpr int kAttnMaxKeys = 64;
template <int D>   // head dim: 64 or 80
__global__ void __launch_bounds__(128) sr_attention_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ kv,
                                                           __nv_bfloat16* __restrict__ out, int C, int q_c8, int kv_c8,
                                                           int out_c8, int N, int NK, float scale) {
  __shared__ __align__(16) float sk[kAttnMaxKeys][D];
  __shared__ __align__(16) float sv[kAttnMaxKeys][D];
  const int b = blockIdx.z, hd = blockIdx.y;
  const int g0 = hd * (D / 8);                 // first channel group of this head inside q / k; v sits C/8 groups later
  // consecutive lanes take consecutive channel groups of one key: the two STS.128 per operand are bank-conflict free (the
  // transposed order -- consecutive keys, 256-byte stride -- serialised every store 32 ways and cost as much as the math)
  for (int i = threadIdx.x; i < NK * (D / 8); i += blockDim.x) {
    const int g = i % (D / 8), j = i / (D / 8);
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(kv + ((static_cast<size_t>(b) * kv_c8 + g0 + g) * NK + j) * 8)), v);
    *reinterpret_cast<float4*>(&sk[j][g * 8]) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(&sk[j][g * 8 + 4]) = make_float4(v[4], v[5], v[6], v[7]);
    unpack8(__ldg(reinterpret_cast<const uint4*>(kv + ((static_cast<size_t>(b) * kv_c8 + (C >> 3) + g0 + g) * NK + j) * 8)), v);
    *reinterpret_cast<float4*>(&sv[j][g * 8]) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(&sv[j][g * 8 + 4]) = make_float4(v[4], v[5], v[6], v[7]);
  }
  __syncthreads();
  // two queries per thread (n0, n0 + 128), scores packed as (query 0, query 1) pairs: every broadcast LDS.128 of K / V feeds
  // 8 FMAs as 4 FFMA2.  Each FFMA2 lane is an IEEE fma and the summation orders (channels, then keys) are the scalar ones.
  const int n0 = blockIdx.x * (2 * blockDim.x) + threadIdx.x, n1 = n0 + blockDim.x;
  if (n0 >= N) return;
  const bool two = n1 < N;
  float2 s[kAttnMaxKeys];
#pragma unroll
  for (int j = 0; j < kAttnMaxKeys; ++j) s[j] = make_float2(0.f, 0.f);
  for (int g = 0; g < D / 8; ++g) {
    float qa[8], qb[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(q + ((static_cast<size_t>(b) * q_c8 + g0 + g) * N + n0) * 8)), qa);
    unpack8(__ldg(reinterpret_cast<const uint4*>(q + ((static_cast<size_t>(b) * q_c8 + g0 + g) * N + (two ? n1 : n0)) * 8)), qb);
    float2 qq[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) qq[e] = make_float2(qa[e], qb[e]);
#pragma unroll
    for (int j = 0; j < kAttnMaxKeys; ++j) {
      if (j < NK) {
        const float4 k0 = *reinterpret_cast<const float4*>(&sk[j][g * 8]), k1 = *reinterpret_cast<const float4*>(&sk[j][g * 8 + 4]);
        s[j] = __ffma2_rn(qq[0], make_float2(k0.x, k0.x), s[j]);
        s[j] = __ffma2_rn(qq[1], make_float2(k0.y, k0.y), s[j]);
        s[j] = __ffma2_rn(qq[2], make_float2(k0.z, k0.z), s[j]);
        s[j] = __ffma2_rn(qq[3], make_float2(k0.w, k0.w), s[j]);
        s[j] = __ffma2_rn(qq[4], make_float2(k1.x, k1.x), s[j]);
        s[j] = __ffma2_rn(qq[5], make_float2(k1.y, k1.y), s[j]);
        s[j] = __ffma2_rn(qq[6], make_float2(k1.z, k1.z), s[j]);
        s[j] = __ffma2_rn(qq[7], make_float2(k1.w, k1.w), s[j]);
      }
    }
  }
  float mx0 = -CUDART_INF_F, mx1 = -CUDART_INF_F;
#pragma unroll
  for (int j = 0; j < kAttnMaxKeys; ++j)
    if (j < NK) {
      s[j].x *= scale, s[j].y *= scale;
      mx0 = fmaxf(mx0, s[j].x), mx1 = fmaxf(mx1, s[j].y);
    }
  float den0 = 0.f, den1 = 0.f;
#pragma unroll
  for (int j = 0; j < kAttnMaxKeys; ++j) {
    s[j].x = (j < NK) ? expf(s[j].x - mx0) : 0.f;
    s[j].y = (j < NK) ? expf(s[j].y - mx1) : 0.f;
    den0 += s[j].x, den1 += s[j].y;
  }
  const float inv0 = 1.f / den0, inv1 = 1.f / den1;
  for (int g = 0; g < D / 8; ++g) {
    float2 oa[4], ob[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) oa[e] = ob[e] = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < kAttnMaxKeys; ++j) {
      if (j < NK) {
        const float4 v0 = *reinterpret_cast<const float4*>(&sv[j][g * 8]), v1 = *reinterpret_cast<const float4*>(&sv[j][g * 8 + 4]);
        const float2 p0 = make_float2(s[j].x, s[j].x), p1 = make_float2(s[j].y, s[j].y);
        const float2 va = make_float2(v0.x, v0.y), vb = make_float2(v0.z, v0.w), vc = make_float2(v1.x, v1.y), vd = make_float2(v1.z, v1.w);
        oa[0] = __ffma2_rn(p0, va, oa[0]), oa[1] = __ffma2_rn(p0, vb, oa[1]), oa[2] = __ffma2_rn(p0, vc, oa[2]), oa[3] = __ffma2_rn(p0, vd, oa[3]);
        ob[0] = __ffma2_rn(p1, va, ob[0]), ob[1] = __ffma2_rn(p1, vb, ob[1]), ob[2] = __ffma2_rn(p1, vc, ob[2]), ob[3] = __ffma2_rn(p1, vd, ob[3]);
      }
    }
    float o[8];
#pragma unroll
    for (int e = 0; e < 4; ++e) o[2 * e] = oa[e].x * inv0, o[2 * e + 1] = oa[e].y * inv0;
    *reinterpret_cast<uint4*>(out + ((static_cast<size_t>(b) * out_c8 + g0 + g) * N + n0) * 8) = pack8(o);
    if (two) {
#pragma unroll
      for (int e = 0; e < 4; ++e) o[2 * e] = ob[e].x * inv1, o[2 * e + 1] = ob[e].y * inv1;
      *reinterpret_cast<uint4*>(out + ((static_cast<size_t>(b) * out_c8 + g0 + g) * N + n1) * 8) = pack8(o);
    }
  }
}

// Depth-wise 3x3 conv (padding 1) + bias [+ GELU]: Mlp.dwconv + act (ChangeFormer.py:283-289,512-523).
// grid (x groups * rows / 128, g8, B): a CTA works on ONE 8-channel group (its 9 x 8 weights and 8 biases in shared memory); a thread
// produces 4 horizontally adjacent pixels from a 3 x 6 window, so every loaded and unpacked neighbour feeds up to three taps, the MACs
// run as packed FFMA2 over channel pairs and the GELU on packed pairs.  The first version (one pixel per thread, scalar math) measured
// at the SM's issue limit (330 instructions per 8 outputs, 171 us against a 41 us HBM floor at stage 1); this one issues ~180.
// SPLIT: src and dst hold hi and lo planes; the taps read hi + lo, the output is written as both planes.
template <bool SPLIT>
__global__ void __launch_bounds__(128) dwconv3x3_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                        const float* __restrict__ wgt, const float* __restrict__ bias, int B, int g8,
                                                        int src_c8, int dst_c8, int h, int w, int gelu) {
  __shared__ __align__(16) float s_w[9][8];
  __shared__ __align__(16) float s_b[8];
  const int hw = h * w;
  const int g = blockIdx.y;
  const size_t b = blockIdx.z;
  if (threadIdx.x < 72) s_w[threadIdx.x % 9][threadIdx.x / 9] = __ldg(wgt + (g * 8 + threadIdx.x / 9) * 9 + threadIdx.x % 9);
  if (threadIdx.x < 8) s_b[threadIdx.x] = __ldg(bias + g * 8 + threadIdx.x);
  __syncthreads();
  const __nv_bfloat16* base = src + (b * src_c8 + g) * static_cast<size_t>(hw) * 8;
  __nv_bfloat16* obase = dst + (b * dst_c8 + g) * static_cast<size_t>(hw) * 8;
  const size_t s_lo = static_cast<size_t>(src_c8 >> 1) * hw * 8, d_lo = static_cast<size_t>(dst_c8 >> 1) * hw * 8;   // split planes
  const int xg = (w + 3) >> 2;                                   // groups of 4 pixels per row
  for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < xg * h; item += gridDim.x * blockDim.x) {
    const int y = item / xg, x0 = (item - y * xg) * 4;
    float2 acc[4][4];
    {
      const float4 b0 = *reinterpret_cast<const float4*>(&s_b[0]), b1 = *reinterpret_cast<const float4*>(&s_b[4]);
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        acc[p][0] = make_float2(b0.x, b0.y), acc[p][1] = make_float2(b0.z, b0.w);
        acc[p][2] = make_float2(b1.x, b1.y), acc[p][3] = make_float2(b1.z, b1.w);
      }
    }
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int yy = y + ky - 1;
      const bool row_ok = yy >= 0 && yy < h;
      uint4 q[6], ql[6];
#pragma unroll
      for (int c = 0; c < 6; ++c) {                              // the row's six loads first: independent, in flight together
        const int xx = x0 + c - 1;
        q[c] = (row_ok && xx >= 0 && xx < w) ? __ldg(reinterpret_cast<const uint4*>(base + (static_cast<size_t>(yy) * w + xx) * 8))
                                             : make_uint4(0u, 0u, 0u, 0u);
        if constexpr (SPLIT)
          ql[c] = (row_ok && xx >= 0 && xx < w) ? __ldg(reinterpret_cast<const uint4*>(base + s_lo + (static_cast<size_t>(yy) * w + xx) * 8))
                                                : make_uint4(0u, 0u, 0u, 0u);
      }
      float2 wk[3][4];
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const float4 w0 = *reinterpret_cast<const float4*>(&s_w[ky * 3 + kx][0]), w1 = *reinterpret_cast<const float4*>(&s_w[ky * 3 + kx][4]);
        wk[kx][0] = make_float2(w0.x, w0.y), wk[kx][1] = make_float2(w0.z, w0.w);
        wk[kx][2] = make_float2(w1.x, w1.y), wk[kx][3] = make_float2(w1.z, w1.w);
      }
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        float v[8];
        unpack8(q[c], v);
        if constexpr (SPLIT) {
          float l[8];
          unpack8(ql[c], l);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] += l[j];
        }
        const float2 vp[4] = {make_float2(v[0], v[1]), make_float2(v[2], v[3]), make_float2(v[4], v[5]), make_float2(v[6], v[7])};
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int p = c - kx;                                  // window column c is tap kx of output pixel p
          if (p >= 0 && p < 4) {
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[p][e] = __ffma2_rn(vp[e], wk[kx][e], acc[p][e]);
          }
        }
      }
    }
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      if (x0 + p < w) {
        float o[8];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 r = gelu ? gelu_fast2(acc[p][e]) : acc[p][e];
          o[2 * e] = r.x, o[2 * e + 1] = r.y;
        }
        if constexpr (SPLIT) {
          uint4 oh, olo;
          split8(o, oh, olo);
          *reinterpret_cast<uint4*>(obase + (static_cast<size_t>(y) * w + x0 + p) * 8) = oh;
          *reinterpret_cast<uint4*>(obase + d_lo + (static_cast<size_t>(y) * w + x0 + p) * 8) = olo;
        } else {
          *reinterpret_cast<uint4*>(obase + (static_cast<size_t>(y) * w + x0 + p) * 8) = pack8(o);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// Tensor-core variant of the spatial-reduction attention for exactly 64 keys (every stage of the 256 x 256 configurations): a warp owns
// 16 queries; S = Q K^T and O = P V are mma.sync m16n8k16 bf16 tiles (the whole problem is 64 MMAs per warp -- far too small for a
// tcgen05 / TMEM pipeline, whose 128-row tiles and allocation hand-shake would dominate), the softmax runs on the accumulator
// fragments (row max / sum over the quad that shares a row), and P is re-used as the A operand of the second product straight from
// registers.  K ([key][d]) and V^T ([d][key]) of the (image, head) sit in shared memory as bf16 with padded rows (no bank conflicts
// on the B-fragment loads).  Q, K, V are bf16 tensors already; P is rounded to bf16 for the second product (one more bf16 rounding
// on a path that is bf16 end to end).  grid (N / 64, heads, images), 128 threads.
// SPLIT (lowering.Program.precision): q, kv and out hold hi and lo planes.  K and V^T are staged as both planes (45 KB at D = 80),
// S = Qh Kh + Ql Kh + Qh Kl and O = Ph Vh + Pl Vh + Ph Vl (three mma.sync per tile; the lo x lo term is below 2^-16 relative) with
// P = exp(s - max) split into hi = bf16(P), lo = bf16(P - hi) after the fp32 softmax; the output is normalised by the fp32 row sum
// and written as both planes.
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16x2(a, b);
  const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&hi);
  lo = pack_bf16x2(a - __low2float(h), b - __high2float(h));
}

template <int D, bool SPLIT>   // head dim: 64 or 80 (multiples of 16)
__global__ void __launch_bounds__(128) sr_attention_mma_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ kv,
                                                               __nv_bfloat16* __restrict__ out, int C, int q_c8, int kv_c8, int out_c8,
                                                               int N, float scale) {
  constexpr int NK = 64, KS = D + 8, VS = NK + 8;              // padded row strides (bf16 elements)
  constexpr int NP = SPLIT ? 2 : 1;                            // planes: hi [, lo]
  __shared__ __align__(16) __nv_bfloat16 sk[NP * NK * KS];     // K [plane][key][d]
  __shared__ __align__(16) __nv_bfloat16 svt[NP * D * VS];     // V^T [plane][d][key]
  const int b = blockIdx.z, hd = blockIdx.y;
  const int g0 = hd * (D / 8);
  for (int i = threadIdx.x; i < NK * (D / 8); i += blockDim.x) {
    const int j = i % NK, g = i / NK;                          // consecutive lanes: consecutive keys (coalesced 16 B loads)
    const uint4 kq = __ldg(reinterpret_cast<const uint4*>(kv + ((static_cast<size_t>(b) * kv_c8 + g0 + g) * NK + j) * 8));
    *reinterpret_cast<uint4*>(&sk[j * KS + g * 8]) = kq;
    const uint4 vq = __ldg(reinterpret_cast<const uint4*>(kv + ((static_cast<size_t>(b) * kv_c8 + (C >> 3) + g0 + g) * NK + j) * 8));
    const __nv_bfloat16* ve = reinterpret_cast<const __nv_bfloat16*>(&vq);
#pragma unroll
    for (int e = 0; e < 8; ++e) svt[(g * 8 + e) * VS + j] = ve[e];
  }
  if constexpr (SPLIT) {
    const int lo = kv_c8 >> 1;                                 // first channel group of the lo plane
    for (int i = threadIdx.x; i < NK * (D / 8); i += blockDim.x) {
      const int j = i % NK, g = i / NK;
      const uint4 kq = __ldg(reinterpret_cast<const uint4*>(kv + ((static_cast<size_t>(b) * kv_c8 + lo + g0 + g) * NK + j) * 8));
      *reinterpret_cast<uint4*>(&sk[NK * KS + j * KS + g * 8]) = kq;
      const uint4 vq = __ldg(reinterpret_cast<const uint4*>(kv + ((static_cast<size_t>(b) * kv_c8 + lo + (C >> 3) + g0 + g) * NK + j) * 8));
      const __nv_bfloat16* ve = reinterpret_cast<const __nv_bfloat16*>(&vq);
#pragma unroll
      for (int e = 0; e < 8; ++e) svt[D * VS + (g * 8 + e) * VS + j] = ve[e];
    }
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = lane >> 2, cq = (lane & 3) * 2;                // fragment row / column pair of this lane
  const int n0 = blockIdx.x * 64 + warp * 16;
  if (n0 >= N) return;
  const int na = min(n0 + r, N - 1), nb = min(n0 + r + 8, N - 1);   // clamped: out-of-range rows are computed but never stored
  // ---- S = Q K^T: 8 key tiles x (D / 16) k-steps
  float sacc[8][4];
#pragma unroll
  for (int t = 0; t < 8; ++t) sacc[t][0] = sacc[t][1] = sacc[t][2] = sacc[t][3] = 0.f;
  const __nv_bfloat16* qb = q + (static_cast<size_t>(b) * q_c8 + g0) * static_cast<size_t>(N) * 8;
#pragma unroll
  for (int ks = 0; ks < D / 16; ++ks) {
    uint32_t a[4];
    const __nv_bfloat16* q0 = qb + static_cast<size_t>(2 * ks) * N * 8;
    const __nv_bfloat16* q1 = q0 + static_cast<size_t>(N) * 8;
    a[0] = __ldg(reinterpret_cast<const uint32_t*>(q0 + static_cast<size_t>(na) * 8 + cq));
    a[1] = __ldg(reinterpret_cast<const uint32_t*>(q0 + static_cast<size_t>(nb) * 8 + cq));
    a[2] = __ldg(reinterpret_cast<const uint32_t*>(q1 + static_cast<size_t>(na) * 8 + cq));
    a[3] = __ldg(reinterpret_cast<const uint32_t*>(q1 + static_cast<size_t>(nb) * 8 + cq));
    uint32_t al[4];
    if constexpr (SPLIT) {
      const size_t lo = static_cast<size_t>(q_c8 >> 1) * N * 8;
      al[0] = __ldg(reinterpret_cast<const uint32_t*>(q0 + lo + static_cast<size_t>(na) * 8 + cq));
      al[1] = __ldg(reinterpret_cast<const uint32_t*>(q0 + lo + static_cast<size_t>(nb) * 8 + cq));
      al[2] = __ldg(reinterpret_cast<const uint32_t*>(q1 + lo + static_cast<size_t>(na) * 8 + cq));
      al[3] = __ldg(reinterpret_cast<const uint32_t*>(q1 + lo + static_cast<size_t>(nb) * 8 + cq));
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const __nv_bfloat16* kr = &sk[(t * 8 + r) * KS + ks * 16 + cq];
      mma_bf16_16816(sacc[t], a, *reinterpret_cast<const uint32_t*>(kr), *reinterpret_cast<const uint32_t*>(kr + 8));
      if constexpr (SPLIT) {
        const __nv_bfloat16* kl = kr + NK * KS;
        mma_bf16_16816(sacc[t], al, *reinterpret_cast<const uint32_t*>(kr), *reinterpret_cast<const uint32_t*>(kr + 8));
        mma_bf16_16816(sacc[t], a, *reinterpret_cast<const uint32_t*>(kl), *reinterpret_cast<const uint32_t*>(kl + 8));
      }
    }
  }
  // ---- softmax over the 64 keys of rows r (values [t][0..1]) and r + 8 (values [t][2..3]); a row lives in the 4 lanes of a quad
  float mx0 = -CUDART_INF_F, mx1 = -CUDART_INF_F;
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    mx0 = fmaxf(mx0, fmaxf(sacc[t][0], sacc[t][1]));
    mx1 = fmaxf(mx1, fmaxf(sacc[t][2], sacc[t][3]));
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  float sum0 = 0.f, sum1 = 0.f;
  uint32_t pa[4][4];                                           // P as A fragments: k-step = 16 keys = two key tiles
  uint32_t pl[4][4];                                           // split: the lo plane of P
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    const float p0 = __expf((sacc[t][0] - mx0) * scale), p1 = __expf((sacc[t][1] - mx0) * scale);
    const float p2 = __expf((sacc[t][2] - mx1) * scale), p3 = __expf((sacc[t][3] - mx1) * scale);
    sum0 += p0 + p1;
    sum1 += p2 + p3;
    if constexpr (SPLIT) {
      split_bf16x2(p0, p1, pa[t >> 1][(t & 1) * 2], pl[t >> 1][(t & 1) * 2]);
      split_bf16x2(p2, p3, pa[t >> 1][(t & 1) * 2 + 1], pl[t >> 1][(t & 1) * 2 + 1]);
    } else {
      pa[t >> 1][(t & 1) * 2] = pack_bf16x2(p0, p1);
      pa[t >> 1][(t & 1) * 2 + 1] = pack_bf16x2(p2, p3);
    }
  }
  sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
  sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
  sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
  sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
  const float inv0 = 1.f / sum0, inv1 = 1.f / sum1;
  // ---- O = P V: D / 8 channel tiles x 4 key steps
  __nv_bfloat16* ob = out + (static_cast<size_t>(b) * out_c8 + g0) * static_cast<size_t>(N) * 8;
#pragma unroll
  for (int t = 0; t < D / 8; ++t) {
    float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const __nv_bfloat16* vr = &svt[(t * 8 + r) * VS + ks * 16 + cq];
      mma_bf16_16816(o, pa[ks], *reinterpret_cast<const uint32_t*>(vr), *reinterpret_cast<const uint32_t*>(vr + 8));
      if constexpr (SPLIT) {
        const __nv_bfloat16* vl = vr + D * VS;
        mma_bf16_16816(o, pl[ks], *reinterpret_cast<const uint32_t*>(vr), *reinterpret_cast<const uint32_t*>(vr + 8));
        mma_bf16_16816(o, pa[ks], *reinterpret_cast<const uint32_t*>(vl), *reinterpret_cast<const uint32_t*>(vl + 8));
      }
    }
    if constexpr (SPLIT) {
      const size_t lo = static_cast<size_t>(out_c8 >> 1) * N * 8;
      uint32_t h, l;
      if (n0 + r < N) {
        split_bf16x2(o[0] * inv0, o[1] * inv0, h, l);
        *reinterpret_cast<uint32_t*>(ob + (static_cast<size_t>(t) * N + n0 + r) * 8 + cq) = h;
        *reinterpret_cast<uint32_t*>(ob + lo + (static_cast<size_t>(t) * N + n0 + r) * 8 + cq) = l;
      }
      if (n0 + r + 8 < N) {
        split_bf16x2(o[2] * inv1, o[3] * inv1, h, l);
        *reinterpret_cast<uint32_t*>(ob + (static_cast<size_t>(t) * N + n0 + r + 8) * 8 + cq) = h;
        *reinterpret_cast<uint32_t*>(ob + lo + (static_cast<size_t>(t) * N + n0 + r + 8) * 8 + cq) = l;
      }
    } else {
      if (n0 + r < N) *reinterpret_cast<uint32_t*>(ob + (static_cast<size_t>(t) * N + n0 + r) * 8 + cq) = pack_bf16x2(o[0] * inv0, o[1] * inv0);
      if (n0 + r + 8 < N) *reinterpret_cast<uint32_t*>(ob + (static_cast<size_t>(t) * N + n0 + r + 8) * 8 + cq) = pack_bf16x2(o[2] * inv1, o[3] * inv1);
    }
  }
}

// ------------------------------------------------------------------------------------------
// Squeeze-and-excitation gates (DTCDSCN: SELayer, models/DTCDSCN.py:11-26; SCSEBlock :144-173).
//   pass 1  chan_sum_kernel: per (image, channel) sums over a pixel range -> partial[b][range][C]  (fixed order: deterministic)
//   pass 2  gate_apply_kernel: every CTA finishes the mean, runs the two tiny FC layers for its image in shared memory
//           (g = sigmoid(W2 relu(W1 mean))), then applies its pixel range:
//             mode 0 (SE block tail):  out = relu(x * g + res)                      (SEBasicBlock.forward :93-109)
//             mode 1 (SCSE + skip):    out = x * (1 + g + sigmoid(ws . x_pixel))     (DecoderBlock: x + scse(x), :129-135,164-173)
//           optionally also writing the space-to-depth copy a following stride-2 conv reads.
// HBM-bound: x is read twice (three times in mode 1), written once (twice with the copy).
constexpr int kGateMaxC = 512;
constexpr int kGateMaxH = 32;

// one warp per (pixel range, 8-channel group, image): lanes stride over the range's pixels, butterfly reduce (fixed order)
// SPLIT: src holds hi + lo planes (lo at src_c8/2 groups) and the sums run over hi + lo.
constexpr int kGateRangePix = 512;
template <bool SPLIT>
__global__ void __launch_bounds__(256) chan_sum_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ partial, int C,
                                                       int src_c8, int hw, int ranges, int n_items) {
  const int item = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (item >= n_items) return;
  const int g8 = C >> 3;
  const int r = item % ranges, g = (item / ranges) % g8, b = item / (ranges * g8);
  const int per = (hw + ranges - 1) / ranges;
  const int p0 = r * per, p1 = min(hw, p0 + per);
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const __nv_bfloat16* base = src + (static_cast<size_t>(b) * src_c8 + g) * static_cast<size_t>(hw) * 8;
#pragma unroll 4
  for (int px = p0 + lane; px < p1; px += 32) {
    float v[8];
    if constexpr (SPLIT) load8_split(base + static_cast<size_t>(px) * 8, static_cast<size_t>(src_c8 >> 1) * hw * 8, v);
    else unpack8(__ldg(reinterpret_cast<const uint4*>(base + static_cast<size_t>(px) * 8)), v);
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] += v[j];
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
  }
  if (lane < 8) {
    float a = s[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) a = lane == j ? s[j] : a;
    partial[(static_cast<size_t>(b) * ranges + r) * C + g * 8 + lane] = a;
  }
}

// grid (pixel blocks, B), 256 threads.  Every CTA redoes the two tiny FC layers of its image (C x hid MACs, warp-cooperative),
// then applies its pixels: work items are (channel group, pixel) so small maps with many channels still fill the CTA.
// SPLIT: src, res, dst and dst2 hold hi + lo planes (lo at half the stored channel groups; dst2's lo plane of class k, group g at
// 4*g8 + k*g8 + g).  Reads are hi + lo, the gate and the output are formed in fp32 as above and written as hi and lo.
constexpr int kGateMaxPix = 1024;
template <bool SPLIT>
__global__ void __launch_bounds__(256) gate_apply_kernel(const __nv_bfloat16* __restrict__ src, const __nv_bfloat16* __restrict__ res,
                                                         __nv_bfloat16* __restrict__ dst, __nv_bfloat16* __restrict__ dst2,
                                                         const float* __restrict__ partial, const float* __restrict__ w1,
                                                         const float* __restrict__ w2, const float* __restrict__ ws, int C, int hid,
                                                         int src_c8, int res_c8, int dst_c8, int dst2_c8, int h, int w, int ranges,
                                                         int mode, int pix_per_block) {
  __shared__ float s_mean[kGateMaxC], s_gate[kGateMaxC], s_hid[kGateMaxH], s_gs[kGateMaxPix];
  const int b = blockIdx.y, hw = h * w, g8 = C >> 3;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f;
    for (int r = 0; r < ranges; ++r) a += partial[(static_cast<size_t>(b) * ranges + r) * C + c];
    s_mean[c] = a / static_cast<float>(hw);
  }
  __syncthreads();
  for (int u = warp; u < hid; u += 8) {                 // lanes stride over c: coalesced w1 rows, fixed-order butterfly
    float a = 0.f;
    for (int c = lane; c < C; c += 32) a = fmaf(__ldg(w1 + u * C + c), s_mean[c], a);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) s_hid[u] = fmaxf(a, 0.f);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f;
    for (int u = 0; u < hid; ++u) a = fmaf(__ldg(w2 + c * hid + u), s_hid[u], a);
    s_gate[c] = 1.f / (1.f + expf(-a));
  }
  const int p_begin = blockIdx.x * pix_per_block;
  const int n_pix = min(hw, p_begin + pix_per_block) - p_begin;
  const __nv_bfloat16* sb = src + static_cast<size_t>(b) * src_c8 * hw * 8;
  const size_t s_lo = static_cast<size_t>(src_c8 >> 1) * hw * 8;      // split: offset of the lo plane
  if (mode == 1) {                                       // spatial gate per pixel: sigmoid(ws . x_pixel)
    for (int i = threadIdx.x; i < n_pix; i += blockDim.x) {
      float a = 0.f;
      for (int g = 0; g < g8; ++g) {
        float v[8];
        if constexpr (SPLIT) load8_split(sb + (static_cast<size_t>(g) * hw + p_begin + i) * 8, s_lo, v);
        else unpack8(__ldg(reinterpret_cast<const uint4*>(sb + (static_cast<size_t>(g) * hw + p_begin + i) * 8)), v);
#pragma unroll
        for (int j = 0; j < 8; ++j) a = fmaf(v[j], __ldg(ws + g * 8 + j), a);
      }
      s_gs[i] = 1.f / (1.f + expf(-a));
    }
  }
  __syncthreads();
  const int hw2 = hw >> 2, w2h = w >> 1;
  for (int it = threadIdx.x; it < n_pix * g8; it += blockDim.x) {
    const int g = it / n_pix, i = it - g * n_pix, pix = p_begin + i;
    float v[8];
    if constexpr (SPLIT) load8_split(sb + (static_cast<size_t>(g) * hw + pix) * 8, s_lo, v);
    else unpack8(__ldg(reinterpret_cast<const uint4*>(sb + (static_cast<size_t>(g) * hw + pix) * 8)), v);
    if (mode == 0) {
      float rv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if constexpr (SPLIT) {
        if (res != nullptr)
          load8_split(res + ((static_cast<size_t>(b) * res_c8 + g) * hw + pix) * 8, static_cast<size_t>(res_c8 >> 1) * hw * 8, rv);
      } else if (res != nullptr) unpack8(__ldg(reinterpret_cast<const uint4*>(res + ((static_cast<size_t>(b) * res_c8 + g) * hw + pix) * 8)), rv);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaxf(fmaf(v[j], s_gate[g * 8 + j], rv[j]), 0.f);
    } else {
      const float gs = s_gs[i];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = v[j] * (1.f + s_gate[g * 8 + j] + gs);
    }
    if constexpr (SPLIT) {
      uint4 qh, ql;
      split8(v, qh, ql);
      __nv_bfloat16* o = dst + ((static_cast<size_t>(b) * dst_c8 + g) * hw + pix) * 8;
      *reinterpret_cast<uint4*>(o) = qh;
      *reinterpret_cast<uint4*>(o + static_cast<size_t>(dst_c8 >> 1) * hw * 8) = ql;
      if (dst2 != nullptr) {
        const int y = pix / w, x = pix - y * w;
        __nv_bfloat16* o2 = dst2 + ((static_cast<size_t>(b) * dst2_c8 + ((y & 1) * 2 + (x & 1)) * g8 + g) * hw2 +
                                    static_cast<size_t>(y >> 1) * w2h + (x >> 1)) * 8;
        *reinterpret_cast<uint4*>(o2) = qh;
        *reinterpret_cast<uint4*>(o2 + static_cast<size_t>(dst2_c8 >> 1) * hw2 * 8) = ql;
      }
      continue;
    }
    const uint4 q = pack8(v);
    *reinterpret_cast<uint4*>(dst + ((static_cast<size_t>(b) * dst_c8 + g) * hw + pix) * 8) = q;
    if (dst2 != nullptr) {
      const int y = pix / w, x = pix - y * w;
      *reinterpret_cast<uint4*>(dst2 + ((static_cast<size_t>(b) * dst2_c8 + ((y & 1) * 2 + (x & 1)) * g8 + g) * hw2 +
                                        static_cast<size_t>(y >> 1) * w2h + (x >> 1)) * 8) = q;
    }
  }
}

// dst = sum of up to 5 tensors (Dblock: x + d1 + d2 + d3 + d4, models/DTCDSCN.py:65-71), elementwise over 16-byte vectors
// SPLIT: every tensor holds hi + lo planes; vecs counts the hi vectors and plane_vecs the vectors of one plane of one image (as in
// absdiff_kernel).  The fp32 sum of the hi + lo values, in source order, is written as hi and lo.
struct AddNParams {
  const __nv_bfloat16* src[5];
  int n;
};
template <bool SPLIT>
__global__ void __launch_bounds__(256) add_n_kernel(const AddNParams p, __nv_bfloat16* __restrict__ dst, size_t vecs, int plane_vecs) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < vecs; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    if constexpr (SPLIT) {
      const size_t hv = i + (i / plane_vecs) * plane_vecs;            // hi vector; its lo vector is plane_vecs further
      const size_t lo_off = static_cast<size_t>(plane_vecs) * 8;
      float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int k = 0; k < p.n; ++k) {
        float v[8];
        load8_split(p.src[k] + hv * 8, lo_off, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] += v[j];
      }
      uint4 qh, ql;
      split8(a, qh, ql);
      reinterpret_cast<uint4*>(dst)[hv] = qh;
      reinterpret_cast<uint4*>(dst)[hv + plane_vecs] = ql;
      continue;
    }
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < p.n; ++k) {
      float v[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(p.src[k]) + i), v);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += v[j];
    }
    reinterpret_cast<uint4*>(dst)[i] = pack8(a);
  }
}

}  // namespace stcd
