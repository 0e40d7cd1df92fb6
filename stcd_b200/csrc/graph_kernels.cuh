// ViG Grapher graph ops (gcn_lib, imported by models/pyramid_vig.py:17; semantics: SURVEY.md App. D):
// dense dilated kNN graph construction and the max-relative aggregation, on the reference's own layout
// (fp32 node features [B][C][N], N = H*W nodes; int64 neighbour tables).
//
// The neighbour ORDER is what the downstream max-relative features depend on, so the distance keeps fp32 accuracy with
// the reference's expression (|x|^2 - 2 x.y + |y|^2 on L2-normalised nodes, plus the relative-position bias): a bf16 or tf32
// distance reorders near-equidistant neighbours.  Two implementations: knn_prep_kernel + knn_pipe_kernel (round 2; tcgen05,
// the inner products as six MMAs over three exact bf16 planes per operand, top-k from TMEM) for k * dilation <= 27, and
// knn_graph_kernel (round 1; fp32 FFMA2 on the CUDA cores, the [64 x M] distance tile in registers) for anything else.
// The dense [B, N, M] tensor of the reference never exists in either.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "ptx.cuh"
#include "transformer_kernels.cuh"     // unpack8 / split8 (split-precision bilinear up-sampling)

namespace stcd {

// xn[b][:, n] = x[b][:, n] / max(||x[b, :, n]||_2, 1e-12)   (F.normalize(x, p=2, dim=1)).  One thread per node, coalesced
// over n; the channel sum runs in index order, the division is IEEE.
// Block = 32 nodes x 8 channel slices (grid: node groups x images): slice s sums channels s, s + 8, ... in index order, the 8
// partial sums are added in slice order (fixed order -> deterministic), then every slice writes its channels.
__global__ void __launch_bounds__(256) normalize_nodes_kernel(const float* __restrict__ x, float* __restrict__ xn, int B, int C,
                                                             int N) {
  __shared__ float part[8][32];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int groups = (N + 31) / 32;
  for (int item = blockIdx.x; item < B * groups; item += gridDim.x) {
    const int b = item / groups, n = (item - b * groups) * 32 + lane;
    const bool ok = n < N;
    const float* p = x + static_cast<size_t>(b) * C * N + n;
    float s = 0.f;
    if (ok)
      for (int c = slice; c < C; c += 8) {
        const float v = __ldg(p + static_cast<size_t>(c) * N);
        s = fmaf(v, v, s);
      }
    __syncthreads();
    part[slice][lane] = s;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += part[k][lane];
    const float den = fmaxf(sqrtf(tot), 1e-12f);
    float* o = xn + static_cast<size_t>(b) * C * N + n;
    if (ok)
      for (int c = slice; c < C; c += 8) o[static_cast<size_t>(c) * N] = __fdiv_rn(__ldg(p + static_cast<size_t>(c) * N), den);
  }
}

constexpr int kKnnQ = 64;     // queries per CTA (8 per warp)
constexpr int kKnnM = 256;    // max keys (8 per lane)
constexpr int kKnnCC = 32;    // channels per shared-memory chunk

// grid (ceil(N / 64), B), 256 threads.  xn, yn: L2-normalised nodes.  nn_idx[b][n][t] = index of the (t*dilation)-th
// nearest key of query n.  Warp w owns queries 8w..8w+7, lane l owns keys 8l..8l+7: per channel the 8 query values are
// two broadcast LDS.128, the 8 key values two LDS.128, feeding 64 FMAs.  The k*dilation selection rounds run the eight
// queries' warp arg-min chains interleaved (independent shuffle chains hide each other's latency).
__global__ void __launch_bounds__(256) knn_graph_kernel(const float* __restrict__ xn, const float* __restrict__ yn,
                                                        const float* __restrict__ relpos, int C, int N, int M, int k,
                                                        int dilation, long long* __restrict__ nn_idx) {
  __shared__ __align__(16) float xs[kKnnCC][kKnnQ];
  __shared__ __align__(16) float ys[kKnnCC][kKnnM];
  const int b = blockIdx.y, n0 = blockIdx.x * kKnnQ;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* xb = xn + static_cast<size_t>(b) * C * N;
  const float* yb = yn + static_cast<size_t>(b) * C * M;
  // packed fp32 accumulators (FFMA2): key pairs (2j, 2j + 1) of one query share an instruction.  Each lane of an FFMA2 is an IEEE
  // fma and the channel order is unchanged, so every dot product is bit-identical to the scalar loop.
  float2 dot2[8][4], xsq2[4], ysq2[4];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
#pragma unroll
    for (int j = 0; j < 4; ++j) dot2[q][j] = make_float2(0.f, 0.f);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) xsq2[j] = ysq2[j] = make_float2(0.f, 0.f);
  // 16-byte staging copies need 16-byte aligned rows
  const bool vec_ok = ((N & 3) == 0) && ((M & 3) == 0) && (((reinterpret_cast<uintptr_t>(xn) | reinterpret_cast<uintptr_t>(yn)) & 15) == 0);
  for (int c0 = 0; c0 < C; c0 += kKnnCC) {
    __syncthreads();
    // cp.async with zero-fill out of range; all copies of a thread are in flight at once
    if (vec_ok) {
      for (int i = threadIdx.x; i < (kKnnQ / 4) * kKnnCC; i += blockDim.x) {
        const int q = (i % (kKnnQ / 4)) * 4, cc = i / (kKnnQ / 4);
        const int n = n0 + q, c = c0 + cc;
        const bool ok = (n < N) && (c < C);
        const float* gp = xb + (ok ? static_cast<size_t>(c) * N + n : 0);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(&xs[cc][q]))),
                     "l"(gp), "r"(ok ? 16 : 0) : "memory");
      }
      for (int i = threadIdx.x; i < (kKnnM / 4) * kKnnCC; i += blockDim.x) {
        const int j = (i % (kKnnM / 4)) * 4, cc = i / (kKnnM / 4);
        const int c = c0 + cc;
        const bool ok = (j < M) && (c < C);
        const float* gp = yb + (ok ? static_cast<size_t>(c) * M + j : 0);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(&ys[cc][j]))),
                     "l"(gp), "r"(ok ? 16 : 0) : "memory");
      }
    } else {
      for (int i = threadIdx.x; i < kKnnQ * kKnnCC; i += blockDim.x) {
        const int q = i % kKnnQ, cc = i / kKnnQ;
        const int n = n0 + q, c = c0 + cc;
        const bool ok = (n < N) && (c < C);
        const float* gp = xb + (ok ? static_cast<size_t>(c) * N + n : 0);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(&xs[cc][q]))),
                     "l"(gp), "r"(ok ? 4 : 0) : "memory");
      }
      for (int i = threadIdx.x; i < kKnnM * kKnnCC; i += blockDim.x) {
        const int j = i % kKnnM, cc = i / kKnnM;
        const int c = c0 + cc;
        const bool ok = (j < M) && (c < C);
        const float* gp = yb + (ok ? static_cast<size_t>(c) * M + j : 0);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(&ys[cc][j]))),
                     "l"(gp), "r"(ok ? 4 : 0) : "memory");
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
#pragma unroll 4
    for (int cc = 0; cc < kKnnCC; ++cc) {
      const float4 xa = *reinterpret_cast<const float4*>(&xs[cc][warp * 8]), xb4 = *reinterpret_cast<const float4*>(&xs[cc][warp * 8 + 4]);
      const float4 ya = *reinterpret_cast<const float4*>(&ys[cc][lane * 8]), yb4 = *reinterpret_cast<const float4*>(&ys[cc][lane * 8 + 4]);
      const float xv[8] = {xa.x, xa.y, xa.z, xa.w, xb4.x, xb4.y, xb4.z, xb4.w};
      const float2 yp[4] = {make_float2(ya.x, ya.y), make_float2(ya.z, ya.w), make_float2(yb4.x, yb4.y), make_float2(yb4.z, yb4.w)};
      const float2 xp[4] = {make_float2(xa.x, xa.y), make_float2(xa.z, xa.w), make_float2(xb4.x, xb4.y), make_float2(xb4.z, xb4.w)};
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float2 xx = make_float2(xv[q], xv[q]);
#pragma unroll
        for (int j = 0; j < 4; ++j) dot2[q][j] = __ffma2_rn(xx, yp[j], dot2[q][j]);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        xsq2[j] = __ffma2_rn(xp[j], xp[j], xsq2[j]);
        ysq2[j] = __ffma2_rn(yp[j], yp[j], ysq2[j]);
      }
    }
  }
  float dot[8][8], xsq[8], ysq[8];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    xsq[2 * j] = xsq2[j].x, xsq[2 * j + 1] = xsq2[j].y;
    ysq[2 * j] = ysq2[j].x, ysq[2 * j + 1] = ysq2[j].y;
#pragma unroll
    for (int q = 0; q < 8; ++q) dot[q][2 * j] = dot2[q][j].x, dot[q][2 * j + 1] = dot2[q][j].y;
  }
  // distances, in place: the reference's order of operations (x_sq + (-2 * inner)) + y_sq, then + relative_pos
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int n = n0 + warp * 8 + q;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int key = lane * 8 + j;
      float dv = __fadd_rn(__fadd_rn(xsq[q], -2.f * dot[q][j]), ysq[j]);
      if (relpos != nullptr && key < M && n < N) dv = __fadd_rn(dv, __ldg(relpos + static_cast<size_t>(n) * M + key));
      dot[q][j] = key < M ? dv : CUDART_INF_F;
    }
  }
  const int kd = k * dilation;
  int phase = 0, slot = 0;      // every dilation-th winner is kept: counters instead of t % dilation, t / dilation
  for (int t = 0; t < kd; ++t) {
    float best[8];
    int bi[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      best[q] = dot[q][0];
      bi[q] = lane * 8;
#pragma unroll
      for (int j = 1; j < 8; ++j)
        if (dot[q][j] < best[q]) {
          best[q] = dot[q][j];
          bi[q] = lane * 8 + j;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float ov = __shfl_xor_sync(0xffffffffu, best[q], o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi[q], o);
        if (ov < best[q] || (ov == best[q] && oi < bi[q])) {   // ties: smaller index
          best[q] = ov;
          bi[q] = oi;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (lane * 8 + j == bi[q]) dot[q][j] = CUDART_INF_F;
    }
    if (phase == 0) {
      if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int n = n0 + warp * 8 + q;
          if (n < N) nn_idx[(static_cast<size_t>(b) * N + n) * k + slot] = bi[q];
        }
      }
      ++slot;
    }
    if (++phase == dilation) phase = 0;
  }
}

// ------------------------------------------------------------------------------------------
// The same dense dilated kNN with the pairwise products on the tensor cores (tcgen05, TMEM accumulator) and the top-k
// selection in the epilogue warps, straight from TMEM (north star: "pairwise distance as a tensor-core GEMM plus a warp-level
// top-k"; call sites models/pyramid_vig.py:17, models/ChangeVIG.py:61-65).
//
// Precision.  The neighbour ORDER feeds a max over neighbours, so the inner products must stay at fp32 accuracy: a bf16 or
// tf32 product reorders near-equidistant neighbours.  Every fp32 operand is therefore split into THREE bf16 planes,
// v = hi + lo + lo2 (24 mantissa bits, i.e. exactly the fp32 value), and the product is the six MMAs
//     hi*hi + hi*lo + lo*hi + lo*lo + hi*lo2 + lo2*hi        (what is dropped is below 2^-25 relative)
// whose bf16 x bf16 terms are exact in the fp32 accumulator.  The distance, the relative-position bias and the ordering
// rule (ascending distance, ties to the smaller index, every dilation-th neighbour kept) are those of knn_graph_kernel.
//
// One CTA = 128 queries of one image against all M <= 256 keys: D[128 x M] (TMEM, fp32) += X[128 x 16] * Y[M x 16]^T per 16
// channels and plane pair, operands in the un-swizzled K-major core-matrix layout [plane][c/8][row][8] (8 rows x 16 B
// contiguous: SBO = 128 B, LBO = rows * 16 B).  Cost: N*M*C*6 MACs at tensor rate -- 30 MMAs of 128 cycles per 128 queries for
// C = 80 -- against N*M*C fp32 FMAs plus k*dilation warp arg-min rounds over a register tile before (23 % of the ChangeGNNV1 step).
// Epilogue: thread q of warps 0-3 owns query q (= TMEM lane q), walks its M distances in index order and keeps the KD
// smallest in a sorted register list (insertion with strict '<': an equal distance stays behind the smaller index).
constexpr int kKnnTQ = 128;    // queries per CTA (= MMA M)

__device__ __forceinline__ void split3_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo, __nv_bfloat16& lo2) {
  hi = __float2bfloat16_rn(v);
  const float r1 = v - __bfloat162float(hi);          // exact
  lo = __float2bfloat16_rn(r1);
  lo2 = __float2bfloat16_rn(r1 - __bfloat162float(lo));
}

__device__ __forceinline__ uint64_t knn_desc(uint32_t saddr, uint32_t lbo_bytes) {     // K-major, no swizzle, SBO = 128 B
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>(128 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  return d;
}

// ------------------------------------------------------------------------------------------
// The operands are normalised and split into their three bf16 planes ONCE per graph op by knn_prep_kernel (it replaces
// normalize_nodes_kernel on this path), stored in global memory in the shared-memory operand layout, and knn_pipe_kernel
// only moves them: a producer warp issues 1-D bulk copies into a two-stage ring, an MMA warp issues the six products per 16
// channels, four epilogue warps select the neighbours from TMEM.  (A first version staged and converted fp32 inside the
// kernel, single-buffered, and re-read the squared norms from L2 per CTA: the tensor pipe waited on serial load latency and
// the ChangeGNNV1 graph ops only went 4.46 -> 3.85 ms; this form takes them to 2.96 ms.)
//
// planes: bf16 [B][3 planes][G_pad = groups of 8 channels, padded to a multiple of 4][R_pad rows][8]; sq: fp32 [B][R_pad]
// (R_pad = rows rounded up to 128: queries are copied 128 at a time, keys MP = M rounded up to 16 at a time; y := x shares x's planes).
// Padding rows / groups are zero (the buffer is cleared once; the kernels never write them).
constexpr int kKnnStageC = 32;          // channels per pipeline stage (4 groups)

__host__ __device__ inline int knn_gpad(int C) { return ((C + 7) / 8 + 3) & ~3; }
__host__ __device__ inline int knn_rpad(int rows, int mult) { return (rows + mult - 1) / mult * mult; }

// grid: node groups x images (grid-stride), 256 threads = 32 nodes x 8 slices.  F.normalize(x, p=2, dim=1) in fp32 exactly as
// normalize_nodes_kernel, then the three-plane split and |xn|^2.
__global__ void __launch_bounds__(256) knn_prep_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ planes, float* __restrict__ sq,
                                                      int B, int C, int N, int G_pad, int R_pad) {
  __shared__ float part[8][32];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int groups = (N + 31) / 32;
  const int G = (C + 7) / 8;
  for (int item = blockIdx.x; item < B * groups; item += gridDim.x) {
    const int b = item / groups, n = (item - b * groups) * 32 + lane;
    const bool ok = n < N;
    const float* p = x + static_cast<size_t>(b) * C * N + n;
    float s = 0.f;
    if (ok)
      for (int c = slice; c < C; c += 8) {
        const float v = __ldg(p + static_cast<size_t>(c) * N);
        s = fmaf(v, v, s);
      }
    __syncthreads();
    part[slice][lane] = s;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += part[k][lane];
    const float den = fmaxf(sqrtf(tot), 1e-12f);
    float s2 = 0.f;
    if (ok) {
      for (int g = slice; g < G; g += 8) {
        __align__(16) __nv_bfloat16 h[8], l[8], l2[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int c = g * 8 + j;
          const float v = c < C ? __fdiv_rn(__ldg(p + static_cast<size_t>(c) * N), den) : 0.f;
          s2 = fmaf(v, v, s2);
          split3_bf16(v, h[j], l[j], l2[j]);
        }
        const size_t plane = static_cast<size_t>(G_pad) * R_pad * 8;      // elements per plane
        __nv_bfloat16* o = planes + static_cast<size_t>(b) * 3 * plane + (static_cast<size_t>(g) * R_pad + n) * 8;
        *reinterpret_cast<uint4*>(o) = *reinterpret_cast<const uint4*>(h);
        *reinterpret_cast<uint4*>(o + plane) = *reinterpret_cast<const uint4*>(l);
        *reinterpret_cast<uint4*>(o + 2 * plane) = *reinterpret_cast<const uint4*>(l2);
      }
    }
    __syncthreads();
    part[slice][lane] = s2;
    __syncthreads();
    if (slice == 0 && ok) {
      float t2 = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) t2 += part[k][lane];
      sq[static_cast<size_t>(b) * R_pad + n] = t2;
    }
  }
}

// grid (ceil(N / 128), B), 192 threads: warps 0-3 epilogue (TMEM lane quarters 0-3), warp 4 producer, warp 5 MMA issuer.
// dynamic shared memory: 2 stages x 3 planes x 4 groups x (128 + MP) rows x 16 B.
template <int KD>
__global__ void __launch_bounds__(192) knn_pipe_kernel(const __nv_bfloat16* __restrict__ xp, const float* __restrict__ xsq, int NR_pad,
                                                       const __nv_bfloat16* __restrict__ yp, const float* __restrict__ ysq, int MR_pad, int MP,
                                                       const float* __restrict__ relpos, int C, int N, int M, int k, int dilation,
                                                       long long* __restrict__ nn_idx) {
  extern __shared__ uint8_t knn_smem_raw[];
  __shared__ __align__(8) uint64_t full[2], empty[2], acc_full;
  __shared__ uint32_t tmem_base_smem;
  __shared__ float s_ysq[kKnnM];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(knn_smem_raw) + 127) & ~uintptr_t(127));
  const int b = blockIdx.y, n0 = blockIdx.x * kKnnTQ;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int G_pad = knn_gpad(C);
  const int n_chunks = G_pad / 4;
  const uint32_t x_grp = kKnnTQ * 16, y_grp = static_cast<uint32_t>(MP) * 16;       // bytes of one 8-channel group in a stage
  const uint32_t x_plane = 4 * x_grp, y_plane = 4 * y_grp;
  const uint32_t stage_bytes = 3 * (x_plane + y_plane);
  uint32_t tmem_cols = 32;
  while (tmem_cols < static_cast<uint32_t>(MP)) tmem_cols <<= 1;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(&acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 5) {
    tmem_alloc(&tmem_base_smem, tmem_cols);
    tmem_relinquish();
  }
  for (int j = threadIdx.x; j < kKnnM; j += blockDim.x) s_ysq[j] = j < M ? __ldg(ysq + static_cast<size_t>(b) * MR_pad + j) : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_smem;
  if (warp == 4) {
    // ---- producer: per stage 12 copies of 128 query rows and 12 of MP key rows (plane x group), one per lane
    const size_t x_pl = static_cast<size_t>(G_pad) * NR_pad * 16, y_pl = static_cast<size_t>(G_pad) * MR_pad * 16;   // bytes per plane in global memory
    const uint8_t* xg = reinterpret_cast<const uint8_t*>(xp) + static_cast<size_t>(b) * 3 * x_pl + static_cast<size_t>(n0) * 16;
    const uint8_t* yg = reinterpret_cast<const uint8_t*>(yp) + static_cast<size_t>(b) * 3 * y_pl;
    for (int c = 0; c < n_chunks; ++c) {
      const int st = c & 1;
      mbar_wait_relaxed(&empty[st], ((c >> 1) & 1) ^ 1);
      if (lane == 0) mbar_expect_tx(&full[st], stage_bytes);
      __syncwarp();
      uint8_t* dst = smem + static_cast<size_t>(st) * stage_bytes;
      if (lane < 24) {
        const int pl = (lane % 12) / 4, g = lane & 3;
        if (lane < 12)
          bulk_load(dst + pl * x_plane + g * x_grp, xg + pl * x_pl + static_cast<size_t>(c * 4 + g) * NR_pad * 16, x_grp, &full[st]);
        else
          bulk_load(dst + 3 * x_plane + pl * y_plane + g * y_grp, yg + pl * y_pl + static_cast<size_t>(c * 4 + g) * MR_pad * 16, y_grp, &full[st]);
      }
    }
    __syncwarp();
  } else if (warp == 5) {
    // ---- MMA issuer: hi*hi, hi*lo, lo*hi, lo*lo, hi*lo2, lo2*hi per 16 channels
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc_bf16(static_cast<uint32_t>(MP));
    uint32_t accum = 0;
    for (int c = 0; c < n_chunks; ++c) {
      const int st = c & 1;
      mbar_wait(&full[st], (c >> 1) & 1);
      tc_fence_after();
      if (leader) {
        const uint32_t xa = smem_u32(smem + static_cast<size_t>(st) * stage_bytes), ya = xa + 3 * x_plane;
        const int pa[6] = {0, 0, 1, 1, 0, 2}, pb[6] = {0, 1, 0, 1, 2, 0};
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
          for (int t = 0; t < 6; ++t) {
            umma_bf16(tmem_d, knn_desc(xa + pa[t] * x_plane + ks * 2 * x_grp, x_grp), knn_desc(ya + pb[t] * y_plane + ks * 2 * y_grp, y_grp), idesc,
                      accum);
            accum = 1;
          }
        }
        umma_commit(&empty[st]);
        if (c == n_chunks - 1) umma_commit(&acc_full);
      }
      __syncwarp();
    }
  } else {
    // ---- epilogue: thread q owns query q (= TMEM lane q)
    const int q = threadIdx.x, n = n0 + q;
    const float xs2 = n < N ? __ldg(xsq + static_cast<size_t>(b) * NR_pad + n) : 0.f;
    float bv[KD];
    int bi[KD];
#pragma unroll
    for (int t = 0; t < KD; ++t) {
      bv[t] = CUDART_INF_F;
      bi[t] = 0x7fffffff;
    }
    const uint32_t trow = tmem_d + (static_cast<uint32_t>(warp * 32) << 16);
    const float* rp = (relpos != nullptr && n < N) ? relpos + static_cast<size_t>(n) * M : nullptr;
    const bool rp_vec = ((M & 3) == 0) && ((reinterpret_cast<uintptr_t>(relpos) & 15) == 0);
    // this query's relative-position row, 16 keys at a time, fetched ONE CHUNK AHEAD (the first chunk before the accumulator
    // is even complete): read at the point of use, every chunk exposed a full L2 round trip -- 16 of them per query
    auto load_rp = [&](int j0, float (&dst)[16]) {
      if (rp != nullptr && rp_vec && j0 + 16 <= M) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 r4 = __ldg(reinterpret_cast<const float4*>(rp + j0) + j);
          dst[4 * j] = r4.x, dst[4 * j + 1] = r4.y, dst[4 * j + 2] = r4.z, dst[4 * j + 3] = r4.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) dst[j] = (rp != nullptr && j0 + j < M) ? __ldg(rp + j0 + j) : 0.f;
      }
    };
    float rp_nxt[16];
    load_rp(0, rp_nxt);
    mbar_wait_relaxed(&acc_full, 0);
    tc_fence_after();
    for (int j0 = 0; j0 < MP; j0 += 16) {
      uint32_t raw[16];
      tmem_ld16(trow + j0, raw);
      float rpv[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) rpv[j] = rp_nxt[j];
      if (j0 + 16 < MP) load_rp(j0 + 16, rp_nxt);
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int key = j0 + j;
        // the reference's order of operations: (x_sq + (-2 * inner)) + y_sq, then + relative_pos
        float dv = __fadd_rn(__fadd_rn(xs2, -2.f * __uint_as_float(raw[j])), s_ysq[key]);
        if (rp != nullptr) dv = __fadd_rn(dv, rpv[j]);
        if (key >= M) dv = CUDART_INF_F;
        if (dv < bv[KD - 1]) {          // strict: an equal distance stays behind the earlier (smaller) index
          bv[KD - 1] = dv;
          bi[KD - 1] = key;
#pragma unroll
          for (int t = KD - 1; t > 0; --t) {
            const bool sw = bv[t] < bv[t - 1];
            const float tv = sw ? bv[t - 1] : bv[t];
            const int ti = sw ? bi[t - 1] : bi[t];
            bv[t - 1] = sw ? bv[t] : bv[t - 1];
            bi[t - 1] = sw ? bi[t] : bi[t - 1];
            bv[t] = tv;
            bi[t] = ti;
          }
        }
      }
    }
    if (n < N) {
      long long* o = nn_idx + (static_cast<size_t>(b) * N + n) * k;
#pragma unroll
      for (int t = 0; t < KD; ++t)
        if (t % dilation == 0 && t / dilation < k) o[t / dilation] = bi[t];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem_d, tmem_cols);
}

// Max-relative aggregation (MRConv2d): m[b][c][n] = max_t ( y[b][c][nn_idx[b][n][t]] - x[b][c][n] ).
// interleave = 0: out [B][C][N] = m;  interleave = 1: out [B][2C][N] with channel 2c = x, 2c+1 = m (the
// channel-interleaved input of MRConv2d's grouped 1x1 conv).  One thread per (b, c, n), coalesced over n; the
// neighbour table of a node is re-read per channel from L1/L2, the y gathers stay inside one M-float row.
__global__ void __launch_bounds__(256) max_relative_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                           const long long* __restrict__ nn_idx, int B, int C, int N, int M,
                                                           int k, int interleave, float* __restrict__ out) {
  const size_t total = static_cast<size_t>(B) * C * N;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t n = i % N;
    const size_t bc = i / N;
    const size_t c = bc % C, b = bc / C;
    const float xv = __ldg(x + i);
    const float* yrow = y + (b * C + c) * M;
    const long long* idx = nn_idx + (b * N + n) * k;
    float m = -CUDART_INF_F;
    for (int t = 0; t < k; ++t) {
      const long long j = __ldg(idx + t);
      m = fmaxf(m, __fsub_rn(__ldg(yrow + j), xv));
    }
    if (interleave) {
      float* o = out + (b * 2 * C + 2 * c) * N + n;
      o[0] = xv;
      o[N] = m;
    } else {
      out[i] = m;
    }
  }
}

// ---- plan-tensor variants (the Grapher inside a lowered net: activations are bf16 [img][c/8][hw][8]) ----

// bf16 [B][c8][N][8] -> fp32 [B][C][N] (the layout the graph kernels read).  One thread per (b, group, n).
__global__ void __launch_bounds__(256) unpack_nodes_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, int B,
                                                           int src_c8, int C, int N) {
  const int g8 = C >> 3;
  const size_t total = static_cast<size_t>(B) * g8 * N;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t n = i % N;
    const size_t r = i / N;
    const size_t g = r % g8, b = r / g8;
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(src + ((b * src_c8 + g) * N + n) * 8));
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
    float* o = dst + (b * C + g * 8) * N + n;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
      o[static_cast<size_t>(2 * j) * N] = __low2float(h);
      o[static_cast<size_t>(2 * j + 1) * N] = __high2float(h);
    }
  }
}

// F.avg_pool2d(x, r, r) on fp32 [B*C][H][W] -> [B*C][H/r][W/r]; sums in row-major window order, then / r^2
__global__ void __launch_bounds__(256) avgpool_nodes_kernel(const float* __restrict__ x, float* __restrict__ y, size_t planes, int H,
                                                            int W, int r) {
  const int ho = H / r, wo = W / r;
  const size_t total = planes * ho * wo;
  const float inv = 1.0f / static_cast<float>(r * r);
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(i % wo);
    const size_t t = i / wo;
    const int oy = static_cast<int>(t % ho);
    const size_t pl = t / ho;
    const float* p = x + (pl * H + static_cast<size_t>(oy) * r) * W + static_cast<size_t>(ox) * r;
    float s = 0.f;
    for (int a = 0; a < r; ++a)
      for (int b = 0; b < r; ++b) s += __ldg(p + static_cast<size_t>(a) * W + b);
    y[i] = s * inv;
  }
}

// max-relative with a bf16 [B][c8][N][8] destination: one thread per (b, 8-channel group, n)
__global__ void __launch_bounds__(256) max_relative_nc8_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                               const long long* __restrict__ nn_idx, int B, int C, int N, int M,
                                                               int k, __nv_bfloat16* __restrict__ dst, int dst_c8) {
  const int g8 = C >> 3;
  const size_t total = static_cast<size_t>(B) * g8 * N;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t n = i % N;
    const size_t r = i / N;
    const size_t g = r % g8, b = r / g8;
    const long long* idx = nn_idx + (b * N + n) * k;
    float xv[8], m[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      xv[j] = __ldg(x + (b * C + g * 8 + j) * N + n);
      m[j] = -CUDART_INF_F;
    }
    for (int t = 0; t < k; ++t) {
      const long long jn = __ldg(idx + t);
#pragma unroll
      for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], __fsub_rn(__ldg(y + (b * C + g * 8 + j) * M + jn), xv[j]));
    }
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      __nv_bfloat162 h = __floats2bfloat162_rn(m[2 * j], m[2 * j + 1]);
      w[j] = *reinterpret_cast<uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(dst + ((b * dst_c8 + g) * N + n) * 8) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// Bilinear up-sampling by an integer factor, align_corners=False (PyTorch's area_pixel_compute_source_index:
// src = (dst + 0.5) / scale - 0.5 clamped at 0), bf16 [B][c8][h][w][8] -> bf16 [B][c8][s*h][s*w][8], fp32 arithmetic.
// SPLIT (lowering.Program.precision): src and dst hold hi and lo planes (channel groups [0, c8/2) and [c8/2, c8)); the four taps
// read hi + lo and the result is written as hi = bf16(v), lo = bf16(v - hi).
template <bool SPLIT>
__global__ void __launch_bounds__(256) bilinear_up_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                          int B, int g8, int src_c8, int dst_c8, int h, int w, int scale) {
  const int ho = h * scale, wo = w * scale;
  const size_t total = static_cast<size_t>(B) * g8 * ho * wo;
  const float rs = 1.0f / static_cast<float>(scale);
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(i % wo);
    size_t t = i / wo;
    const int oy = static_cast<int>(t % ho);
    t /= ho;
    const size_t g = t % g8, b = t / g8;
    const float sy = fmaxf(rs * (static_cast<float>(oy) + 0.5f) - 0.5f, 0.f);
    const float sx = fmaxf(rs * (static_cast<float>(ox) + 0.5f) - 0.5f, 0.f);
    const int y0 = static_cast<int>(sy), x0 = static_cast<int>(sx);
    const int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
    const float ly = sy - static_cast<float>(y0), lx = sx - static_cast<float>(x0);
    const float hy = 1.f - ly, hx = 1.f - lx;
    const __nv_bfloat16* base = src + (b * src_c8 + g) * static_cast<size_t>(h) * w * 8;
    const uint4 q00 = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<size_t>(y0) * w + x0) * 8));
    const uint4 q01 = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<size_t>(y0) * w + x1) * 8));
    const uint4 q10 = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<size_t>(y1) * w + x0) * 8));
    const uint4 q11 = __ldg(reinterpret_cast<const uint4*>(base + (static_cast<size_t>(y1) * w + x1) * 8));
    const uint32_t a[4] = {q00.x, q00.y, q00.z, q00.w}, bq[4] = {q01.x, q01.y, q01.z, q01.w};
    const uint32_t c[4] = {q10.x, q10.y, q10.z, q10.w}, dq[4] = {q11.x, q11.y, q11.z, q11.w};
    if constexpr (SPLIT) {
      const size_t s_lo = static_cast<size_t>(src_c8 >> 1) * h * w * 8;
      const uint4 l00 = __ldg(reinterpret_cast<const uint4*>(base + s_lo + (static_cast<size_t>(y0) * w + x0) * 8));
      const uint4 l01 = __ldg(reinterpret_cast<const uint4*>(base + s_lo + (static_cast<size_t>(y0) * w + x1) * 8));
      const uint4 l10 = __ldg(reinterpret_cast<const uint4*>(base + s_lo + (static_cast<size_t>(y1) * w + x0) * 8));
      const uint4 l11 = __ldg(reinterpret_cast<const uint4*>(base + s_lo + (static_cast<size_t>(y1) * w + x1) * 8));
      float v00[8], v01[8], v10[8], v11[8], t8[8], r[8];
      unpack8(q00, v00), unpack8(q01, v01), unpack8(q10, v10), unpack8(q11, v11);
      unpack8(l00, t8);
#pragma unroll
      for (int j = 0; j < 8; ++j) v00[j] += t8[j];
      unpack8(l01, t8);
#pragma unroll
      for (int j = 0; j < 8; ++j) v01[j] += t8[j];
      unpack8(l10, t8);
#pragma unroll
      for (int j = 0; j < 8; ++j) v10[j] += t8[j];
      unpack8(l11, t8);
#pragma unroll
      for (int j = 0; j < 8; ++j) v11[j] += t8[j];
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = hy * (hx * v00[j] + lx * v01[j]) + ly * (hx * v10[j] + lx * v11[j]);
      uint4 oh, ol;
      split8(r, oh, ol);
      __nv_bfloat16* op = dst + ((b * dst_c8 + g) * static_cast<size_t>(ho) * wo + static_cast<size_t>(oy) * wo + ox) * 8;
      *reinterpret_cast<uint4*>(op) = oh;
      *reinterpret_cast<uint4*>(op + static_cast<size_t>(dst_c8 >> 1) * ho * wo * 8) = ol;
      continue;
    }
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 v00 = *reinterpret_cast<const __nv_bfloat162*>(&a[j]), v01 = *reinterpret_cast<const __nv_bfloat162*>(&bq[j]);
      const __nv_bfloat162 v10 = *reinterpret_cast<const __nv_bfloat162*>(&c[j]), v11 = *reinterpret_cast<const __nv_bfloat162*>(&dq[j]);
      const float lo = hy * (hx * __low2float(v00) + lx * __low2float(v01)) + ly * (hx * __low2float(v10) + lx * __low2float(v11));
      const float hi = hy * (hx * __high2float(v00) + lx * __high2float(v01)) + ly * (hx * __high2float(v10) + lx * __high2float(v11));
      __nv_bfloat162 r = __floats2bfloat162_rn(lo, hi);
      o[j] = *reinterpret_cast<uint32_t*>(&r);
    }
    *reinterpret_cast<uint4*>(dst + ((b * dst_c8 + g) * static_cast<size_t>(ho) * wo + static_cast<size_t>(oy) * wo + ox) * 8) =
        make_uint4(o[0], o[1], o[2], o[3]);
  }
}

}  // namespace stcd
