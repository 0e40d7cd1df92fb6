// Bandwidth kernels around the GEMM path: input packing (fp32 NCHW -> bf16 NHWC) and the
// evaluator's binarise + confusion-matrix histogram (K9).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stcd_b200.h"
#include "ptx.cuh"

namespace stcd {

// mma.sync m16n8k16 bf16 -> fp32 (the small tensor-core tiles of the attention and SegCD-head kernels)
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}



// x1, x2: fp32 NCHW [n_valid, cin, h, w] -> dst bf16 [2*chunk][c8][h][w][8] (c8 = 1 or 2 channel
// groups); channels >= cin are zero; T1 images occupy [0, chunk), T2 images [chunk, 2*chunk).
// One thread per pixel: reads are coalesced per channel plane, each thread writes one 16-byte
// pixel chunk per channel group (a warp writes 512 contiguous bytes).
__global__ void __launch_bounds__(256) input_pack_kernel(const float* __restrict__ x1, const float* __restrict__ x2,
                                                         __nv_bfloat16* __restrict__ dst, int chunk, int n_valid,
                                                         int cin, int c8, int hw, int split) {
  const size_t total = static_cast<size_t>(2) * chunk * hw;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(i / hw);
    const int pix = static_cast<int>(i - static_cast<size_t>(n) * hw);
    const int s = n / chunk, b = n - s * chunk;
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) v[c] = 0.f;
    if (b < n_valid) {
      const float* src = (s ? x2 : x1) + static_cast<size_t>(b) * cin * hw + pix;
#pragma unroll
      for (int c = 0; c < 16; ++c)
        if (c < cin) v[c] = __ldg(src + static_cast<size_t>(c) * hw);
      if (split) {     // split precision: channels [8, 16) hold the lo parts x - bf16(x) of channels [0, 8)
#pragma unroll
        for (int c = 0; c < 8; ++c) v[8 + c] = v[c] - __bfloat162float(__float2bfloat16_rn(v[c]));
      }
    }
    uint32_t w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      w[j] = *reinterpret_cast<uint32_t*>(&h);
    }
    __nv_bfloat16* o = dst + (static_cast<size_t>(n) * c8 * hw + pix) * 8;
    *reinterpret_cast<uint4*>(o) = make_uint4(w[0], w[1], w[2], w[3]);
    if (c8 > 1) *reinterpret_cast<uint4*>(o + static_cast<size_t>(hw) * 8) = make_uint4(w[4], w[5], w[6], w[7]);
  }
}

// The same for cin <= 4 with four consecutive pixels per thread (hw % 4 == 0): one 16-byte load per channel plane and 64
// contiguous bytes stored.  The one-pixel kernel keeps 12 bytes per thread in flight -- 24 KB per SM, 2.1 TB/s for the whole
// chip at DRAM latency: 110 us for 128 images of 256 x 256 against a 36 us floor (round-2 floor table).
template <int CIN>
__global__ void __launch_bounds__(256) input_pack4_kernel(const float* __restrict__ x1, const float* __restrict__ x2,
                                                          __nv_bfloat16* __restrict__ dst, int chunk, int n_valid, int c8, int hw) {
  const int hw4 = hw >> 2;
  const size_t total = static_cast<size_t>(2) * chunk * hw4;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(i / hw4);
    const int pix = static_cast<int>(i - static_cast<size_t>(n) * hw4) << 2;
    const int s = n / chunk, b = n - s * chunk;
    float4 v[CIN];
#pragma unroll
    for (int c = 0; c < CIN; ++c) v[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b < n_valid) {
      const float* src = (s ? x2 : x1) + static_cast<size_t>(b) * CIN * hw + pix;
#pragma unroll
      for (int c = 0; c < CIN; ++c) v[c] = __ldg(reinterpret_cast<const float4*>(src + static_cast<size_t>(c) * hw));
    }
    uint4 o4[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float f[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < CIN; ++c) f[c] = q == 0 ? v[c].x : q == 1 ? v[c].y : q == 2 ? v[c].z : v[c].w;
      o4[q] = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), 0u, 0u);
    }
    __nv_bfloat16* o = dst + (static_cast<size_t>(n) * c8 * hw + pix) * 8;
    st_global_256(o, o4[0], o4[1]);
    st_global_256(o + 16, o4[2], o4[3]);
    for (int g = 1; g < c8; ++g) {      // stored channel groups beyond the first are zero
      __nv_bfloat16* z = o + static_cast<size_t>(g) * hw * 8;
      const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
      st_global_256(z, zero, zero);
      st_global_256(z + 16, zero, zero);
    }
  }
}

// ------------------------------------------------------------------------------------------
// uint8 input pipeline (SURVEY.md §8(f)-1): the reference's CD_Dataset (data/dataset.py:196-203) turns uint8 HWC
// RGB into normalised fp32 CHW on the host -- ToTensor (x / 255) then Normalize ((x - mean) / std) -- and ships
// 12 B per pixel-image over PCIe.  These variants take the uint8 HWC images themselves (3 B per pixel-image) and
// evaluate the reference's fp32 expression with IEEE ops before the bf16 rounding, so the packed tensor is
// bit-identical to packing the host-normalised fp32 input.
struct NormParams {
  float mean[4], stdv[4];
};

__device__ __forceinline__ float norm_u8(uint8_t u, float mean, float stdv) {
  return __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(u), 255.0f), mean), stdv);
}

// x1, x2: uint8 HWC [n_valid][h][w][CIN] -> dst bf16 [2*chunk][c8][h][w][8]
template <int CIN>
__global__ void __launch_bounds__(256) input_pack_u8_kernel(const uint8_t* __restrict__ x1, const uint8_t* __restrict__ x2,
                                                            __nv_bfloat16* __restrict__ dst, int chunk, int n_valid, int c8,
                                                            int hw, const NormParams np) {
  const size_t total = static_cast<size_t>(2) * chunk * hw;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(i / hw);
    const int pix = static_cast<int>(i - static_cast<size_t>(n) * hw);
    const int s = n / chunk, b = n - s * chunk;
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) v[c] = 0.f;
    if (b < n_valid) {
      const uint8_t* src = (s ? x2 : x1) + (static_cast<size_t>(b) * hw + pix) * CIN;
#pragma unroll
      for (int c = 0; c < CIN; ++c) v[c] = norm_u8(__ldg(src + c), np.mean[c], np.stdv[c]);
    }
    uint32_t w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      w[j] = *reinterpret_cast<uint32_t*>(&h);
    }
    __nv_bfloat16* o = dst + (static_cast<size_t>(n) * c8 * hw + pix) * 8;
    *reinterpret_cast<uint4*>(o) = make_uint4(w[0], w[1], w[2], w[3]);
    if (c8 > 1) *reinterpret_cast<uint4*>(o + static_cast<size_t>(hw) * 8) = make_uint4(w[4], w[5], w[6], w[7]);
  }
}

// space-to-depth variant: uint8 HWC [n_valid][2h][2w][CIN] -> dst bf16 [2*chunk][2][h][w][8], channel (py*2+px)*CIN + c
template <int CIN>
__global__ void __launch_bounds__(256) input_pack_s2d_u8_kernel(const uint8_t* __restrict__ x1, const uint8_t* __restrict__ x2,
                                                                __nv_bfloat16* __restrict__ dst, int chunk, int n_valid, int h,
                                                                int w, const NormParams np) {
  const int hw = h * w;
  const size_t total = static_cast<size_t>(2) * chunk * hw;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(i / hw);
    const int pix = static_cast<int>(i - static_cast<size_t>(n) * hw);
    const int y = pix / w, x = pix - y * w;
    const int s = n / chunk, b = n - s * chunk;
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) v[c] = 0.f;
    if (b < n_valid) {
      const uint8_t* src = (s ? x2 : x1) + ((static_cast<size_t>(b) * 2 * h + 2 * y) * (2 * w) + 2 * x) * CIN;
#pragma unroll
      for (int py = 0; py < 2; ++py)
#pragma unroll
        for (int px = 0; px < 2; ++px)
#pragma unroll
          for (int c = 0; c < CIN; ++c)
            v[(py * 2 + px) * CIN + c] = norm_u8(__ldg(src + (static_cast<size_t>(py) * 2 * w + px) * CIN + c), np.mean[c], np.stdv[c]);
    }
    uint32_t wd[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      __nv_bfloat162 hv = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      wd[j] = *reinterpret_cast<uint32_t*>(&hv);
    }
    __nv_bfloat16* o = dst + (static_cast<size_t>(n) * 2 * hw + pix) * 8;
    *reinterpret_cast<uint4*>(o) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
    *reinterpret_cast<uint4*>(o + static_cast<size_t>(hw) * 8) = make_uint4(wd[4], wd[5], wd[6], wd[7]);
  }
}

// ------------------------------------------------------------------------------------------
// K9: pred/label -> confusion matrix.  cm[g*K + p] += #{label == g && pred == p}
// (rows = ground truth, cols = prediction: train_stcd.py:576-578).
// Thread-local counters -> warp REDUX -> one shared-memory row per warp -> 64-bit global
// atomics, one set per CTA.  Integer arithmetic throughout: bit-exact.

__device__ __forceinline__ int binarise_sigmoid_gt(float x, float thr) {
  // the reference's fp32 expression, evaluated with IEEE ops: sigmoid(x) > thr (train_stcd.py:477,483)
  const float s = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x)));
  return s > thr ? 1 : 0;
}

template <int PK>
__device__ __forceinline__ int pred_at(const void* pred, size_t n, size_t i, size_t pix, float thr) {
  if (PK == STCD_PRED_ARGMAX2) {
    const float* p = static_cast<const float*>(pred) + n * 2 * pix + i;
    return (__ldg(p + pix) > __ldg(p)) ? 1 : 0;  // torch.argmax: first max wins ties -> class 0
  } else if (PK == STCD_PRED_SIGMOID_GT) {
    return binarise_sigmoid_gt(__ldg(static_cast<const float*>(pred) + n * pix + i), thr);
  } else if (PK == STCD_PRED_RAW_GE) {
    return (__ldg(static_cast<const float*>(pred) + n * pix + i) >= thr) ? 1 : 0;
  } else if (PK == STCD_PRED_U8) {
    return __ldg(static_cast<const uint8_t*>(pred) + n * pix + i);
  } else if (PK == STCD_PRED_U8_GE1) {
    return __ldg(static_cast<const uint8_t*>(pred) + n * pix + i) >= 1 ? 1 : 0;
  } else if (PK == STCD_PRED_I32) {
    return __ldg(static_cast<const int32_t*>(pred) + n * pix + i);
  } else {
    return static_cast<int>(__ldg(static_cast<const long long*>(pred) + n * pix + i));
  }
}

template <int PK>
__device__ __forceinline__ void pred4_at(const void* pred, size_t n, size_t i, size_t pix, float thr, int (&out)[4]) {
  // i % 4 == 0, pix % 4 == 0, base pointers 16-byte aligned
  if (PK == STCD_PRED_ARGMAX2) {
    const float* p = static_cast<const float*>(pred) + n * 2 * pix + i;
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + pix));
    out[0] = b.x > a.x;
    out[1] = b.y > a.y;
    out[2] = b.z > a.z;
    out[3] = b.w > a.w;
  } else if (PK == STCD_PRED_SIGMOID_GT || PK == STCD_PRED_RAW_GE) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(static_cast<const float*>(pred) + n * pix + i));
    const float x[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) out[j] = (PK == STCD_PRED_SIGMOID_GT) ? binarise_sigmoid_gt(x[j], thr) : (x[j] >= thr);
  } else if (PK == STCD_PRED_U8 || PK == STCD_PRED_U8_GE1) {
    const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(pred) + n * pix + i));
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int u = (w >> (8 * j)) & 0xff;
      out[j] = (PK == STCD_PRED_U8_GE1) ? (u >= 1 ? 1 : 0) : u;
    }
  } else if (PK == STCD_PRED_I32) {
    const int4 a = __ldg(reinterpret_cast<const int4*>(static_cast<const int32_t*>(pred) + n * pix + i));
    out[0] = a.x;
    out[1] = a.y;
    out[2] = a.z;
    out[3] = a.w;
  } else {
    const longlong2* p = reinterpret_cast<const longlong2*>(static_cast<const long long*>(pred) + n * pix + i);
    const longlong2 a = __ldg(p), b = __ldg(p + 1);
    out[0] = static_cast<int>(a.x);
    out[1] = static_cast<int>(a.y);
    out[2] = static_cast<int>(b.x);
    out[3] = static_cast<int>(b.y);
  }
}

template <int LK>
__device__ __forceinline__ long long label_at(const void* label, size_t idx) {
  if (LK == STCD_LABEL_I64) return __ldg(static_cast<const long long*>(label) + idx);
  if (LK == STCD_LABEL_U8) return __ldg(static_cast<const uint8_t*>(label) + idx);
  if (LK == STCD_LABEL_U8_GE1) return __ldg(static_cast<const uint8_t*>(label) + idx) >= 1 ? 1 : 0;
  return __ldg(static_cast<const int32_t*>(label) + idx);
}
template <int LK>
__device__ __forceinline__ void label4_at(const void* label, size_t idx, long long (&out)[4]) {
  if (LK == STCD_LABEL_I64) {
    const longlong2* p = reinterpret_cast<const longlong2*>(static_cast<const long long*>(label) + idx);
    const longlong2 a = __ldg(p), b = __ldg(p + 1);
    out[0] = a.x;
    out[1] = a.y;
    out[2] = b.x;
    out[3] = b.y;
  } else if (LK == STCD_LABEL_U8 || LK == STCD_LABEL_U8_GE1) {
    const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(label) + idx));
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t u = (w >> (8 * j)) & 0xff;
      out[j] = (LK == STCD_LABEL_U8_GE1) ? (u >= 1 ? 1 : 0) : u;
    }
  } else {
    const int4 a = __ldg(reinterpret_cast<const int4*>(static_cast<const int32_t*>(label) + idx));
    out[0] = a.x;
    out[1] = a.y;
    out[2] = a.z;
    out[3] = a.w;
  }
}

// num_class == 2 fast path. `vec` = 1 when pix % 4 == 0 and all pointers are 16-byte aligned.
template <int PK, int LK>
__global__ void __launch_bounds__(256) confusion2_kernel(const void* __restrict__ pred, const void* __restrict__ label,
                                                         size_t n_img, size_t pix, float thr, int vec,
                                                         unsigned long long* __restrict__ cm,
                                                         uint8_t* __restrict__ pred_out) {
  uint32_t c[4] = {0, 0, 0, 0};
  const size_t tid = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t nthr = static_cast<size_t>(gridDim.x) * blockDim.x;
  if (vec) {
    const size_t qpi = pix >> 2, nq = n_img * qpi;
    for (size_t q = tid; q < nq; q += nthr) {
      const size_t n = q / qpi, i = (q - n * qpi) << 2;
      int pr[4];
      long long lb[4];
      pred4_at<PK>(pred, n, i, pix, thr, pr);
      label4_at<LK>(label, n * pix + i, lb);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const bool ok = (lb[j] >= 0) && (lb[j] < 2) && (pr[j] >= 0) && (pr[j] < 2);
        const int bin = static_cast<int>(lb[j]) * 2 + pr[j];
#pragma unroll
        for (int b = 0; b < 4; ++b) c[b] += (ok && bin == b) ? 1u : 0u;
      }
      if (pred_out != nullptr) {
        const uint32_t w = (pr[0] & 0xff) | ((pr[1] & 0xff) << 8) | ((pr[2] & 0xff) << 16) | ((pr[3] & 0xff) << 24);
        *reinterpret_cast<uint32_t*>(pred_out + n * pix + i) = w;
      }
    }
  } else {
    const size_t ne = n_img * pix;
    for (size_t e = tid; e < ne; e += nthr) {
      const size_t n = e / pix, i = e - n * pix;
      const int pr = pred_at<PK>(pred, n, i, pix, thr);
      const long long lb = label_at<LK>(label, e);
      const bool ok = (lb >= 0) && (lb < 2) && (pr >= 0) && (pr < 2);
      const int bin = static_cast<int>(lb) * 2 + pr;
#pragma unroll
      for (int b = 0; b < 4; ++b) c[b] += (ok && bin == b) ? 1u : 0u;
      if (pred_out != nullptr) pred_out[e] = static_cast<uint8_t>(pr);
    }
  }
  __shared__ uint32_t wsum[8][4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    const uint32_t s = __reduce_add_sync(0xffffffffu, c[b]);
    if (lane == 0) wsum[warp][b] = s;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    unsigned long long s = 0;
    for (int w = 0; w < (blockDim.x >> 5); ++w) s += wsum[w][threadIdx.x];
    if (s) atomicAdd(cm + threadIdx.x, s);
  }
}

// Pseudo-label masks (train_stcd.py:176-196): mask = on_value where the binarised prediction is 1, else 0.
// HBM-bound: 4 (or 8) B read + 1 B written per pixel.
template <int PK>
__global__ void __launch_bounds__(256) binarise_mask_kernel(const void* __restrict__ logits, size_t n_img, size_t pix, float thr,
                                                            int on_value, uint8_t* __restrict__ mask) {
  const size_t ne = n_img * pix;
  for (size_t e = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; e < ne;
       e += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t n = e / pix, i = e - n * pix;
    mask[e] = pred_at<PK>(logits, n, i, pix, thr) ? static_cast<uint8_t>(on_value) : static_cast<uint8_t>(0);
  }
}

// generic num_class <= 32 (class-id predictions only): shared-memory histogram per CTA.
template <int PK, int LK>
__global__ void __launch_bounds__(256) confusionK_kernel(const void* __restrict__ pred, const void* __restrict__ label,
                                                         size_t n_img, size_t pix, int K,
                                                         unsigned long long* __restrict__ cm) {
  __shared__ uint32_t hist[32 * 32];
  for (int i = threadIdx.x; i < K * K; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  const size_t ne = n_img * pix;
  for (size_t e = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; e < ne;
       e += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t n = e / pix, i = e - n * pix;
    const int pr = pred_at<PK>(pred, n, i, pix, 0.f);
    const long long lb = label_at<LK>(label, e);
    if (lb >= 0 && lb < K && pr >= 0 && pr < K) atomicAdd(&hist[static_cast<int>(lb) * K + pr], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < K * K; i += blockDim.x)
    if (hist[i]) atomicAdd(cm + i, static_cast<unsigned long long>(hist[i]));
}


// ------------------------------------------------------------------------------------------
// K7: SNUNet ECAM tail (models/SNUNet.py:144-149) over the four level-0 node outputs x_k
// (bf16 [img][C/8][h][w][8] each):
//   out   = cat(x_0..x_3)                    (4C channels)
//   intra = x_0 + x_1 + x_2 + x_3            (C channels)
//   ca    = sigmoid(fc2(relu(fc1(avg(out)))) + fc2(relu(fc1(max(out)))))       [4C]   (ChannelAttention, :46-59)
//   ca1   = the same block with its own weights on intra                       [C]
//   y     = conv_final(ca * (out + ca1.repeat(4)))                             [n_class]
// Pass 1 (ecam_stats_kernel) reduces sum/max per (image, channel) into per-block partials (fixed
// order: deterministic); pass 2 (ecam_head_kernel) finishes the reduction, runs the two tiny MLPs
// and applies the per-image 1x1 head  y = sum_c (Wf[k,c] ca[c]) out[c] + (bf[k] + sum_c Wf[k,c] ca[c] ca1[c % C]).
// Both are HBM-bound: each reads the 4C bf16 channels of every pixel once.

struct EcamParams {
  const __nv_bfloat16* src[4];
  int32_t c;         // channels per source (multiple of 8, <= 64)
  int32_t hw;        // pixels per image
  int32_t n_img;     // images in the workspace tensors (chunk)
  int32_t n_valid;   // images to write
  int32_t n_class;   // <= 4
  int32_t r, r1;     // hidden units of ca / ca1 (<= 16)
  int32_t ranges;    // partial blocks per image (pass 1 grid.x)
  float* partial;    // [n_img][ranges][2][5C]: sums then maxes; index k*C + ch for out, 4C + ch for intra
  const float* ca_fc1;   // [r][4C]
  const float* ca_fc2;   // [4C][r]
  const float* ca1_fc1;  // [r1][C]
  const float* ca1_fc2;  // [C][r1]
  const float* w_final;  // [n_class][4C]
  const float* b_final;  // [n_class]
  float* out;            // fp32 NCHW [n_valid][n_class][hw]
  int32_t split;         // split precision: every source holds 2 * c/8 channel groups (hi plane, lo plane); value = hi + lo
};

__device__ __forceinline__ void unpack8_bf16_f(uint4 q, float* v) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
    v[2 * j] = __low2float(h);
    v[2 * j + 1] = __high2float(h);
  }
}


// ------------------------------------------------------------------------------------------
// Space-to-depth input pack for the 7x7 stride-2 ResNet stem: x1, x2 fp32 NCHW [n_valid, cin, 2h, 2w]
// -> dst bf16 [2*chunk][2][h][w][8], channel (py*2 + px)*cin + c = x[c][2y + py][2x + px] (4*cin <= 16).
// One thread per half-resolution pixel: each (c, py) row is read as one float2, so a warp reads 256
// contiguous bytes per row and writes 2 x 512 contiguous bytes.  HBM-bound: 16*cin B read + 32 B written.
// SPLIT: dst is [2*chunk][4][h][w][8], the hi plane bf16(x) in channels [0, 16) (same order) and the lo plane bf16(x - hi) in
// [16, 32).
template <int CIN, bool SPLIT>
__global__ void __launch_bounds__(256) input_pack_s2d_kernel(const float* __restrict__ x1, const float* __restrict__ x2,
                                                             __nv_bfloat16* __restrict__ dst, int chunk, int n_valid,
                                                             int h, int w) {
  constexpr int cin = CIN;
  const int hw = h * w;
  const size_t total = static_cast<size_t>(2) * chunk * hw;
  const size_t plane = static_cast<size_t>(4) * hw;   // full-resolution channel plane
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(i / hw);
    const int pix = static_cast<int>(i - static_cast<size_t>(n) * hw);
    const int y = pix / w, x = pix - y * w;
    const int s = n / chunk, b = n - s * chunk;
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) v[c] = 0.f;
    if (b < n_valid) {
      const float* src = (s ? x2 : x1) + static_cast<size_t>(b) * cin * plane + static_cast<size_t>(2 * y) * (2 * w) + 2 * x;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (c < cin) {
#pragma unroll
          for (int py = 0; py < 2; ++py) {
            const float2 q = __ldg(reinterpret_cast<const float2*>(src + c * plane + static_cast<size_t>(py) * (2 * w)));
            v[(py * 2 + 0) * cin + c] = q.x;
            v[(py * 2 + 1) * cin + c] = q.y;
          }
        }
      }
    }
    uint32_t wd[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      __nv_bfloat162 hv = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      wd[j] = *reinterpret_cast<uint32_t*>(&hv);
    }
    __nv_bfloat16* o = dst + (static_cast<size_t>(n) * (SPLIT ? 4 : 2) * hw + pix) * 8;
    *reinterpret_cast<uint4*>(o) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
    *reinterpret_cast<uint4*>(o + static_cast<size_t>(hw) * 8) = make_uint4(wd[4], wd[5], wd[6], wd[7]);
    if constexpr (SPLIT) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const __nv_bfloat162 hv = *reinterpret_cast<const __nv_bfloat162*>(&wd[j]);
        const __nv_bfloat162 lv = __floats2bfloat162_rn(v[2 * j] - __low2float(hv), v[2 * j + 1] - __high2float(hv));
        wd[j] = *reinterpret_cast<const uint32_t*>(&lv);
      }
      *reinterpret_cast<uint4*>(o + static_cast<size_t>(2) * hw * 8) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
      *reinterpret_cast<uint4*>(o + static_cast<size_t>(3) * hw * 8) = make_uint4(wd[4], wd[5], wd[6], wd[7]);
    }
  }
}

// ------------------------------------------------------------------------------------------
// MaxPool2d(3, stride 2, padding 1) over a map stored space-to-depth: src bf16 [n][4*c8][h][w][8] (group
// cls*c8 + g, cls = py*2 + px, holds full-res pixel (2y + py, 2x + px)) -> dst bf16 [n][c8][h][w][8].
// out(y, x) = max over full-res rows 2y-1..2y+1, cols 2x-1..2x+1 = parity-1 rows y-1 and y, parity-0 row y.
// One thread per (pixel, 8-channel group); max on packed bf16 is exact.  HBM-bound: 4 reads + 1 write of
// 16 B per thread at the algorithmic level (the 9 loads hit L1/L2 for the shared neighbours).
__device__ __forceinline__ uint4 max8_bf16(uint4 a, uint4 b) {
  uint4 r;
  const __nv_bfloat162 x0 = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a.x), *reinterpret_cast<const __nv_bfloat162*>(&b.x));
  const __nv_bfloat162 x1 = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a.y), *reinterpret_cast<const __nv_bfloat162*>(&b.y));
  const __nv_bfloat162 x2 = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a.z), *reinterpret_cast<const __nv_bfloat162*>(&b.z));
  const __nv_bfloat162 x3 = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a.w), *reinterpret_cast<const __nv_bfloat162*>(&b.w));
  r.x = *reinterpret_cast<const uint32_t*>(&x0);
  r.y = *reinterpret_cast<const uint32_t*>(&x1);
  r.z = *reinterpret_cast<const uint32_t*>(&x2);
  r.w = *reinterpret_cast<const uint32_t*>(&x3);
  return r;
}

// SPLIT: src stores 8c channels (hi of class k at k*c, lo at 4c + k*c), dst 2c (hi, then lo at dst_c8/2 groups).  The max runs
// over the fp32 values hi + lo (first maximum wins, in the order below) and the winner's (hi, lo) pair is copied: a selection,
// so nothing is rounded.
template <bool SPLIT>
__global__ void __launch_bounds__(256) maxpool3x3s2_s2d_kernel(const __nv_bfloat16* __restrict__ src,
                                                               __nv_bfloat16* __restrict__ dst, int n_img, int c8, int dst_c8,
                                                               int h, int w) {
  const int hw = h * w;
  const size_t total = static_cast<size_t>(n_img) * c8 * hw;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int pix = static_cast<int>(i % hw);
    const size_t r = i / hw;
    const int g = static_cast<int>(r % c8);
    const int n = static_cast<int>(r / c8);
    const int y = pix / w, x = pix - y * w;
    const __nv_bfloat16* base = src + (static_cast<size_t>(n) * (SPLIT ? 8 : 4) * c8 + g) * hw * 8;
    const size_t cls = static_cast<size_t>(c8) * hw * 8;     // stride between parity classes
    auto ld = [&](int k, int yy, int xx) { return __ldg(reinterpret_cast<const uint4*>(base + k * cls + (static_cast<size_t>(yy) * w + xx) * 8)); };
    if constexpr (SPLIT) {
      float bh[8], bl[8], bv[8];
      auto take = [&](int k, int yy, int xx, bool first) {
        float hv[8], lv[8];
        unpack8_bf16_f(ld(k, yy, xx), hv);
        unpack8_bf16_f(ld(4 + k, yy, xx), lv);          // lo plane of class k
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float v = hv[j] + lv[j];
          if (first || v > bv[j]) {
            bv[j] = v;
            bh[j] = hv[j];
            bl[j] = lv[j];
          }
        }
      };
      take(0, y, x, true);
      take(1, y, x, false);
      take(2, y, x, false);
      take(3, y, x, false);
      if (x > 0) {
        take(1, y, x - 1, false);
        take(3, y, x - 1, false);
      }
      if (y > 0) {
        take(2, y - 1, x, false);
        take(3, y - 1, x, false);
        if (x > 0) take(3, y - 1, x - 1, false);
      }
      uint32_t wh[4], wl[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        wh[j] = pack_bf16x2(bh[2 * j], bh[2 * j + 1]);       // exact: bf16 values
        wl[j] = pack_bf16x2(bl[2 * j], bl[2 * j + 1]);
      }
      __nv_bfloat16* o = dst + ((static_cast<size_t>(n) * dst_c8 + g) * hw + pix) * 8;
      *reinterpret_cast<uint4*>(o) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
      *reinterpret_cast<uint4*>(o + static_cast<size_t>(dst_c8 >> 1) * hw * 8) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
      continue;
    }
    uint4 m = ld(0, y, x);                       // (2y, 2x)
    m = max8_bf16(m, ld(1, y, x));               // (2y, 2x+1)
    m = max8_bf16(m, ld(2, y, x));               // (2y+1, 2x)
    m = max8_bf16(m, ld(3, y, x));               // (2y+1, 2x+1)
    if (x > 0) {
      m = max8_bf16(m, ld(1, y, x - 1));         // (2y, 2x-1)
      m = max8_bf16(m, ld(3, y, x - 1));         // (2y+1, 2x-1)
    }
    if (y > 0) {
      m = max8_bf16(m, ld(2, y - 1, x));         // (2y-1, 2x)
      m = max8_bf16(m, ld(3, y - 1, x));         // (2y-1, 2x+1)
      if (x > 0) m = max8_bf16(m, ld(3, y - 1, x - 1));
    }
    *reinterpret_cast<uint4*>(dst + ((static_cast<size_t>(n) * dst_c8 + g) * hw + pix) * 8) = m;
  }
}

// ------------------------------------------------------------------------------------------
// SegCD tail (decoders/unet/model.py:321-330): head = Conv2d(C, 1, 3, padding=1) applied to d1, d2 and
// |d1 - d2|, then change = min(head(|d1 - d2|), |m1 - m2|).  d: bf16 [2*chunk][C/8][h][w][8] (T1 images then
// T2 images).  A CTA stages a (16+2) x (32+2) pixel halo tile of both streams in shared memory (zero
// padded), each thread computes 2 pixels x 3 convolutions in fp32 with fp32 weights.  HBM-bound at the
// algorithmic level: 2 * C * 2 B read + 12 B written per pixel.
constexpr int kHeadTW = 32, kHeadTH = 16;

// dst[b] = |src[b] - src[chunk + b]| on packed bf16 (fp32 subtract, one rounding): torch.abs(f1 - f2) of FFCTLCD
// (decoders/unet/model.py:412).  Elementwise over 16-byte vectors: layout-agnostic.  HBM-bound: 4 B read + 2 B written.
// signed_diff: dst = (add ? add : 0) + src[T1] - src[T2]  (DTCDSCN's skip terms "decoder(...) + e_x - e_y", models/DTCDSCN.py:296-300)
// SPLIT: every tensor holds hi + lo planes; vec_per_stream counts the hi vectors of a stream and plane_vecs the vectors of one
// plane of one image (hi vector i of image b sits at b * 2 * plane_vecs + i % plane_vecs, its lo vector plane_vecs further).
// The operands are read as hi + lo and the fp32 result is written as hi = bf16(v), lo = bf16(v - hi).
template <bool SPLIT>
__global__ void __launch_bounds__(256) absdiff_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                      size_t vec_per_stream, int signed_diff, const __nv_bfloat16* __restrict__ add,
                                                      int plane_vecs) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < vec_per_stream;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    if constexpr (SPLIT) {
      const size_t b = i / plane_vecs, hv = i + b * plane_vecs;        // hi vector of image b; the lo vector is plane_vecs further
      const size_t sv = 2 * vec_per_stream;                            // vectors per stream, both planes
      const uint4* s4 = reinterpret_cast<const uint4*>(src);
      float a[8], b_[8], al[8], bl[8];
      unpack8_bf16_f(__ldg(s4 + hv), a);
      unpack8_bf16_f(__ldg(s4 + hv + plane_vecs), al);
      unpack8_bf16_f(__ldg(s4 + sv + hv), b_);
      unpack8_bf16_f(__ldg(s4 + sv + hv + plane_vecs), bl);
      float d[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        a[j] += al[j];
        b_[j] += bl[j];
      }
      if (add != nullptr) {
        float c[8], cl[8];
        unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(add) + hv), c);
        unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(add) + hv + plane_vecs), cl);
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] = (c[j] + cl[j]) + a[j];      // reference order: (d + e_x) - e_y
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) d[j] = signed_diff ? a[j] - b_[j] : fabsf(a[j] - b_[j]);
      uint32_t wh[4], wl[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const __nv_bfloat162 h2 = __floats2bfloat162_rn(d[2 * j], d[2 * j + 1]);
        const __nv_bfloat162 l2 = __floats2bfloat162_rn(d[2 * j] - __low2float(h2), d[2 * j + 1] - __high2float(h2));
        wh[j] = *reinterpret_cast<const uint32_t*>(&h2);
        wl[j] = *reinterpret_cast<const uint32_t*>(&l2);
      }
      reinterpret_cast<uint4*>(dst)[hv] = make_uint4(wh[0], wh[1], wh[2], wh[3]);
      reinterpret_cast<uint4*>(dst)[hv + plane_vecs] = make_uint4(wl[0], wl[1], wl[2], wl[3]);
      continue;
    }
    float a[8], b[8];
    unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(src) + i), a);
    unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(src) + vec_per_stream + i), b);
    if (add != nullptr) {
      float c[8];
      unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(add) + i), c);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = (c[j] + a[j]);     // reference order: (d + e_x) - e_y
    }
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float d0 = a[2 * j] - b[2 * j], d1 = a[2 * j + 1] - b[2 * j + 1];
      __nv_bfloat162 hv = signed_diff ? __floats2bfloat162_rn(d0, d1) : __floats2bfloat162_rn(fabsf(d0), fabsf(d1));
      w[j] = *reinterpret_cast<uint32_t*>(&hv);
    }
    reinterpret_cast<uint4*>(dst)[i] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// DIFF = false: the third stream is |d1 - d2| (SegCD); DIFF = true: it is read from `dd`, the decoder output of the
// |f1 - f2| features (FFCTLCD, decoders/unet/model.py:411-413), staged as a third tile.
template <int C8, bool DIFF>
__global__ void __launch_bounds__(256) segcd_head_kernel(const __nv_bfloat16* __restrict__ d, const __nv_bfloat16* __restrict__ dd,
                                                         const float* __restrict__ wgt, float bias, int chunk, int h, int w,
                                                         float* __restrict__ m1, float* __restrict__ m2, float* __restrict__ change) {
  constexpr int PW = kHeadTW + 2, PH = kHeadTH + 2, C = 8 * C8;
  constexpr int NS = DIFF ? 3 : 2;
  extern __shared__ uint4 s_head_dyn[];         // [NS][C8][PH][PW] (58 KB for the 3-stream C=16 instance: dynamic, opt-in)
  uint4 (*s_d)[C8][PH][PW] = reinterpret_cast<uint4 (*)[C8][PH][PW]>(s_head_dyn);
  __shared__ __align__(16) float s_w[9 * C];
  const int n = blockIdx.z;
  const int x0 = blockIdx.x * kHeadTW, y0 = blockIdx.y * kHeadTH;
  const size_t hw = static_cast<size_t>(h) * w;
  for (int i = threadIdx.x; i < 9 * C; i += blockDim.x) s_w[i] = wgt[i];
  // Staging: one warp per (stream, channel group, tile row) -- 2 * C8 * 18 rows of 34 pixels, 16 B each -- with
  // cp.async (zero-fill outside the image): no index divisions, every load of the tile in flight at once.
  {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int row = warp; row < NS * C8 * PH; row += 8) {
      const int py = row % PH;                 // PH = 18: one division per row, warp-uniform
      const int sg = row / PH;
      const int g = sg % C8, sidx = sg / C8;
      const int yy = y0 + py - 1;
      const bool row_ok = (yy >= 0) && (yy < h);
      const __nv_bfloat16* src_row = (sidx < 2 ? d + (static_cast<size_t>(sidx * chunk + n) * C8 + g) * hw * 8
                                               : dd + (static_cast<size_t>(n) * C8 + g) * hw * 8) +
                                     static_cast<size_t>(row_ok ? yy : 0) * w * 8;
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
        const int px = lane + 32 * pass;
        if (px < PW) {
          const int xx = x0 + px - 1;
          const bool ok = row_ok && xx >= 0 && xx < w;
          const void* gp = src_row + static_cast<size_t>(ok ? xx : 0) * 8;
          const uint32_t sp = static_cast<uint32_t>(__cvta_generic_to_shared(&s_d[sidx][g][py][px]));
          const int nbytes = ok ? 16 : 0;      // src-size 0: the 16 destination bytes are zero-filled
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sp), "l"(gp), "r"(nbytes) : "memory");
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  __syncthreads();
  // each thread: 2 vertically adjacent pixels (rows ty0, ty0 + 1).  Per filter column kx the 3 x C weights
  // sit in registers; each of the 4 input rows is loaded and unpacked once and feeds both output rows.
  const int tx = threadIdx.x & 31, ty0 = (threadIdx.x >> 5) * 2;
  float a1[2] = {bias, bias}, a2[2] = {bias, bias}, ad[2] = {bias, bias};
#pragma unroll 1
  for (int kx = 0; kx < 3; ++kx) {
    float wk[3][C];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int j = 0; j < C; j += 4) {
        const float4 q = *reinterpret_cast<const float4*>(&s_w[(ky * 3 + kx) * C + j]);
        wk[ky][j] = q.x;
        wk[ky][j + 1] = q.y;
        wk[ky][j + 2] = q.z;
        wk[ky][j + 3] = q.w;
      }
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      float v1[C], v2[C], v3[DIFF ? C : 1];
#pragma unroll
      for (int g = 0; g < C8; ++g) {
        unpack8_bf16_f(s_d[0][g][ty0 + rr][tx + kx], v1 + 8 * g);
        unpack8_bf16_f(s_d[1][g][ty0 + rr][tx + kx], v2 + 8 * g);
        if (DIFF) unpack8_bf16_f(s_d[NS - 1][g][ty0 + rr][tx + kx], v3 + 8 * g);
      }
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int ky = rr - r;
        if (ky >= 0 && ky < 3) {
#pragma unroll
          for (int j = 0; j < C; ++j) {
            a1[r] = fmaf(v1[j], wk[ky][j], a1[r]);
            a2[r] = fmaf(v2[j], wk[ky][j], a2[r]);
            ad[r] = fmaf(DIFF ? v3[j] : fabsf(v1[j] - v2[j]), wk[ky][j], ad[r]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int yy = y0 + ty0 + r, xx = x0 + tx;
    if (yy < h && xx < w) {
      const size_t o = static_cast<size_t>(n) * hw + static_cast<size_t>(yy) * w + xx;
      m1[o] = a1[r];
      m2[o] = a2[r];
      change[o] = fminf(ad[r], fabsf(a1[r] - a2[r]));
    }
  }
}

// Tensor-core variant of the SegCD head for C = 16 without a feature-level diff tensor (config C3): the three 3x3 convs 16 -> 1 over
// d1, d2 and |d1 - d2| were 432 FMAs per pixel on the FP32 pipe (the kernel's bound).  A warp takes 16 consecutive pixels of a tile
// row; one filter tap is one m16n8k16 step (K = its 16 channels), the A fragments come straight from the staged bf16 tile as 32-bit
// LDS (a warp's loads cover 128 contiguous bytes), the weights sit in column 0 of the B fragment (rounded to bf16 like every conv
// weight of the path), |d1 - d2| is formed on the packed pairs (HSUB2 + abs: the same single rounding as fp32 subtract -> bf16).
// 27 MMAs per 16 pixels; 7 of the 8 output columns are padding, which is irrelevant at this size.
__global__ void __launch_bounds__(256) segcd_head_mma_kernel(const __nv_bfloat16* __restrict__ d, const float* __restrict__ wgt, float bias,
                                                             int chunk, int h, int w, float* __restrict__ m1, float* __restrict__ m2,
                                                             float* __restrict__ change) {
  constexpr int PW = kHeadTW + 2, PH = kHeadTH + 2, C8 = 2, C = 16;
  extern __shared__ uint4 s_head_dyn[];         // [2][C8][PH][PW]
  uint4 (*s_d)[C8][PH][PW] = reinterpret_cast<uint4 (*)[C8][PH][PW]>(s_head_dyn);
  const int n = blockIdx.z;
  const int x0 = blockIdx.x * kHeadTW, y0 = blockIdx.y * kHeadTH;
  const size_t hw = static_cast<size_t>(h) * w;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int row = warp; row < 2 * C8 * PH; row += 8) {
    const int py = row % PH;
    const int sg = row / PH;
    const int g = sg % C8, sidx = sg / C8;
    const int yy = y0 + py - 1;
    const bool row_ok = (yy >= 0) && (yy < h);
    const __nv_bfloat16* src_row = d + (static_cast<size_t>(sidx * chunk + n) * C8 + g) * hw * 8 + static_cast<size_t>(row_ok ? yy : 0) * w * 8;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int px = lane + 32 * pass;
      if (px < PW) {
        const int xx = x0 + px - 1;
        const bool ok = row_ok && xx >= 0 && xx < w;
        const void* gp = src_row + static_cast<size_t>(ok ? xx : 0) * 8;
        const uint32_t sp = static_cast<uint32_t>(__cvta_generic_to_shared(&s_d[sidx][g][py][px]));
        const int nbytes = ok ? 16 : 0;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sp), "l"(gp), "r"(nbytes) : "memory");
      }
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  const int r = lane >> 2, cq = (lane & 3) * 2;
  uint32_t b0[9], b1[9];                        // B fragments: column 0 (lanes with r == 0) holds the tap's 16 weights
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    b0[t] = r == 0 ? pack_bf16x2(__ldg(wgt + t * C + cq), __ldg(wgt + t * C + cq + 1)) : 0u;
    b1[t] = r == 0 ? pack_bf16x2(__ldg(wgt + t * C + 8 + cq), __ldg(wgt + t * C + 8 + cq + 1)) : 0u;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  // A fragments by ldmatrix: a staged pixel is one 16-byte row (8 channels), so the four 8 x 8 matrices of an m16n8k16 A operand
  // -- pixels 0-7 / 8-15 x channel groups 0 / 1 -- are one ldmatrix.x4 (lane l gives row l & 7 of matrix l >> 3) instead of
  // four 32-bit LDS per stream and tap: the kernel ran at 30 % of the HBM roof with the LSU as its busiest pipe.
  const uint32_t sb32 = static_cast<uint32_t>(__cvta_generic_to_shared(s_head_dyn));
  const uint32_t lane_off = static_cast<uint32_t>((((lane >> 4) * PH) * PW + ((lane >> 3) & 1) * 8 + (lane & 7)) * 16);
  auto ldm4 = [&](int s, int py, int px0, uint32_t (&a)[4]) {      // pixels px0 .. px0 + 15 of row py, stream s, 16 channels
    const uint32_t addr = sb32 + static_cast<uint32_t>(((s * C8 * PH + py) * PW + px0) * 16) + lane_off;
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3])
                 : "r"(addr));
  };
#pragma unroll 1
  for (int i = 0; i < (kHeadTW / 16) * kHeadTH / 8; ++i) {         // 32 row segments of 16 pixels, 4 per warp
    const int seg = warp * ((kHeadTW / 16) * kHeadTH / 8) + i;
    const int ty = seg / (kHeadTW / 16), xw = (seg % (kHeadTW / 16)) * 16;
    float c1[4] = {0.f, 0.f, 0.f, 0.f}, c2[4] = {0.f, 0.f, 0.f, 0.f}, cd[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int py = ty + ky;
        uint32_t a1[4], a2[4], ad[4];
        ldm4(0, py, xw + kx, a1);
        ldm4(1, py, xw + kx, a2);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const __nv_bfloat162 df = __habs2(__hsub2(*reinterpret_cast<const __nv_bfloat162*>(&a1[e]), *reinterpret_cast<const __nv_bfloat162*>(&a2[e])));
          ad[e] = *reinterpret_cast<const uint32_t*>(&df);
        }
        mma_bf16_16816(c1, a1, b0[ky * 3 + kx], b1[ky * 3 + kx]);
        mma_bf16_16816(c2, a2, b0[ky * 3 + kx], b1[ky * 3 + kx]);
        mma_bf16_16816(cd, ad, b0[ky * 3 + kx], b1[ky * 3 + kx]);
      }
    }
    if (cq == 0) {                                                 // column 0 of the accumulator tile: rows r and r + 8
      const int yy = y0 + ty;
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int xx = x0 + xw + r + 8 * hrow;
        if (yy < h && xx < w) {
          const float v1 = c1[2 * hrow] + bias, v2 = c2[2 * hrow] + bias, vd = cd[2 * hrow] + bias;
          const size_t o = static_cast<size_t>(n) * hw + static_cast<size_t>(yy) * w + xx;
          m1[o] = v1;
          m2[o] = v2;
          change[o] = fminf(vd, fabsf(v1 - v2));
        }
      }
    }
  }
}

// grid (ranges, C/8, n_img), 256 threads
template <bool SPLIT>
__global__ void __launch_bounds__(256) ecam_stats_kernel(const EcamParams p) {
  const int r = blockIdx.x, g = blockIdx.y, n = blockIdx.z;
  const int per = (p.hw + p.ranges - 1) / p.ranges;
  const int p0 = r * per, p1 = min(p.hw, p0 + per);
  float s[5][8], m[5][8];
#pragma unroll
  for (int k = 0; k < 5; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s[k][j] = 0.f;
      m[k][j] = -INFINITY;
    }
  const int c8s = (p.c >> 3) * (SPLIT ? 2 : 1);     // stored channel groups per source
  const size_t base = (static_cast<size_t>(n) * c8s + g) * p.hw;
  const size_t lo_off = static_cast<size_t>(p.c >> 3) * p.hw * 8;
  for (int px = p0 + threadIdx.x; px < p1; px += blockDim.x) {
    float it[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) it[j] = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float v[8];
      unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(p.src[k] + (base + px) * 8)), v);
      if (SPLIT) {
        float lo[8];
        unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(p.src[k] + (base + px) * 8 + lo_off)), lo);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] += lo[j];
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[k][j] += v[j];
        m[k][j] = fmaxf(m[k][j], v[j]);
        it[j] += v[j];
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s[4][j] += it[j];
      m[4][j] = fmaxf(m[4][j], it[j]);
    }
  }
  __shared__ float sh_s[8][40], sh_m[8][40];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 5; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float a = s[k][j], b = m[k][j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b = fmaxf(b, __shfl_xor_sync(0xffffffffu, b, o));
      }
      if (lane == 0) {
        sh_s[warp][k * 8 + j] = a;
        sh_m[warp][k * 8 + j] = b;
      }
    }
  __syncthreads();
  if (threadIdx.x < 40) {
    float a = 0.f, b = -INFINITY;
    for (int w = 0; w < 8; ++w) {
      a += sh_s[w][threadIdx.x];
      b = fmaxf(b, sh_m[w][threadIdx.x]);
    }
    const int k = threadIdx.x >> 3, j = threadIdx.x & 7;
    const int c5 = 5 * p.c;
    float* dst = p.partial + (static_cast<size_t>(n) * p.ranges + r) * 2 * c5;
    dst[k * p.c + g * 8 + j] = a;
    dst[c5 + k * p.c + g * 8 + j] = b;
  }
}

constexpr int kEcamPixPerBlock = 2048;

// grid (ceil(hw / kEcamPixPerBlock), n_valid), 256 threads
template <bool SPLIT>
__global__ void __launch_bounds__(256) ecam_head_kernel(const EcamParams p) {
  __shared__ float s_avg[320], s_max[320];        // 5C <= 320
  __shared__ float s_hid[4][16];                  // ca: avg, max; ca1: avg, max
  __shared__ float s_ca[256], s_ca1[64];
  __shared__ __align__(16) float s_w[4][256];     // per-image head weights
  __shared__ float s_b[4];
  const int n = blockIdx.y;
  const int c = p.c, c4 = 4 * p.c, c5 = 5 * p.c;
  for (int i = threadIdx.x; i < c5; i += blockDim.x) {
    float a = 0.f, b = -INFINITY;
    for (int r = 0; r < p.ranges; ++r) {
      const float* src = p.partial + (static_cast<size_t>(n) * p.ranges + r) * 2 * c5;
      a += src[i];
      b = fmaxf(b, src[c5 + i]);
    }
    s_avg[i] = a / static_cast<float>(p.hw);
    s_max[i] = b;
  }
  __syncthreads();
  if (threadIdx.x < 2 * p.r) {                    // ca hidden layer: fc1 over the 4C out channels
    const int u = threadIdx.x % p.r, which = threadIdx.x / p.r;
    const float* v = which ? s_max : s_avg;
    float a = 0.f;
    for (int i = 0; i < c4; ++i) a = fmaf(p.ca_fc1[u * c4 + i], v[i], a);
    s_hid[which][u] = fmaxf(a, 0.f);
  } else if (threadIdx.x >= 32 && threadIdx.x < 32 + 2 * p.r1) {   // ca1 hidden layer over the C intra channels
    const int t = threadIdx.x - 32;
    const int u = t % p.r1, which = t / p.r1;
    const float* v = (which ? s_max : s_avg) + c4;
    float a = 0.f;
    for (int i = 0; i < c; ++i) a = fmaf(p.ca1_fc1[u * c + i], v[i], a);
    s_hid[2 + which][u] = fmaxf(a, 0.f);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < c4 + c; i += blockDim.x) {
    if (i < c4) {
      float a = 0.f, b = 0.f;
      for (int u = 0; u < p.r; ++u) {
        a = fmaf(p.ca_fc2[i * p.r + u], s_hid[0][u], a);
        b = fmaf(p.ca_fc2[i * p.r + u], s_hid[1][u], b);
      }
      s_ca[i] = 1.f / (1.f + expf(-(a + b)));
    } else {
      const int j = i - c4;
      float a = 0.f, b = 0.f;
      for (int u = 0; u < p.r1; ++u) {
        a = fmaf(p.ca1_fc2[j * p.r1 + u], s_hid[2][u], a);
        b = fmaf(p.ca1_fc2[j * p.r1 + u], s_hid[3][u], b);
      }
      s_ca1[j] = 1.f / (1.f + expf(-(a + b)));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < p.n_class * c4; i += blockDim.x) {
    const int k = i / c4, ch = i - k * c4;
    s_w[k][ch] = p.w_final[i] * s_ca[ch];
  }
  __syncthreads();
  if (threadIdx.x < p.n_class) {
    float a = p.b_final[threadIdx.x];
    for (int ch = 0; ch < c4; ++ch) a = fmaf(s_w[threadIdx.x][ch], s_ca1[ch % c], a);
    s_b[threadIdx.x] = a;
  }
  __syncthreads();
  const int g8 = c >> 3;
  const int px_end = min(p.hw, (static_cast<int>(blockIdx.x) + 1) * kEcamPixPerBlock);
  for (int px = blockIdx.x * kEcamPixPerBlock + threadIdx.x; px < px_end; px += blockDim.x) {
    float acc[4] = {s_b[0], s_b[1], s_b[2], s_b[3]};
    for (int k = 0; k < 4; ++k) {
      for (int g = 0; g < g8; ++g) {
        float v[8];
        const size_t at = ((static_cast<size_t>(n) * (SPLIT ? 2 * g8 : g8) + g) * p.hw + px) * 8;
        unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(p.src[k] + at)), v);
        if (SPLIT) {     // value = hi plane + lo plane
          float lo[8];
          unpack8_bf16_f(__ldg(reinterpret_cast<const uint4*>(p.src[k] + at + static_cast<size_t>(g8) * p.hw * 8)), lo);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] += lo[j];
        }
        const int ch = k * c + g * 8;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (q < p.n_class) {
            const float4 w0 = *reinterpret_cast<const float4*>(&s_w[q][ch]);
            const float4 w1 = *reinterpret_cast<const float4*>(&s_w[q][ch + 4]);
            acc[q] = fmaf(v[0], w0.x, acc[q]);
            acc[q] = fmaf(v[1], w0.y, acc[q]);
            acc[q] = fmaf(v[2], w0.z, acc[q]);
            acc[q] = fmaf(v[3], w0.w, acc[q]);
            acc[q] = fmaf(v[4], w1.x, acc[q]);
            acc[q] = fmaf(v[5], w1.y, acc[q]);
            acc[q] = fmaf(v[6], w1.z, acc[q]);
            acc[q] = fmaf(v[7], w1.w, acc[q]);
          }
        }
      }
    }
    for (int q = 0; q < p.n_class; ++q) p.out[(static_cast<size_t>(n) * p.n_class + q) * p.hw + px] = acc[q];
  }
}

}  // namespace stcd
