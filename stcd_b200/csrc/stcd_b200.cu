// libstcd_b200.so — plan executor + C-ABI (include/stcd_b200.h).
//
// A plan is a list of fused ops over NHWC bf16 activation tensors living in one device
// workspace.  The host side (stcd_b200/lowering.py) lowers a reference nn.Module state_dict
// into this list; this file owns memory, TMA descriptors and launches.  No CPU fallback: every
// entry point that computes needs an sm_100 device and fails loudly without one.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/stcd_b200.h"
#include "aux_kernels.cuh"
#include "conv_ws.cuh"
#include "graph_kernels.cuh"
#include "transformer_kernels.cuh"
#include "bit_kernels.cuh"
#include "attn_gate_kernels.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                                  \
  do {                                                                                                  \
    cudaError_t e__ = (expr);                                                                           \
    if (e__ != cudaSuccess)                                                                             \
      return fail(STCD_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Tensor {
  int mult, h, w, c, dtype;
  size_t bytes = 0, offset = 0;
  void* ptr = nullptr;
};

struct ConvOp {
  stcd_conv_desc d;
  std::vector<uint16_t> weights;
  std::vector<stcd_chunk> chunks;
  std::vector<stcd_tap> taps;
  std::vector<float> scale, shift, scale2, shift2;
  // device side
  size_t w_off = 0, c_off = 0, t_off = 0, s_off = 0;  // offsets in the constant arena
  stcd::TmapPack tm;
  stcd::ConvParams p;
  dim3 grid;
  size_t smem = 0;
  int mt = 1;
  int occ = 0;                 // CTAs per SM the shared-memory plan was sized for
  uint32_t epi = 0;
  stcd::ConvKernelFn fn = nullptr;
  int threads = 256;           // 256 (four epilogue warps) or 384 (eight)
  long long* trace = nullptr;
};

struct PackOp {
  int dst, cin;
  int s2d = 0;
  int u8 = 0;                 // inputs are uint8 HWC, normalised in the pack kernel
  stcd::NormParams norm;
};

struct PoolOp {
  int src, dst, c;
};

struct GraphOp {
  int src, dst, c, k, dilation, r;
  std::vector<float> relpos;   // [N][M] or empty
  float* relpos_dev = nullptr;
  float* xf = nullptr;         // fp32 [imgs][C][N]
  float* yf = nullptr;         // fp32 [imgs][C][M] (r > 1)
  float* xn = nullptr;         // fp32 [imgs][C][N], L2-normalised nodes
  float* yn = nullptr;         // fp32 [imgs][C][M] (r > 1)
  long long* idx = nullptr;    // [imgs][N][k]
  // tensor-core path: L2-normalised nodes as three bf16 planes in the MMA operand layout + their squared norms
  __nv_bfloat16* xp = nullptr;
  __nv_bfloat16* yp = nullptr; // r > 1
  float* xsq = nullptr;
  float* ysq = nullptr;        // r > 1
};

struct BilinearOp {
  int src, dst, c, scale;
};

struct LayerNormOp {
  int src, dst, dst2, c;
  float eps;
  std::vector<float> gb;   // gamma | beta
  float* gb_dev = nullptr;
};

struct AttentionOp {
  int q, kv, dst, c, heads;
  float scale;
};

struct DWConvOp {
  int src, dst, c, gelu;
  std::vector<float> wb;   // weight [c][9] | bias [c]
  float* wb_dev = nullptr;
};

struct AbsDiffOp {
  int src, dst, c;
  int signed_diff = 0;
  int add = -1;
};

struct GateOp {
  int src, res, dst, dst2, c, hid, mode, ranges;
  std::vector<float> w;      // w1 [hid][c] | w2 [c][hid] | ws [c] (mode 1)
  float* w_dev = nullptr;
  float* partial = nullptr;  // [imgs][ranges][c]
};

struct BitOp {
  int src, dst;
  stcd_bit_desc d;
  std::vector<float> w;        // conv_a | pos | enc | dec
  float* w_dev = nullptr;
  float* tokens = nullptr;     // [2*chunk][L][c]
  float* tok_mixed = nullptr;  // [chunk][2L][c] after the encoder
  size_t coef_smem = 0;
  float* coef = nullptr;       // [2*chunk][n_dec][A | Bm]
  size_t mixer_smem = 0;
};

struct ChanAttnOp {
  int n_src, src[4], stream[4], c[4], dst, c_tot, hid, ranges;
  std::vector<float> w;        // fc1 [hid][C] | fc2^T [hid][C]
  float* w_dev = nullptr;
  float* psum = nullptr;       // [chunk][ranges][c_tot]
  float* pmax = nullptr;
  float* gate = nullptr;       // [chunk][c_tot]
};

struct SpatialGateOp {
  int src, dst, c;
  std::vector<float> w;        // conv [98] | scale [c] | shift [c]
  float* w_dev = nullptr;
  float2* stats = nullptr;     // [mult*chunk][h*w]
};

struct GlGateOp {
  int src, dst, c, ranges;
  int hid = 0;                 // > 0: csam_V20 (channel MLP + two 3x3 spatial convs) instead of Global_Local's gate
  std::vector<float> w;
  float* w_dev = nullptr;
  float* psum = nullptr;
  float* pmax = nullptr;
  float2* stats = nullptr;
};

struct VffmOp {
  int low, high, mixed, local, dst, c, inter, ranges;
  std::vector<float> w;
  float* w_dev = nullptr;
  float* psum = nullptr;
  float* pmax = nullptr;
};

struct SumOp {
  int src[5], n, dst;
};

struct SegHeadOp {
  int src, c, out_ext;
  int diff_src = -1;
  float bias;
  std::vector<float> w;  // [9][c]
  float* w_dev = nullptr;
};

struct EcamOp {
  stcd_ecam_desc d;
  std::vector<float> w;     // ca_fc1 | ca_fc2 | ca1_fc1 | ca1_fc2 | w_final | b_final
  float* w_dev = nullptr;
  float* partial = nullptr;
  stcd::EcamParams p;
  int hw = 0;
};

struct Op {
  int kind;  // 0 conv, 1 input pack, 2 ECAM head, 3 max-pool (space-to-depth source), 4 SegCD head, 5 graph conv, 6 bilinear up, 7 layer norm, 8 attention, 9 dw conv, 10 T1 - T2 (abs or signed), 11 channel gate, 12 sum, 13 BIT token path, 14 channel attention, 15 spatial gate, 16 global-local gate, 17 VFFM
  int idx;
};

}  // namespace

struct stcd_plan {
  int device = 0;
  int chunk = 0;
  int split = 0;             // STCD_PRECISION_SPLIT: every tensor holds a hi and a lo plane, every op runs its split form
  bool finalized = false;
  std::vector<Tensor> tensors;
  std::vector<ConvOp> convs;
  std::vector<PackOp> packs;
  std::vector<EcamOp> ecams;
  std::vector<PoolOp> pools;
  std::vector<SegHeadOp> heads;
  std::vector<GraphOp> graphs;
  std::vector<BilinearOp> bilinears;
  std::vector<LayerNormOp> lns;
  std::vector<AttentionOp> attns;
  std::vector<DWConvOp> dws;
  std::vector<AbsDiffOp> absdiffs;
  std::vector<GateOp> gates;
  std::vector<SumOp> sums;
  std::vector<BitOp> bits;
  std::vector<ChanAttnOp> chan_attns;
  std::vector<SpatialGateOp> spatial_gates;
  std::vector<GlGateOp> gl_gates;
  std::vector<VffmOp> vffms;
  std::vector<Op> ops;
  uint8_t* workspace = nullptr;
  size_t workspace_bytes = 0;
  uint8_t* arena = nullptr;  // weights, K-programs, scale/shift
  size_t arena_bytes = 0;
  int n_ext = 0;
  int in_c = 0, in_h = 0, in_w = 0;
  int in_u8 = 0;  // 1: the plan's inputs are uint8 HWC images (stcd_plan_add_input_pack_u8)
  int pdl = 1;  // programmatic dependent launch between the conv kernels (STCD_PDL=0 disables)
  std::vector<size_t> ext_elems;  // per external output: elements per image
  // host-buffer path
  cudaStream_t s_copy = nullptr, s_comp = nullptr, s_d2h = nullptr;
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
  float* stage_in[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  std::vector<float*> stage_out[2];
  // CUDA graphs of one chunk's launch list, keyed by the caller's pointers (opt-in: STCD_GRAPH=1; see stcd_plan_finalize for
  // the measurement that keeps it off by default).
  struct GraphEntry {
    const void* x1 = nullptr;
    const void* x2 = nullptr;
    int n_valid = 0;
    std::vector<float*> outs;
    cudaGraphExec_t exec = nullptr;
    int seen = 0;               // a key is captured the second time it shows up (pointers that never repeat stay on plain launches)
    uint64_t last_use = 0;
  };
  std::vector<GraphEntry> graph_cache;
  uint64_t graph_clock = 0;
  int graph_mode = 1;           // 0: off; set to 0 for good when a capture or instantiation fails
  cudaStream_t s_capture = nullptr;
};
constexpr size_t kGraphCacheSize = 16;

namespace {

int check_sm100(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(STCD_ERR_NO_DEVICE, "no CUDA device visible: libstcd_b200 has no CPU fallback");
  }
  if (device < 0 || device >= n) return fail(STCD_ERR_INVALID, "device %d out of range (%d visible)", device, n);
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(STCD_ERR_NO_DEVICE, "device %d is sm_%d%d; libstcd_b200 is built for sm_100a only", device, prop.major,
                prop.minor);
  return STCD_OK;
}

int encode_act_map(CUtensorMap* m, void* base, int n, int h, int w, int c, int kc, int sx, int sy, int ex, int ey,
                   int tile_w = stcd::kTileW, int tile_h = stcd::kTileH) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(STCD_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  if (sx == 1 && sy == 1) {
    // (8 ch, x) are contiguous in HBM and in the shared-memory operand layout alike: merge them into
    // one dimension so a box row is (8 + ex) * 16 bytes instead of 16 (TMA cost is per box row).
    cuuint64_t gdim[4] = {(cuuint64_t)w * 8, (cuuint64_t)h, (cuuint64_t)(c / 8), (cuuint64_t)n};
    cuuint64_t gstr[3] = {(cuuint64_t)w * 16, (cuuint64_t)h * w * 16, (cuuint64_t)(c / 8) * h * w * 16};
    cuuint32_t box[4] = {(cuuint32_t)((tile_w + ex) * 8), (cuuint32_t)(tile_h + ey), (cuuint32_t)(kc / 8), 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if (box[0] > 256) return fail(STCD_ERR_INVALID, "halo %d too wide for one TMA box row", ex);
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
      return fail(STCD_ERR_CUDA, "cuTensorMapEncodeTiled(act4 n=%d h=%d w=%d c=%d kc=%d e=%d,%d) -> %d", n, h, w, c, kc, ex, ey, (int)r);
    return STCD_OK;
  }
  // [img][c/8][h][w][8] bf16: dims fastest-first {8, w, h, c/8, img}
  cuuint64_t gdim[5] = {8, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)(c / 8), (cuuint64_t)n};
  cuuint64_t gstr[4] = {16, (cuuint64_t)w * 16, (cuuint64_t)h * w * 16, (cuuint64_t)(c / 8) * h * w * 16};
  cuuint32_t box[5] = {8, (cuuint32_t)((tile_w + ex) * sx), (cuuint32_t)((tile_h + ey) * sy), (cuuint32_t)(kc / 8), 1};
  cuuint32_t estr[5] = {1, (cuuint32_t)sx, (cuuint32_t)sy, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(STCD_ERR_CUDA, "cuTensorMapEncodeTiled(act n=%d h=%d w=%d c=%d kc=%d s=%d,%d e=%d,%d) -> %d", n, h, w, c, kc,
                sx, sy, ex, ey, (int)r);
  return STCD_OK;
}

bool valid_tensor(const stcd_plan* p, int id) { return id >= 0 && id < (int)p->tensors.size(); }

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

int launch_conv(const stcd_plan* plan, const ConvOp& op, int n_valid, float* const* outs, cudaStream_t st) {
  stcd::ConvParams p = op.p;
  p.n_valid = n_valid;
  if (op.d.out_ext >= 0) {
    p.out_f32 = outs[op.d.out_ext];
    if (!p.out_f32) return fail(STCD_ERR_INVALID, "external output %d is NULL", op.d.out_ext);
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = op.grid;
  cfg.blockDim = dim3(op.threads, 1, 1);
  cfg.dynamicSmemBytes = op.smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = plan->pdl ? 1 : 0;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, op.fn, op.tm, p));
  (void)plan;
  return STCD_OK;
}

// Dense dilated kNN, fp32 register-tile kernel (k * dilation > 27, or STCD_KNN_MMA=0)
int launch_knn(const float* xn, const float* yn, const float* relpos, int B, int C, int N, int M, int k, int dilation, long long* idx,
               cudaStream_t st) {
  stcd::knn_graph_kernel<<<dim3((N + stcd::kKnnQ - 1) / stcd::kKnnQ, B), 256, 0, st>>>(xn, yn, relpos, C, N, M, k, dilation, idx);
  CUDA_TRY(cudaGetLastError());
  return STCD_OK;
}

// bytes of the plane + squared-norm workspace of `rows` nodes x C channels for B images (rows padded to 128)
size_t knn_planes_bytes(int B, int C, int rows) {
  return (size_t)B * 3 * stcd::knn_gpad(C) * stcd::knn_rpad(rows, 128) * 16;
}
size_t knn_sq_bytes(int B, int rows) { return (size_t)B * stcd::knn_rpad(rows, 128) * sizeof(float); }

// Tensor-core kNN on pre-split planes (knn_prep_kernel + knn_pipe_kernel).  xf / yf: fp32 [B][C][N] / [B][C][M] (yf NULL: y := x).
// xp / xsq (and yp / ysq when yf is given): zero-initialised workspaces of knn_planes_bytes / knn_sq_bytes.
int launch_knn_pipe(const float* xf, const float* yf, const float* relpos, int B, int C, int N, int M, int k, int dilation,
                    __nv_bfloat16* xp, float* xsq, __nv_bfloat16* yp, float* ysq, long long* idx, cudaStream_t st) {
  const int kd = k * dilation;
  const int G_pad = stcd::knn_gpad(C), NR = stcd::knn_rpad(N, 128), MR = yf ? stcd::knn_rpad(M, 128) : NR, MP = (M + 15) & ~15;
  auto ng = [](int B_, int n_) { return (unsigned)std::max(1, std::min(B_ * ((n_ + 31) / 32), 148 * 16)); };
  stcd::knn_prep_kernel<<<ng(B, N), 256, 0, st>>>(xf, xp, xsq, B, C, N, G_pad, NR);
  if (yf) stcd::knn_prep_kernel<<<ng(B, M), 256, 0, st>>>(yf, yp, ysq, B, C, M, G_pad, MR);
  const size_t smem = (size_t)2 * 3 * 4 * (stcd::kKnnTQ + MP) * 16 + 128;
  const dim3 grid((N + stcd::kKnnTQ - 1) / stcd::kKnnTQ, B);
#define STCD_KNN_PIPE(KD)                                                                                                      \
  do {                                                                                                                         \
    static bool attr_set = false;                                                                                              \
    if (!attr_set) {                                                                                                           \
      CUDA_TRY(cudaFuncSetAttribute(stcd::knn_pipe_kernel<KD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));      \
      attr_set = true;                                                                                                         \
    }                                                                                                                          \
    stcd::knn_pipe_kernel<KD><<<grid, 192, smem, st>>>(xp, xsq, NR, yf ? yp : xp, yf ? ysq : xsq, MR, MP, relpos, C, N, M, k, dilation, idx); \
  } while (0)
  if (kd <= 9) STCD_KNN_PIPE(9);
  else if (kd <= 18) STCD_KNN_PIPE(18);
  else STCD_KNN_PIPE(27);
#undef STCD_KNN_PIPE
  CUDA_TRY(cudaGetLastError());
  return STCD_OK;
}

int run_chunk(stcd_plan* plan, const void* x1v, const void* x2v, int n_valid, float* const* outs, cudaStream_t st,
              cudaEvent_t* ev = nullptr) {
  int op_i = 0;
  const float* x1 = static_cast<const float*>(x1v);
  const float* x2 = static_cast<const float*>(x2v);
  if (ev) CUDA_TRY(cudaEventRecord(ev[0], st));
  for (const Op& o : plan->ops) {
    if (o.kind == 0) {
      int r = launch_conv(plan, plan->convs[o.idx], n_valid, outs, st);
      if (r) return r;
    } else if (o.kind == 2) {
      const EcamOp& e = plan->ecams[o.idx];
      stcd::EcamParams q = e.p;
      q.n_valid = n_valid;
      q.out = outs[e.d.out_ext];
      if (!q.out) return fail(STCD_ERR_INVALID, "external output %d is NULL", e.d.out_ext);
      const dim3 g_stats(q.ranges, q.c / 8, n_valid), g_head((e.hw + stcd::kEcamPixPerBlock - 1) / stcd::kEcamPixPerBlock, n_valid);
      if (q.split) stcd::ecam_stats_kernel<true><<<g_stats, 256, 0, st>>>(q);
      else stcd::ecam_stats_kernel<false><<<g_stats, 256, 0, st>>>(q);
      CUDA_TRY(cudaGetLastError());
      if (q.split) stcd::ecam_head_kernel<true><<<g_head, 256, 0, st>>>(q);
      else stcd::ecam_head_kernel<false><<<g_head, 256, 0, st>>>(q);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 3) {
      const PoolOp& k = plan->pools[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const size_t total = (size_t)td.mult * plan->chunk * (k.c / 8) * td.h * td.w;
      const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
      auto kern = plan->split ? stcd::maxpool3x3s2_s2d_kernel<true> : stcd::maxpool3x3s2_s2d_kernel<false>;
      kern<<<blocks, 256, 0, st>>>((const __nv_bfloat16*)ts.ptr, (__nv_bfloat16*)td.ptr, td.mult * plan->chunk, k.c / 8, td.c / 8, td.h,
                                   td.w);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 5) {
      const GraphOp& k = plan->graphs[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const int B = ts.mult * plan->chunk, N = ts.h * ts.w, M = N / (k.r * k.r);
      auto nb = [](size_t total, int cap) { return (unsigned)std::max<size_t>(1, std::min<size_t>((total + 255) / 256, (size_t)148 * cap)); };
      stcd::unpack_nodes_kernel<<<nb((size_t)B * (k.c / 8) * N, 8), 256, 0, st>>>((const __nv_bfloat16*)ts.ptr, k.xf, B, ts.c / 8, k.c, N);
      const float* y = k.xf;
      if (k.r > 1) {
        stcd::avgpool_nodes_kernel<<<nb((size_t)B * k.c * M, 8), 256, 0, st>>>(k.xf, k.yf, (size_t)B * k.c, ts.h, ts.w, k.r);
        y = k.yf;
      }
      if (k.xp) {      // tensor-core path: normalise + split once, then the pipelined kernel
        int r = launch_knn_pipe(k.xf, k.r > 1 ? k.yf : nullptr, k.relpos_dev, B, k.c, N, M, k.k, k.dilation, k.xp, k.xsq, k.yp, k.ysq, k.idx, st);
        if (r) return r;
      } else {
        auto ng = [](int B_, int n_) { return (unsigned)std::max(1, std::min(B_ * ((n_ + 31) / 32), 148 * 16)); };
        stcd::normalize_nodes_kernel<<<ng(B, N), 256, 0, st>>>(k.xf, k.xn, B, k.c, N);
        if (k.r > 1) stcd::normalize_nodes_kernel<<<ng(B, M), 256, 0, st>>>(k.yf, k.yn, B, k.c, M);
        int r = launch_knn(k.xn, k.r > 1 ? k.yn : k.xn, k.relpos_dev, B, k.c, N, M, k.k, k.dilation, k.idx, st);
        if (r) return r;
      }
      stcd::max_relative_nc8_kernel<<<nb((size_t)B * (k.c / 8) * N, 8), 256, 0, st>>>(k.xf, y, k.idx, B, k.c, N, M, k.k,
                                                                                      (__nv_bfloat16*)td.ptr, td.c / 8);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 10) {
      const AbsDiffOp& k = plan->absdiffs[o.idx];
      const Tensor& td = plan->tensors[k.dst];
      const size_t vecs = td.bytes / 16 / (plan->split ? 2 : 1); // 16-byte (hi) vectors per stream (dst holds one stream)
      const int plane_vecs = (td.c / 16) * td.h * td.w;            // split: vectors of one plane of one image
      auto kern = plan->split ? stcd::absdiff_kernel<true> : stcd::absdiff_kernel<false>;
      kern<<<(unsigned)std::max<size_t>(1, std::min<size_t>((vecs + 255) / 256, 148 * 16)), 256, 0, st>>>(
          (const __nv_bfloat16*)plan->tensors[k.src].ptr, (__nv_bfloat16*)td.ptr, vecs, k.signed_diff,
          k.add >= 0 ? (const __nv_bfloat16*)plan->tensors[k.add].ptr : nullptr, plane_vecs);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 11) {
      const GateOp& k = plan->gates[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const int B = ts.mult * plan->chunk, hw = ts.h * ts.w;
      const int n_items = B * (k.c / 8) * k.ranges;   // one warp each
      (plan->split ? stcd::chan_sum_kernel<true> : stcd::chan_sum_kernel<false>)<<<(n_items + 7) / 8, 256, 0, st>>>(
          (const __nv_bfloat16*)ts.ptr, k.partial, k.c, ts.c / 8, hw, k.ranges, n_items);
      // ~2048 (pixel, channel group) items per CTA: enough CTAs to fill the machine on every level of the pyramid
      const int ppb = std::max(32, std::min(stcd::kGateMaxPix, 2048 / (k.c / 8)));
      const float* w1 = k.w_dev;
      const float* w2 = w1 + (size_t)k.hid * k.c;
      const float* ws = k.mode == 1 ? w2 + (size_t)k.c * k.hid : nullptr;
      (plan->split ? stcd::gate_apply_kernel<true> : stcd::gate_apply_kernel<false>)<<<dim3((hw + ppb - 1) / ppb, B), 256, 0, st>>>(
          (const __nv_bfloat16*)ts.ptr, k.res >= 0 ? (const __nv_bfloat16*)plan->tensors[k.res].ptr : nullptr, (__nv_bfloat16*)td.ptr,
          k.dst2 >= 0 ? (__nv_bfloat16*)plan->tensors[k.dst2].ptr : nullptr, k.partial, w1, w2, ws, k.c, k.hid, ts.c / 8,
          k.res >= 0 ? plan->tensors[k.res].c / 8 : 0, td.c / 8, k.dst2 >= 0 ? plan->tensors[k.dst2].c / 8 : 0, ts.h, ts.w, k.ranges, k.mode,
          ppb);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 14) {
      const ChanAttnOp& k = plan->chan_attns[o.idx];
      const Tensor& td = plan->tensors[k.dst];
      const int B = plan->chunk, hw = td.h * td.w;
      int c_off = 0;
      for (int i = 0; i < k.n_src; ++i) {
        const Tensor& ts = plan->tensors[k.src[i]];
        const __nv_bfloat16* sp = (const __nv_bfloat16*)ts.ptr + (size_t)k.stream[i] * B * ts.c * hw;
        const int n_items = B * (k.c[i] / 8) * k.ranges;
        stcd::chan_stats_kernel<<<(n_items + 7) / 8, 256, 0, st>>>(sp, k.psum, k.pmax, k.c[i], ts.c / 8, hw, k.ranges, n_items, k.c_tot, c_off);
        c_off += k.c[i];
      }
      stcd::ca_fc_kernel<<<dim3((k.c_tot + 255) / 256, B), 256, 0, st>>>(k.psum, k.pmax, k.w_dev, k.w_dev + (size_t)k.hid * k.c_tot, k.gate, k.c_tot, k.hid, hw, k.ranges);
      c_off = 0;
      for (int i = 0; i < k.n_src; ++i) {
        const Tensor& ts = plan->tensors[k.src[i]];
        const __nv_bfloat16* sp = (const __nv_bfloat16*)ts.ptr + (size_t)k.stream[i] * B * ts.c * hw;
        const size_t total = (size_t)B * (k.c[i] / 8) * hw;
        stcd::ca_apply_kernel<<<(unsigned)std::max<size_t>(1, std::min<size_t>((total + 255) / 256, 148 * 16)), 256, 0, st>>>(
            sp, (__nv_bfloat16*)td.ptr, k.gate, B, k.c[i], ts.c / 8, td.c / 8, hw, k.c_tot, c_off);
        c_off += k.c[i];
      }
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 16) {
      const GlGateOp& k = plan->gl_gates[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const int B = ts.mult * plan->chunk, hw = ts.h * ts.w;
      const int n_items = B * (k.c / 8) * k.ranges;
      stcd::chan_stats_kernel<<<(n_items + 7) / 8, 256, 0, st>>>((const __nv_bfloat16*)ts.ptr, k.psum, k.pmax, k.c, ts.c / 8, hw, k.ranges,
                                                                 n_items, k.c, 0);
      stcd::sa_stats_kernel<<<dim3((hw + 255) / 256, B), 256, 0, st>>>((const __nv_bfloat16*)ts.ptr, k.stats, k.c, ts.c / 8, hw);
      const dim3 tg((ts.w + stcd::kSaTW - 1) / stcd::kSaTW, (ts.h + stcd::kSaTH - 1) / stcd::kSaTH, B), tb(stcd::kSaTW, stcd::kSaTH);
      if (k.hid > 0)
        stcd::csam_apply_kernel<<<tg, tb, 0, st>>>((const __nv_bfloat16*)ts.ptr, (__nv_bfloat16*)td.ptr, k.stats, k.psum, k.pmax, k.w_dev, k.c,
                                                   k.hid, ts.c / 8, td.c / 8, ts.h, ts.w, k.ranges);
      else
        stcd::gl_apply_kernel<<<tg, tb, 0, st>>>((const __nv_bfloat16*)ts.ptr, (__nv_bfloat16*)td.ptr, k.stats, k.psum, k.pmax, k.w_dev, k.c,
                                                 ts.c / 8, td.c / 8, ts.h, ts.w, k.ranges);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 17) {
      const VffmOp& k = plan->vffms[o.idx];
      const Tensor& tm = plan->tensors[k.mixed];
      const int B = tm.mult * plan->chunk, hw = tm.h * tm.w;
      const int n_items = B * (k.c / 8) * k.ranges;
      stcd::chan_stats_kernel<<<(n_items + 7) / 8, 256, 0, st>>>((const __nv_bfloat16*)tm.ptr, k.psum, k.pmax, k.c, tm.c / 8, hw, k.ranges,
                                                                 n_items, k.c, 0);
      const int ppb = std::max(32, std::min(1024, 4096 / (k.c / 8)));
      stcd::vffm_apply_kernel<<<dim3((hw + ppb - 1) / ppb, B), 256, 0, st>>>(
          (const __nv_bfloat16*)plan->tensors[k.low].ptr, (const __nv_bfloat16*)plan->tensors[k.high].ptr,
          (const __nv_bfloat16*)plan->tensors[k.local].ptr, (__nv_bfloat16*)plan->tensors[k.dst].ptr, k.psum, k.pmax, k.w_dev, k.c, k.inter,
          hw, k.ranges, ppb);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 15) {
      const SpatialGateOp& k = plan->spatial_gates[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const int B = ts.mult * plan->chunk, hw = ts.h * ts.w;
      stcd::sa_stats_kernel<<<dim3((hw + 255) / 256, B), 256, 0, st>>>((const __nv_bfloat16*)ts.ptr, k.stats, k.c, ts.c / 8, hw);
      stcd::sa_apply_kernel<<<dim3((ts.w + stcd::kSaTW - 1) / stcd::kSaTW, (ts.h + stcd::kSaTH - 1) / stcd::kSaTH, B),
                              dim3(stcd::kSaTW, stcd::kSaTH), 0, st>>>((const __nv_bfloat16*)ts.ptr, (__nv_bfloat16*)td.ptr, k.stats, k.w_dev,
                                                                       k.w_dev + 98, k.w_dev + 98 + k.c, k.c, ts.c / 8, td.c / 8, ts.h, ts.w);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 13) {
      const BitOp& k = plan->bits[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const int imgs = 2 * plan->chunk, hw = ts.h * ts.w;
      const float* conv_a = k.w_dev;
      const float* pos = conv_a + stcd::kBitL * stcd::kBitC;
      const float* enc = pos + 2 * stcd::kBitL * stcd::kBitC;
      const float* dec = enc + (size_t)k.d.n_enc * stcd::bit_enc_size(k.d.inner_enc);
      (plan->split ? stcd::bit_tokenizer_kernel<true> : stcd::bit_tokenizer_kernel<false>)<<<imgs, 256, 0, st>>>(
          (const __nv_bfloat16*)ts.ptr, conv_a, k.tokens, ts.c / 8, hw);
      const float scale = 1.f / sqrtf((float)stcd::kBitC);     // dim ** -0.5 with dim = 32 (help_funcs.py:74,118), not dim_head
      stcd::bit_token_mixer_kernel<<<plan->chunk, 256, k.mixer_smem, st>>>(k.tokens, pos, enc, k.tok_mixed, plan->chunk, k.d.n_enc,
                                                                          k.d.inner_enc, scale);
      stcd::bit_coef_kernel<<<dim3(plan->chunk, k.d.n_dec), 256, k.coef_smem, st>>>(k.tok_mixed, dec, k.coef, plan->chunk, k.d.n_dec,
                                                                                   k.d.inner_dec, scale);
      (plan->split ? stcd::bit_decoder_kernel<true> : stcd::bit_decoder_kernel<false>)<<<
          dim3((hw + 2 * stcd::kBitDecThreads - 1) / (2 * stcd::kBitDecThreads), imgs), stcd::kBitDecThreads, 0, st>>>(
          (const __nv_bfloat16*)ts.ptr, (__nv_bfloat16*)td.ptr, dec, k.coef, ts.c / 8, td.c / 8, hw, k.d.n_dec, k.d.inner_dec, k.d.softmax);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 12) {
      const SumOp& k = plan->sums[o.idx];
      const Tensor& td = plan->tensors[k.dst];
      stcd::AddNParams ap;
      ap.n = k.n;
      for (int i = 0; i < 5; ++i) ap.src[i] = i < k.n ? (const __nv_bfloat16*)plan->tensors[k.src[i]].ptr : nullptr;
      const size_t vecs = td.bytes / 16 / (plan->split ? 2 : 1); // (hi) vectors
      auto kern = plan->split ? stcd::add_n_kernel<true> : stcd::add_n_kernel<false>;
      kern<<<(unsigned)std::max<size_t>(1, std::min<size_t>((vecs + 255) / 256, 148 * 16)), 256, 0, st>>>(ap, (__nv_bfloat16*)td.ptr, vecs,
                                                                                                        (td.c / 16) * td.h * td.w);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 7) {
      const LayerNormOp& k = plan->lns[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const int B = ts.mult * plan->chunk;
      const size_t total = (size_t)B * ts.h * ts.w;
      __nv_bfloat16* d2 = k.dst2 >= 0 ? (__nv_bfloat16*)plan->tensors[k.dst2].ptr : nullptr;
      // 4 threads per pixel (a warp = 8 pixels x 4 channel slices)
      const unsigned blocks = (unsigned)std::max<size_t>(1, std::min<size_t>((total * 4 + 255) / 256, 148 * 16));
      auto kern = plan->split ? stcd::layernorm_kernel<true> : stcd::layernorm_kernel<false>;
      kern<<<blocks, 256, 0, st>>>((const __nv_bfloat16*)ts.ptr, (__nv_bfloat16*)td.ptr, d2, k.gb_dev, k.gb_dev + k.c, B, k.c, ts.c / 8,
                                   td.c / 8, k.dst2 >= 0 ? plan->tensors[k.dst2].c / 8 : 0, ts.h, ts.w, k.eps);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 8) {
      const AttentionOp& k = plan->attns[o.idx];
      const Tensor& tq = plan->tensors[k.q];
      const Tensor& tk = plan->tensors[k.kv];
      const Tensor& td = plan->tensors[k.dst];
      const int B = tq.mult * plan->chunk, N = tq.h * tq.w, NK = tk.h * tk.w, D = k.c / k.heads;
      const dim3 grid((N + 255) / 256, k.heads, B);                       // two queries per thread
      const bool use_mma = NK == 64 && env_int("STCD_ATTN_MMA", 1);        // every stage of the 256 x 256 configurations
      if (plan->split)                                                     // split precision: tensor-core kernel only (NK == 64)
        (D == 64 ? stcd::sr_attention_mma_kernel<64, true> : stcd::sr_attention_mma_kernel<80, true>)<<<dim3((N + 63) / 64, k.heads, B), 128, 0, st>>>(
            (const __nv_bfloat16*)tq.ptr, (const __nv_bfloat16*)tk.ptr, (__nv_bfloat16*)td.ptr, k.c, tq.c / 8, tk.c / 8, td.c / 8, N, k.scale);
      else if (use_mma && D == 64)
        stcd::sr_attention_mma_kernel<64, false><<<dim3((N + 63) / 64, k.heads, B), 128, 0, st>>>(
            (const __nv_bfloat16*)tq.ptr, (const __nv_bfloat16*)tk.ptr, (__nv_bfloat16*)td.ptr, k.c, tq.c / 8, tk.c / 8, td.c / 8, N, k.scale);
      else if (use_mma && D == 80)
        stcd::sr_attention_mma_kernel<80, false><<<dim3((N + 63) / 64, k.heads, B), 128, 0, st>>>(
            (const __nv_bfloat16*)tq.ptr, (const __nv_bfloat16*)tk.ptr, (__nv_bfloat16*)td.ptr, k.c, tq.c / 8, tk.c / 8, td.c / 8, N, k.scale);
      else if (D == 64)
        stcd::sr_attention_kernel<64><<<grid, 128, 0, st>>>((const __nv_bfloat16*)tq.ptr, (const __nv_bfloat16*)tk.ptr, (__nv_bfloat16*)td.ptr,
                                                           k.c, tq.c / 8, tk.c / 8, td.c / 8, N, NK, k.scale);
      else
        stcd::sr_attention_kernel<80><<<grid, 128, 0, st>>>((const __nv_bfloat16*)tq.ptr, (const __nv_bfloat16*)tk.ptr, (__nv_bfloat16*)td.ptr,
                                                           k.c, tq.c / 8, tk.c / 8, td.c / 8, N, NK, k.scale);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 9) {
      const DWConvOp& k = plan->dws[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const int B = ts.mult * plan->chunk;
      const int hwp = ts.h * ts.w;
      const int items = ((ts.w + 3) / 4) * ts.h;                        // one thread per 4 horizontally adjacent pixels
      const dim3 grid((unsigned)std::max(1, (items + 127) / 128), (unsigned)(k.c / 8), (unsigned)B);
      (void)hwp;
      auto kern = plan->split ? stcd::dwconv3x3_kernel<true> : stcd::dwconv3x3_kernel<false>;
      kern<<<grid, 128, 0, st>>>((const __nv_bfloat16*)ts.ptr, (__nv_bfloat16*)td.ptr, k.wb_dev, k.wb_dev + (size_t)k.c * 9, B, k.c / 8,
                                 ts.c / 8, td.c / 8, ts.h, ts.w, k.gelu);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 6) {
      const BilinearOp& k = plan->bilinears[o.idx];
      const Tensor& ts = plan->tensors[k.src];
      const Tensor& td = plan->tensors[k.dst];
      const int B = ts.mult * plan->chunk;
      const size_t total = (size_t)B * (k.c / 8) * td.h * td.w;
      auto kern = plan->split ? stcd::bilinear_up_kernel<true> : stcd::bilinear_up_kernel<false>;
      kern<<<(unsigned)std::max<size_t>(1, std::min<size_t>((total + 255) / 256, 148 * 16)), 256, 0, st>>>(
          (const __nv_bfloat16*)ts.ptr, (__nv_bfloat16*)td.ptr, B, k.c / 8, ts.c / 8, td.c / 8, ts.h, ts.w, k.scale);
      CUDA_TRY(cudaGetLastError());
    } else if (o.kind == 4) {
      const SegHeadOp& k = plan->heads[o.idx];
      const Tensor& t = plan->tensors[k.src];
      float* m1 = outs[k.out_ext];
      float* m2 = outs[k.out_ext + 1];
      float* ch = outs[k.out_ext + 2];
      if (!m1 || !m2 || !ch) return fail(STCD_ERR_INVALID, "external outputs %d..%d must not be NULL", k.out_ext, k.out_ext + 2);
      if (n_valid > 0) {
        const dim3 grid((t.w + stcd::kHeadTW - 1) / stcd::kHeadTW, (t.h + stcd::kHeadTH - 1) / stcd::kHeadTH, n_valid);
        const __nv_bfloat16* dp = (const __nv_bfloat16*)t.ptr;
        const __nv_bfloat16* ddp = k.diff_src >= 0 ? (const __nv_bfloat16*)plan->tensors[k.diff_src].ptr : nullptr;
        const size_t tile = (size_t)(stcd::kHeadTH + 2) * (stcd::kHeadTW + 2) * 16 * (k.c / 8);
        if (k.diff_src < 0) {
          if (k.c == 8)
            stcd::segcd_head_kernel<1, false><<<grid, 256, 2 * tile, st>>>(dp, ddp, k.w_dev, k.bias, plan->chunk, t.h, t.w, m1, m2, ch);
          else if (env_int("STCD_HEAD_MMA", 1))
            stcd::segcd_head_mma_kernel<<<grid, 256, 2 * tile, st>>>(dp, k.w_dev, k.bias, plan->chunk, t.h, t.w, m1, m2, ch);
          else
            stcd::segcd_head_kernel<2, false><<<grid, 256, 2 * tile, st>>>(dp, ddp, k.w_dev, k.bias, plan->chunk, t.h, t.w, m1, m2, ch);
        } else {
          if (k.c == 8)
            stcd::segcd_head_kernel<1, true><<<grid, 256, 3 * tile, st>>>(dp, ddp, k.w_dev, k.bias, plan->chunk, t.h, t.w, m1, m2, ch);
          else
            stcd::segcd_head_kernel<2, true><<<grid, 256, 3 * tile, st>>>(dp, ddp, k.w_dev, k.bias, plan->chunk, t.h, t.w, m1, m2, ch);
        }
        CUDA_TRY(cudaGetLastError());
      }
    } else {
      const PackOp& k = plan->packs[o.idx];
      const Tensor& t = plan->tensors[k.dst];
      const int hw = t.h * t.w;
      const size_t total = (size_t)2 * plan->chunk * hw;
      const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 8);
      if (k.u8) {
        const uint8_t* u1 = static_cast<const uint8_t*>(x1v);
        const uint8_t* u2 = static_cast<const uint8_t*>(x2v);
        __nv_bfloat16* dp = (__nv_bfloat16*)t.ptr;
#define STCD_PACK_U8(CIN)                                                                                                    \
  if (k.s2d)                                                                                                                 \
    stcd::input_pack_s2d_u8_kernel<CIN><<<blocks, 256, 0, st>>>(u1, u2, dp, plan->chunk, n_valid, t.h, t.w, k.norm);         \
  else                                                                                                                       \
    stcd::input_pack_u8_kernel<CIN><<<blocks, 256, 0, st>>>(u1, u2, dp, plan->chunk, n_valid, t.c / 8, hw, k.norm)
        switch (k.cin) {
          case 1: STCD_PACK_U8(1); break;
          case 2: STCD_PACK_U8(2); break;
          case 3: STCD_PACK_U8(3); break;
          default: STCD_PACK_U8(4); break;
        }
#undef STCD_PACK_U8
      } else if (k.s2d) {
        __nv_bfloat16* dp = (__nv_bfloat16*)t.ptr;
#define STCD_PACK_S2D(CIN)                                                                                                   \
  (plan->split ? stcd::input_pack_s2d_kernel<CIN, true> : stcd::input_pack_s2d_kernel<CIN, false>)<<<blocks, 256, 0, st>>>( \
      x1, x2, dp, plan->chunk, n_valid, t.h, t.w)
        switch (k.cin) {
          case 1: STCD_PACK_S2D(1); break;
          case 2: STCD_PACK_S2D(2); break;
          case 3: STCD_PACK_S2D(3); break;
          default: STCD_PACK_S2D(4); break;
        }
#undef STCD_PACK_S2D
      } else if (!plan->split && k.cin <= 4 && hw % 4 == 0 && (reinterpret_cast<uintptr_t>(x1) | reinterpret_cast<uintptr_t>(x2)) % 16 == 0) {
        __nv_bfloat16* dp = (__nv_bfloat16*)t.ptr;
        const int blocks4 = (int)std::min<size_t>((total / 4 + 255) / 256, 148 * 8);
        switch (k.cin) {
          case 1: stcd::input_pack4_kernel<1><<<blocks4, 256, 0, st>>>(x1, x2, dp, plan->chunk, n_valid, t.c / 8, hw); break;
          case 2: stcd::input_pack4_kernel<2><<<blocks4, 256, 0, st>>>(x1, x2, dp, plan->chunk, n_valid, t.c / 8, hw); break;
          case 3: stcd::input_pack4_kernel<3><<<blocks4, 256, 0, st>>>(x1, x2, dp, plan->chunk, n_valid, t.c / 8, hw); break;
          default: stcd::input_pack4_kernel<4><<<blocks4, 256, 0, st>>>(x1, x2, dp, plan->chunk, n_valid, t.c / 8, hw); break;
        }
      } else
        stcd::input_pack_kernel<<<blocks, 256, 0, st>>>(x1, x2, (__nv_bfloat16*)t.ptr, plan->chunk, n_valid, k.cin, t.c / 8, hw, plan->split);
      CUDA_TRY(cudaGetLastError());
    }
    ++op_i;
    if (ev) CUDA_TRY(cudaEventRecord(ev[op_i], st));
  }
  return STCD_OK;
}

}  // namespace

// ================================================================================ C-ABI
// Entry points run on the plan's (or the buffers') device and leave the caller's current device as they found it:
// a model on cuda:1 must not flip PyTorch's current device for the calling thread.
struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int dev) {
    if (dev >= 0 && cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};
// device that owns a device pointer (-1: not a device pointer / unknown, stay on the current device)
static int device_of(const void* ptr) {
  cudaPointerAttributes a;
  if (ptr && cudaPointerGetAttributes(&a, ptr) == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged))
    return a.device;
  cudaGetLastError();
  return -1;
}

extern "C" {

const char* stcd_last_error(void) { return g_err.c_str(); }
int stcd_abi_version(void) { return STCD_ABI_VERSION; }

int stcd_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, i) == cudaSuccess && prop.major == 10) ++ok;
  }
  return ok;
}

int stcd_plan_create(int device, int chunk_pairs, int precision, stcd_plan** out) {
  if (!out) return fail(STCD_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (chunk_pairs < 1 || chunk_pairs > 4096) return fail(STCD_ERR_INVALID, "chunk_pairs %d out of range", chunk_pairs);
  if (precision != STCD_PRECISION_BF16 && precision != STCD_PRECISION_SPLIT)
    return fail(STCD_ERR_INVALID, "precision %d is neither STCD_PRECISION_BF16 (0) nor STCD_PRECISION_SPLIT (1)", precision);
  if (device != -1) {          // device -1: a validation plan (descriptors are checked and recorded, finalize refuses)
    int r = check_sm100(device);
    if (r) return r;
  }
  stcd_plan* p = new stcd_plan();
  p->device = device;
  p->chunk = chunk_pairs;
  p->split = precision == STCD_PRECISION_SPLIT;
  *out = p;
  return STCD_OK;
}

void stcd_plan_destroy(stcd_plan* plan) {
  if (!plan) return;
  DeviceGuard dev_guard(plan->device);
  for (auto& g : plan->graph_cache)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  if (plan->s_capture) cudaStreamDestroy(plan->s_capture);
  for (ConvOp& op : plan->convs)
    if (op.trace) cudaFree(op.trace);
  for (EcamOp& e : plan->ecams) {
    if (e.w_dev) cudaFree(e.w_dev);
    if (e.partial) cudaFree(e.partial);
  }
  for (SegHeadOp& e : plan->heads)
    if (e.w_dev) cudaFree(e.w_dev);
  for (LayerNormOp& k : plan->lns)
    if (k.gb_dev) cudaFree(k.gb_dev);
  for (ChanAttnOp& k : plan->chan_attns) {
    if (k.w_dev) cudaFree(k.w_dev);
    if (k.psum) cudaFree(k.psum);
    if (k.pmax) cudaFree(k.pmax);
    if (k.gate) cudaFree(k.gate);
  }
  for (SpatialGateOp& k : plan->spatial_gates) {
    if (k.w_dev) cudaFree(k.w_dev);
    if (k.stats) cudaFree(k.stats);
  }
  for (GlGateOp& k : plan->gl_gates) {
    if (k.w_dev) cudaFree(k.w_dev);
    if (k.psum) cudaFree(k.psum);
    if (k.pmax) cudaFree(k.pmax);
    if (k.stats) cudaFree(k.stats);
  }
  for (VffmOp& k : plan->vffms) {
    if (k.w_dev) cudaFree(k.w_dev);
    if (k.psum) cudaFree(k.psum);
    if (k.pmax) cudaFree(k.pmax);
  }
  for (BitOp& k : plan->bits) {
    if (k.w_dev) cudaFree(k.w_dev);
    if (k.tokens) cudaFree(k.tokens);
    if (k.tok_mixed) cudaFree(k.tok_mixed);
    if (k.coef) cudaFree(k.coef);
  }
  for (GateOp& k : plan->gates) {
    if (k.w_dev) cudaFree(k.w_dev);
    if (k.partial) cudaFree(k.partial);
  }
  for (DWConvOp& k : plan->dws)
    if (k.wb_dev) cudaFree(k.wb_dev);
  for (GraphOp& g : plan->graphs) {
    if (g.relpos_dev) cudaFree(g.relpos_dev);
    if (g.xf) cudaFree(g.xf);
    if (g.yf) cudaFree(g.yf);
    if (g.xn) cudaFree(g.xn);
    if (g.yn) cudaFree(g.yn);
    if (g.xp) cudaFree(g.xp);
    if (g.yp) cudaFree(g.yp);
    if (g.xsq) cudaFree(g.xsq);
    if (g.ysq) cudaFree(g.ysq);
    if (g.idx) cudaFree(g.idx);
  }
  if (plan->workspace) cudaFree(plan->workspace);
  if (plan->arena) cudaFree(plan->arena);
  for (int b = 0; b < 2; ++b) {
    for (int s = 0; s < 2; ++s)
      if (plan->stage_in[b][s]) cudaFree(plan->stage_in[b][s]);
    for (float* q : plan->stage_out[b])
      if (q) cudaFree(q);
    if (plan->ev_h2d[b]) cudaEventDestroy(plan->ev_h2d[b]);
    if (plan->ev_comp[b]) cudaEventDestroy(plan->ev_comp[b]);
    if (plan->ev_d2h[b]) cudaEventDestroy(plan->ev_d2h[b]);
  }
  if (plan->s_copy) cudaStreamDestroy(plan->s_copy);
  if (plan->s_comp) cudaStreamDestroy(plan->s_comp);
  if (plan->s_d2h) cudaStreamDestroy(plan->s_d2h);
  delete plan;
}

int stcd_plan_add_tensor(stcd_plan* plan, int img_mult, int h, int w, int c, int dtype) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (img_mult < 1 || img_mult > 2 || h < 1 || w < 1 || c < 8 || (c % 8) != 0 || dtype != STCD_BF16)
    return -fail(STCD_ERR_INVALID, "bad tensor decl mult=%d h=%d w=%d c=%d dtype=%d (c must be a multiple of 8, bf16)",
                 img_mult, h, w, c, dtype);
  if (plan->split && (c % 16))
    return -fail(STCD_ERR_INVALID, "split plan: tensor channels %d not a multiple of 16 (a hi and a lo plane of 8-channel groups)", c);
  Tensor t;
  t.mult = img_mult;
  t.h = h;
  t.w = w;
  t.c = c;
  t.dtype = dtype;
  t.bytes = (size_t)img_mult * plan->chunk * h * w * c * 2;
  plan->tensors.push_back(t);
  return (int)plan->tensors.size() - 1;
}

int stcd_plan_add_input_pack(stcd_plan* plan, int dst_tensor, int cin) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "bad dst tensor %d", dst_tensor);
  const Tensor& t = plan->tensors[dst_tensor];
  if (plan->split && (t.mult != 2 || t.c != 16 || cin < 1 || cin > 8))
    return -fail(STCD_ERR_INVALID, "split input pack needs a [2*chunk][2][h][w][8] tensor (hi plane, lo plane) and cin <= 8 (got mult=%d c=%d cin=%d)",
                 t.mult, t.c, cin);
  if (t.mult != 2 || (t.c != 8 && t.c != 16) || cin < 1 || cin > t.c)
    return -fail(STCD_ERR_INVALID, "input pack needs a [2*chunk][1 or 2][h][w][8] tensor and cin <= its channels (got mult=%d c=%d cin=%d)",
                 t.mult, t.c, cin);
  plan->packs.push_back({dst_tensor, cin});
  plan->ops.push_back({1, (int)plan->packs.size() - 1});
  plan->in_c = cin;
  plan->in_h = t.h;
  plan->in_w = t.w;
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_input_pack_s2d(stcd_plan* plan, int dst_tensor, int cin) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "bad dst tensor %d", dst_tensor);
  const Tensor& t = plan->tensors[dst_tensor];
  if (t.mult != 2 || t.c != (plan->split ? 32 : 16) || cin < 1 || cin > 4)
    return -fail(STCD_ERR_INVALID, "space-to-depth input pack needs a [2*chunk][%d][h][w][8] tensor and cin <= 4 (got mult=%d c=%d cin=%d)",
                 plan->split ? 4 : 2, t.mult, t.c, cin);
  PackOp k;
  k.dst = dst_tensor;
  k.cin = cin;
  k.s2d = 1;
  plan->packs.push_back(k);
  plan->ops.push_back({1, (int)plan->packs.size() - 1});
  plan->in_c = cin;
  plan->in_h = 2 * t.h;
  plan->in_w = 2 * t.w;
  return (int)plan->ops.size() - 1;
}

// entry points of ops that have no split form start with this: a split plan refuses them
static int refuse_split(const stcd_plan* plan, const char* op) {
  return plan && plan->split ? -fail(STCD_ERR_INVALID, "%s has no split form (split plan)", op) : 0;
}

int stcd_plan_add_input_pack_u8(stcd_plan* plan, int dst_tensor, int cin, int s2d, const float* mean, const float* std_) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (int r = refuse_split(plan, "uint8 input pack")) return r;
  if (!mean || !std_) return -fail(STCD_ERR_INVALID, "mean/std are NULL");
  if (cin < 1 || cin > 4) return -fail(STCD_ERR_INVALID, "uint8 input pack: cin %d not in [1, 4]", cin);
  for (int c = 0; c < cin; ++c)
    if (!(std_[c] > 0.f)) return -fail(STCD_ERR_INVALID, "std[%d] must be positive", c);
  const int r = s2d ? stcd_plan_add_input_pack_s2d(plan, dst_tensor, cin) : stcd_plan_add_input_pack(plan, dst_tensor, cin);
  if (r < 0) return r;
  PackOp& k = plan->packs.back();
  k.u8 = 1;
  for (int c = 0; c < 4; ++c) {
    k.norm.mean[c] = c < cin ? mean[c] : 0.f;
    k.norm.stdv[c] = c < cin ? std_[c] : 1.f;
  }
  plan->in_u8 = 1;
  return r;
}

// split plan: each tensor (ids >= 0, already validated) stores an op's c logical channels twice over, the hi plane first and the
// lo plane at half its stored channels
static int check_split_planes(const stcd_plan* plan, const char* op, std::initializer_list<int> tensor_ids, int c) {
  if (!plan->split) return 0;
  for (int id : tensor_ids)
    if (id >= 0 && plan->tensors[id].c < 2 * c)
      return -fail(STCD_ERR_INVALID, "split %s: tensor %d stores %d channels, not the 2 x %d of a hi and a lo plane", op, id,
                   plan->tensors[id].c, c);
  return 0;
}

int stcd_plan_add_maxpool_s2d(stcd_plan* plan, int src_tensor, int dst_tensor, int c) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "bad tensor id");
  if (int r = check_split_planes(plan, "max-pool", {dst_tensor}, c)) return r;
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  // split plan: src stores 8c (4 parity classes x 2 planes)
  if (c < 8 || (c % 8) || ts.c != (plan->split ? 8 : 4) * c || td.c < c || ts.h != td.h || ts.w != td.w || ts.mult != td.mult)
    return -fail(STCD_ERR_INVALID, "max-pool: src [%d*chunk,%d,%d,%d] must be the space-to-depth form of dst [%d*chunk,%d,%d,%d] (c=%d)",
                 ts.mult, ts.h, ts.w, ts.c, td.mult, td.h, td.w, td.c, c);
  plan->pools.push_back({src_tensor, dst_tensor, c});
  plan->ops.push_back({3, (int)plan->pools.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_graph_conv(stcd_plan* plan, int src_tensor, int dst_tensor, int c, int k, int dilation, int r, const float* relpos) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (int e = refuse_split(plan, "graph conv")) return e;
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "bad tensor id");
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (c < 8 || (c % 8) || ts.c < c || td.c < c || ts.h != td.h || ts.w != td.w || ts.mult != td.mult)
    return -fail(STCD_ERR_INVALID, "graph conv: src [%d*chunk,%d,%d,%d] / dst [%d*chunk,%d,%d,%d] must match and hold c=%d channels", ts.mult,
                 ts.h, ts.w, ts.c, td.mult, td.h, td.w, td.c, c);
  if (k < 1 || dilation < 1 || r < 1 || (ts.h % r) || (ts.w % r)) return -fail(STCD_ERR_INVALID, "graph conv: bad k/dilation/r");
  const int N = ts.h * ts.w, M = N / (r * r);
  if (M > stcd::kKnnM || k * dilation > M) return -fail(STCD_ERR_INVALID, "graph conv: M=%d keys (max %d), k*dilation=%d", M, stcd::kKnnM, k * dilation);
  GraphOp g;
  g.src = src_tensor;
  g.dst = dst_tensor;
  g.c = c;
  g.k = k;
  g.dilation = dilation;
  g.r = r;
  if (relpos) g.relpos.assign(relpos, relpos + (size_t)N * M);
  plan->graphs.push_back(std::move(g));
  plan->ops.push_back({5, (int)plan->graphs.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_layernorm(stcd_plan* plan, int src_tensor, int dst_tensor, int dst_s2d, int c, const float* gamma, const float* beta,
                            float eps) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor) || (dst_s2d >= 0 && !valid_tensor(plan, dst_s2d)) || !gamma || !beta)
    return -fail(STCD_ERR_INVALID, "layer norm: bad tensor id / NULL gamma, beta");
  if (int r = check_split_planes(plan, "layer norm", {src_tensor, dst_tensor}, c)) return r;
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (c < 8 || (c % 8) || ts.c < c || td.c < c || ts.h != td.h || ts.w != td.w || ts.mult != td.mult || !(eps > 0.f))
    return -fail(STCD_ERR_INVALID, "layer norm: src [%d*chunk,%d,%d,%d] / dst [%d*chunk,%d,%d,%d] must match and hold c=%d channels", ts.mult,
                 ts.h, ts.w, ts.c, td.mult, td.h, td.w, td.c, c);
  if (dst_s2d >= 0) {      // split plan: 8c (4 parity classes x 2 planes)
    const Tensor& t2 = plan->tensors[dst_s2d];
    if ((ts.h % 2) || (ts.w % 2) || t2.h != ts.h / 2 || t2.w != ts.w / 2 || t2.c != (plan->split ? 8 : 4) * c || t2.mult != ts.mult)
      return -fail(STCD_ERR_INVALID, "layer norm: space-to-depth copy must be [%d*chunk,%d,%d,%d]", ts.mult, ts.h / 2, ts.w / 2,
                   (plan->split ? 8 : 4) * c);
  }
  LayerNormOp k;
  k.src = src_tensor;
  k.dst = dst_tensor;
  k.dst2 = dst_s2d;
  k.c = c;
  k.eps = eps;
  k.gb.assign(gamma, gamma + c);
  k.gb.insert(k.gb.end(), beta, beta + c);
  plan->lns.push_back(std::move(k));
  plan->ops.push_back({7, (int)plan->lns.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_sr_attention(stcd_plan* plan, int q_tensor, int kv_tensor, int dst_tensor, int c, int heads, float scale) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, q_tensor) || !valid_tensor(plan, kv_tensor) || !valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "bad tensor id");
  const Tensor& tq = plan->tensors[q_tensor];
  const Tensor& tk = plan->tensors[kv_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (heads < 1 || c < 8 || (c % heads) || ((c / heads) != 64 && (c / heads) != 80))
    return -fail(STCD_ERR_INVALID, "attention: c=%d heads=%d: head dim must be 64 or 80", c, heads);
  const int cs = plan->split ? 2 * c : c;        // stored channels of q and dst (split plan: hi and lo planes)
  if (tq.c != cs || td.c != cs || tk.c != 2 * cs || tq.h != td.h || tq.w != td.w || tq.mult != td.mult || tq.mult != tk.mult)
    return -fail(STCD_ERR_INVALID, "attention: q/dst must be [m*chunk,h,w,%d] and kv [m*chunk,hk,wk,%d]%s", cs, 2 * cs,
                 plan->split ? " (hi and lo planes)" : "");
  if (plan->split && tk.h * tk.w != 64)
    return -fail(STCD_ERR_INVALID, "split attention: %d keys (the tensor-core kernel takes exactly 64)", tk.h * tk.w);
  if (tk.h * tk.w > stcd::kAttnMaxKeys) return -fail(STCD_ERR_INVALID, "attention: %d keys (max %d)", tk.h * tk.w, stcd::kAttnMaxKeys);
  plan->attns.push_back({q_tensor, kv_tensor, dst_tensor, c, heads, scale});
  plan->ops.push_back({8, (int)plan->attns.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_dwconv3x3(stcd_plan* plan, int src_tensor, int dst_tensor, int c, const float* weight, const float* bias, int gelu) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor) || !weight || !bias) return -fail(STCD_ERR_INVALID, "dw conv: bad tensor id / NULL weights");
  if (int r = check_split_planes(plan, "dw conv", {src_tensor, dst_tensor}, c)) return r;
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (c < 8 || (c % 8) || ts.c < c || td.c < c || ts.h != td.h || ts.w != td.w || ts.mult != td.mult)
    return -fail(STCD_ERR_INVALID, "dw conv: src [%d*chunk,%d,%d,%d] / dst [%d*chunk,%d,%d,%d] must match and hold c=%d channels", ts.mult, ts.h,
                 ts.w, ts.c, td.mult, td.h, td.w, td.c, c);
  DWConvOp k;
  k.src = src_tensor;
  k.dst = dst_tensor;
  k.c = c;
  k.gelu = gelu ? 1 : 0;
  k.wb.assign(weight, weight + (size_t)c * 9);
  k.wb.insert(k.wb.end(), bias, bias + c);
  plan->dws.push_back(std::move(k));
  plan->ops.push_back({9, (int)plan->dws.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_bilinear_up(stcd_plan* plan, int src_tensor, int dst_tensor, int c, int scale) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "bad tensor id");
  if (int r = check_split_planes(plan, "bilinear up", {src_tensor, dst_tensor}, c)) return r;
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (c < 8 || (c % 8) || ts.c < c || td.c < c || scale < 1 || scale > 32 || td.h != ts.h * scale || td.w != ts.w * scale || ts.mult != td.mult)
    return -fail(STCD_ERR_INVALID, "bilinear up: src [%d*chunk,%d,%d,%d] x%d does not give dst [%d*chunk,%d,%d,%d] (c=%d)", ts.mult, ts.h, ts.w,
                 ts.c, scale, td.mult, td.h, td.w, td.c, c);
  plan->bilinears.push_back({src_tensor, dst_tensor, c, scale});
  plan->ops.push_back({6, (int)plan->bilinears.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_absdiff(stcd_plan* plan, int src_tensor, int dst_tensor) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "bad tensor id");
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (ts.mult != 2 || td.mult != 1 || ts.h != td.h || ts.w != td.w || ts.c != td.c)
    return -fail(STCD_ERR_INVALID, "abs-diff: src must be [2*chunk,%d,%d,%d] (both streams) and dst the same with one stream", td.h, td.w, td.c);
  plan->absdiffs.push_back({src_tensor, dst_tensor, td.c});
  plan->ops.push_back({10, (int)plan->absdiffs.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_subdiff(stcd_plan* plan, int src_tensor, int add, int dst_tensor) {
  if (plan && add >= 0) {
    if (!valid_tensor(plan, add) || !valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "bad tensor id");
    const Tensor& ta = plan->tensors[add];
    const Tensor& td = plan->tensors[dst_tensor];
    if (ta.mult != 1 || ta.h != td.h || ta.w != td.w || ta.c != td.c) return -fail(STCD_ERR_INVALID, "signed diff: addend shape");
  }
  const int r = stcd_plan_add_absdiff(plan, src_tensor, dst_tensor);
  if (r >= 0) {
    plan->absdiffs.back().signed_diff = 1;
    plan->absdiffs.back().add = add;
  }
  return r;
}

int stcd_plan_add_channel_gate(stcd_plan* plan, int src_tensor, int res, int dst_tensor, int dst_s2d, int c, int hid, const float* w1,
                               const float* w2, const float* ws, int mode) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor) || (res >= 0 && !valid_tensor(plan, res)) ||
      (dst_s2d >= 0 && !valid_tensor(plan, dst_s2d)) || !w1 || !w2 || (mode == 1 && !ws) || mode < 0 || mode > 1)
    return -fail(STCD_ERR_INVALID, "channel gate: bad tensor id / NULL weights / mode");
  if (int r = check_split_planes(plan, "channel gate", {src_tensor, res, dst_tensor}, c)) return r;
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (c < 8 || (c % 8) || c > stcd::kGateMaxC || hid < 1 || hid > stcd::kGateMaxH || ts.c < c || td.c < c || ts.h != td.h || ts.w != td.w ||
      ts.mult != td.mult)
    return -fail(STCD_ERR_INVALID, "channel gate: c=%d (<= %d) hid=%d (<= %d); src/dst must match", c, stcd::kGateMaxC, hid, stcd::kGateMaxH);
  if (res >= 0) {
    const Tensor& tr = plan->tensors[res];
    if (tr.h != ts.h || tr.w != ts.w || tr.c < c || tr.mult != ts.mult) return -fail(STCD_ERR_INVALID, "channel gate: residual shape");
  }
  if (dst_s2d >= 0) {      // split plan: 8c (4 parity classes x 2 planes)
    const Tensor& t2 = plan->tensors[dst_s2d];
    if ((ts.h % 2) || (ts.w % 2) || t2.h != ts.h / 2 || t2.w != ts.w / 2 || t2.c != (plan->split ? 8 : 4) * c || t2.mult != ts.mult)
      return -fail(STCD_ERR_INVALID, "channel gate: space-to-depth copy must be [%d*chunk,%d,%d,%d]", ts.mult, ts.h / 2, ts.w / 2,
                   (plan->split ? 8 : 4) * c);
  }
  GateOp k;
  k.src = src_tensor;
  k.res = res;
  k.dst = dst_tensor;
  k.dst2 = dst_s2d;
  k.c = c;
  k.hid = hid;
  k.mode = mode;
  k.ranges = std::max(1, std::min(16, ts.h * ts.w / stcd::kGateRangePix));
  k.w.assign(w1, w1 + (size_t)hid * c);
  k.w.insert(k.w.end(), w2, w2 + (size_t)c * hid);
  if (mode == 1) k.w.insert(k.w.end(), ws, ws + c);
  plan->gates.push_back(std::move(k));
  plan->ops.push_back({11, (int)plan->gates.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_bit_transformer(stcd_plan* plan, int src_tensor, int dst_tensor, const stcd_bit_desc* d) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!d || !valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor) || !d->conv_a || !d->pos || !d->enc || !d->dec)
    return -fail(STCD_ERR_INVALID, "BIT transformer: bad tensor id / NULL descriptor or weights");
  if (d->c != stcd::kBitC || d->token_len != stcd::kBitL || d->heads != stcd::kBitHeads || d->mlp != stcd::kBitMlp)
    return -fail(STCD_ERR_INVALID, "BIT transformer: c=%d token_len=%d heads=%d mlp=%d; the kernels serve 32 / 4 / 8 / 64", d->c, d->token_len,
                 d->heads, d->mlp);
  if (d->n_enc < 0 || d->n_enc > 16 || d->n_dec < 1 || d->n_dec > 32 || d->inner_enc < 8 || d->inner_enc > 1024 || (d->inner_enc % 8) ||
      d->inner_dec < 8 || d->inner_dec > 1024 || (d->inner_dec % 8))
    return -fail(STCD_ERR_INVALID, "BIT transformer: depths %d/%d, inner dims %d/%d out of range", d->n_enc, d->n_dec, d->inner_enc, d->inner_dec);
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  const int cs = (plan->split ? 2 : 1) * stcd::kBitC;      // stored channels (split plan: hi and lo planes)
  if (ts.mult != 2 || td.mult != 2 || ts.c != cs || td.c != cs || ts.h != td.h || ts.w != td.w)
    return -fail(STCD_ERR_INVALID, "BIT transformer: src and dst must be [2*chunk,h,w,%d] (both streams)", cs);
  BitOp k;
  k.src = src_tensor;
  k.dst = dst_tensor;
  k.d = *d;
  k.w.assign(d->conv_a, d->conv_a + stcd::kBitL * stcd::kBitC);
  k.w.insert(k.w.end(), d->pos, d->pos + 2 * stcd::kBitL * stcd::kBitC);
  k.w.insert(k.w.end(), d->enc, d->enc + (size_t)d->n_enc * stcd::bit_enc_size(d->inner_enc));
  k.w.insert(k.w.end(), d->dec, d->dec + (size_t)d->n_dec * stcd::bit_dec_size(d->inner_dec));
  k.d.conv_a = k.d.pos = k.d.enc = k.d.dec = nullptr;
  k.mixer_smem = sizeof(float) * (size_t)(8 * 3 * d->inner_enc);
  k.coef_smem = sizeof(float) * (size_t)(2 * 8 * d->inner_dec);
  plan->bits.push_back(std::move(k));
  plan->ops.push_back({13, (int)plan->bits.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_channel_attention(stcd_plan* plan, const int* src_tensors, const int* src_streams, const int* src_c, int n_src,
                                    int dst_tensor, int hid, const float* fc1, const float* fc2) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (int r = refuse_split(plan, "channel attention")) return r;
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!src_tensors || !src_streams || !src_c || n_src < 1 || n_src > 4 || !valid_tensor(plan, dst_tensor) || !fc1 || !fc2 || hid < 1 ||
      hid > stcd::kCaMaxH)
    return -fail(STCD_ERR_INVALID, "channel attention: 1..4 sources, hid <= %d, non-NULL weights", stcd::kCaMaxH);
  const Tensor& td = plan->tensors[dst_tensor];
  ChanAttnOp k;
  k.n_src = n_src;
  k.dst = dst_tensor;
  k.hid = hid;
  k.c_tot = 0;
  for (int i = 0; i < n_src; ++i) {
    if (!valid_tensor(plan, src_tensors[i])) return -fail(STCD_ERR_INVALID, "channel attention: bad tensor id");
    const Tensor& ts = plan->tensors[src_tensors[i]];
    if (src_streams[i] < 0 || src_streams[i] >= ts.mult || src_c[i] < 8 || (src_c[i] % 8) || src_c[i] > ts.c || ts.h != td.h || ts.w != td.w)
      return -fail(STCD_ERR_INVALID, "channel attention: source %d (stream %d, %d channels) does not fit its tensor / the destination", i,
                   src_streams[i], src_c[i]);
    k.src[i] = src_tensors[i];
    k.stream[i] = src_streams[i];
    k.c[i] = src_c[i];
    k.c_tot += src_c[i];
  }
  if (td.mult != 1 || td.c != k.c_tot || k.c_tot > stcd::kCaMaxC)
    return -fail(STCD_ERR_INVALID, "channel attention: dst must be [chunk,h,w,%d] (<= %d channels)", k.c_tot, stcd::kCaMaxC);
  k.ranges = std::max(1, std::min(16, td.h * td.w / stcd::kGateRangePix));
  k.w.assign(fc1, fc1 + (size_t)hid * k.c_tot);
  k.w.resize((size_t)2 * hid * k.c_tot);                       // fc2 [C][hid] stored transposed: [hid][C]
  for (int c = 0; c < k.c_tot; ++c)
    for (int u = 0; u < hid; ++u) k.w[(size_t)hid * k.c_tot + (size_t)u * k.c_tot + c] = fc2[(size_t)c * hid + u];
  plan->chan_attns.push_back(std::move(k));
  plan->ops.push_back({14, (int)plan->chan_attns.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_spatial_gate(stcd_plan* plan, int src_tensor, int dst_tensor, int c, const float* w, const float* scale, const float* shift) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (int r = refuse_split(plan, "spatial gate")) return r;
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor) || !w || !scale || !shift)
    return -fail(STCD_ERR_INVALID, "spatial gate: bad tensor id / NULL weights");
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (c < 8 || (c % 8) || ts.c < c || td.c < c || ts.h != td.h || ts.w != td.w || ts.mult != td.mult)
    return -fail(STCD_ERR_INVALID, "spatial gate: c=%d; src and dst must have the same shape", c);
  SpatialGateOp k;
  k.src = src_tensor;
  k.dst = dst_tensor;
  k.c = c;
  k.w.assign(w, w + 98);
  k.w.insert(k.w.end(), scale, scale + c);
  k.w.insert(k.w.end(), shift, shift + c);
  plan->spatial_gates.push_back(std::move(k));
  plan->ops.push_back({15, (int)plan->spatial_gates.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_global_local_gate(stcd_plan* plan, int src_tensor, int dst_tensor, int c, const float* prm) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (int r = refuse_split(plan, "global-local gate")) return r;
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, src_tensor) || !valid_tensor(plan, dst_tensor) || !prm) return -fail(STCD_ERR_INVALID, "global-local gate: bad tensor id / NULL weights");
  const Tensor& ts = plan->tensors[src_tensor];
  const Tensor& td = plan->tensors[dst_tensor];
  if (c < 8 || (c % 8) || c > stcd::kGlMaxC || ts.c < c || td.c < c || ts.h != td.h || ts.w != td.w || ts.mult != td.mult)
    return -fail(STCD_ERR_INVALID, "global-local gate: c=%d (<= %d); src and dst must have the same shape", c, stcd::kGlMaxC);
  GlGateOp k;
  k.src = src_tensor;
  k.dst = dst_tensor;
  k.c = c;
  k.ranges = std::max(1, std::min(16, ts.h * ts.w / stcd::kGateRangePix));
  k.w.assign(prm, prm + 4 * (size_t)c + 51);
  plan->gl_gates.push_back(std::move(k));
  plan->ops.push_back({16, (int)plan->gl_gates.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_csam_gate(stcd_plan* plan, int src_tensor, int dst_tensor, int c, int hid, const float* prm) {
  if (int r = refuse_split(plan, "csam gate")) return r;
  if (hid < 1 || hid > stcd::kGlMaxC / 4) return -fail(STCD_ERR_INVALID, "csam gate: hid=%d (1..%d)", hid, stcd::kGlMaxC / 4);
  const int r = stcd_plan_add_global_local_gate(plan, src_tensor, dst_tensor, c, prm);   // same tensors and checks; weights replaced below
  if (r < 0) return r;
  GlGateOp& k = plan->gl_gates.back();
  k.hid = hid;
  k.w.assign(prm, prm + 7 * (size_t)c + 2 * (size_t)hid * c + 27);
  return r;
}

int stcd_plan_add_vffm(stcd_plan* plan, int low, int high, int mixed, int local, int dst, int c, int inter, const float* prm) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (int r = refuse_split(plan, "VFFM")) return r;
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  const int ids[5] = {low, high, mixed, local, dst};
  for (int id : ids)
    if (!valid_tensor(plan, id)) return -fail(STCD_ERR_INVALID, "VFFM: bad tensor id");
  if (!prm || c < 8 || (c % 8) || c > stcd::kGlMaxC || inter < 1 || inter > stcd::kGlMaxC / 4)
    return -fail(STCD_ERR_INVALID, "VFFM: c=%d (<= %d), inter=%d (<= %d)", c, stcd::kGlMaxC, inter, stcd::kGlMaxC / 4);
  const Tensor& t0 = plan->tensors[low];
  for (int id : ids) {
    const Tensor& t = plan->tensors[id];
    if (t.c != c || t.h != t0.h || t.w != t0.w || t.mult != t0.mult) return -fail(STCD_ERR_INVALID, "VFFM: all five tensors must be [m*chunk,h,w,%d]", c);
  }
  VffmOp k;
  k.low = low, k.high = high, k.mixed = mixed, k.local = local, k.dst = dst, k.c = c, k.inter = inter;
  k.ranges = std::max(1, std::min(16, t0.h * t0.w / stcd::kGateRangePix));
  k.w.assign(prm, prm + 2 * ((size_t)2 * inter * c + 2 * inter + 2 * c));
  plan->vffms.push_back(std::move(k));
  plan->ops.push_back({17, (int)plan->vffms.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_sum(stcd_plan* plan, const int* src_tensors, int n, int dst_tensor) {
  if (!plan) return -fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!src_tensors || n < 1 || n > 5 || !valid_tensor(plan, dst_tensor)) return -fail(STCD_ERR_INVALID, "sum: 1..5 sources");
  const Tensor& td = plan->tensors[dst_tensor];
  SumOp k;
  k.n = n;
  k.dst = dst_tensor;
  for (int i = 0; i < 5; ++i) k.src[i] = -1;
  for (int i = 0; i < n; ++i) {
    if (!valid_tensor(plan, src_tensors[i])) return -fail(STCD_ERR_INVALID, "sum: bad tensor id");
    const Tensor& t = plan->tensors[src_tensors[i]];
    if (t.h != td.h || t.w != td.w || t.c != td.c || t.mult != td.mult) return -fail(STCD_ERR_INVALID, "sum: shapes differ");
    k.src[i] = src_tensors[i];
  }
  plan->sums.push_back(k);
  plan->ops.push_back({12, (int)plan->sums.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_seg_head(stcd_plan* plan, const stcd_seghead_desc* d) {
  if (!plan || !d) return -fail(STCD_ERR_STATE, "plan/desc is NULL");
  if (int r = refuse_split(plan, "seg head")) return r;
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (!valid_tensor(plan, d->src) || !d->weight || d->out_ext < 0) return -fail(STCD_ERR_INVALID, "seg head: bad src / NULL weight / out_ext");
  const Tensor& t = plan->tensors[d->src];
  if ((d->c != 8 && d->c != 16) || t.c != d->c || t.mult != 2)
    return -fail(STCD_ERR_INVALID, "seg head: src is [%d*chunk,%d,%d,%d]; need both streams (mult 2) and c = %d in {8, 16}", t.mult, t.h,
                 t.w, t.c, d->c);
  SegHeadOp k;
  k.src = d->src;
  k.c = d->c;
  k.out_ext = d->out_ext;
  k.bias = d->bias;
  k.diff_src = d->diff_src;
  if (d->diff_src >= 0) {
    if (!valid_tensor(plan, d->diff_src)) return -fail(STCD_ERR_INVALID, "seg head: bad diff_src tensor %d", d->diff_src);
    const Tensor& tdiff = plan->tensors[d->diff_src];
    if (tdiff.mult != 1 || tdiff.c != d->c || tdiff.h != t.h || tdiff.w != t.w)
      return -fail(STCD_ERR_INVALID, "seg head: diff_src must be [chunk,%d,%d,%d]", t.h, t.w, d->c);
  }
  k.w.assign(d->weight, d->weight + 9 * d->c);
  plan->n_ext = std::max(plan->n_ext, d->out_ext + 3);
  if ((int)plan->ext_elems.size() < plan->n_ext) plan->ext_elems.resize(plan->n_ext, 0);
  for (int i = 0; i < 3; ++i) plan->ext_elems[d->out_ext + i] = (size_t)t.h * t.w;
  plan->heads.push_back(std::move(k));
  plan->ops.push_back({4, (int)plan->heads.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_conv(stcd_plan* plan, const stcd_conv_desc* d) {
  if (!plan || !d) return -fail(STCD_ERR_STATE, "plan/desc is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (d->n_src < 1 || d->n_src > STCD_MAX_SRC) return -fail(STCD_ERR_INVALID, "n_src %d", d->n_src);
  if (d->kc < 16 || d->kc > 128 || (d->kc % 16)) return -fail(STCD_ERR_INVALID, "kc %d must be a multiple of 16 in [16, 128]", d->kc);
  if (d->n_tile < 16 || d->n_tile > 256 || d->n_tile % 16) return -fail(STCD_ERR_INVALID, "n_tile %d", d->n_tile);
  if (d->cout < 1 || d->cout_pad < d->cout || d->cout_pad % d->n_tile)
    return -fail(STCD_ERR_INVALID, "cout %d / cout_pad %d / n_tile %d", d->cout, d->cout_pad, d->n_tile);
  if (d->n_phase < 1 || d->n_phase > STCD_MAX_PHASE) return -fail(STCD_ERR_INVALID, "n_phase %d", d->n_phase);
  if (!d->weights || !d->chunks || !d->taps || !d->scale || !d->shift)
    return -fail(STCD_ERR_INVALID, "NULL weights/chunks/taps/scale/shift");
  if ((d->scale2 == nullptr) != (d->shift2 == nullptr)) return -fail(STCD_ERR_INVALID, "scale2/shift2 must come together");
  if (d->relu < 0 || d->relu > 3) return -fail(STCD_ERR_INVALID, "activation kind %d not in [0, 3]", d->relu);
  if (d->act_pre && (!d->scale2 || !d->relu)) return -fail(STCD_ERR_INVALID, "act_pre needs an activation and the second affine");
  if (d->img_mult < 1 || d->img_mult > 2) return -fail(STCD_ERR_INVALID, "img_mult %d", d->img_mult);
  if (d->pair && d->img_mult != 1) return -fail(STCD_ERR_INVALID, "pair ops iterate over chunk_pairs images (img_mult=1)");
  if (d->out_diff >= 0 && !d->pair) return -fail(STCD_ERR_INVALID, "out_diff needs pair=1");
  const int mt = d->pair ? 2 : 1;
  if (2 * mt * d->n_tile > 512)
    return -fail(STCD_ERR_INVALID, "double-buffered accumulators need %d TMEM columns (> 512)", 2 * mt * d->n_tile);
  if (d->pair && (plan->chunk < 1)) return -fail(STCD_ERR_INVALID, "pair op on an empty chunk");
  if (plan->split && (d->fold_cs || d->xf_cs))
    return -fail(STCD_ERR_INVALID, "split precision: no folded or horizontally folded stores");
  if (d->xf_cs) {
    bool ok = d->xf_cs >= 16 && d->xf_cs % 16 == 0 && d->n_tile == 3 * d->xf_cs && d->cout_pad == d->n_tile && d->cout <= d->xf_cs &&
              d->n_phase == 1 && d->osy == 1 && d->osx == 1 && !d->out0_s2d && !d->fold_cs;
    for (int s = 0; s < d->n_src && ok; ++s) ok = d->src_sy[s] == 1 && d->src_sx[s] == 1 && d->src_ex[s] == 0 && d->src_ey[s] == 2;
    for (int t = 0; t < d->n_taps && ok; ++t) ok = d->taps[t].tx == 0 && d->taps[t].ty >= 0 && d->taps[t].ty <= 2;
    for (int c = 0; c < d->n_chunks && ok; ++c) ok = d->chunks[c].bx == 0 && d->chunks[c].by == -1 && d->chunks[c].n_taps == 3;
    if (!ok)
      return -fail(STCD_ERR_INVALID, "horizontal tap folding (xf_cs=%d) needs n_tile == cout_pad == 3*xf_cs, cout <= xf_cs, one phase, "
                   "stride-1 sources with halo (2, 0), three taps (dy, 0) per chunk and a plain (not space-to-depth / folded) store", d->xf_cs);
  }
  if (d->hg < 1 || d->wg < 1 || d->osy < 1 || d->osx < 1) return -fail(STCD_ERR_INVALID, "bad grid/stride");
  for (int s = 0; s < d->n_src; ++s) {
    if (!valid_tensor(plan, d->src[s])) return -fail(STCD_ERR_INVALID, "bad src tensor %d", d->src[s]);
    if (d->src_sy[s] < 1 || d->src_sy[s] > 8 || d->src_sx[s] < 1 || d->src_sx[s] > 8)
      return -fail(STCD_ERR_INVALID, "bad src stride");
    if (d->src_ey[s] < 0 || d->src_ex[s] < 0 || d->src_ey[s] > 32 || d->src_ex[s] > 32)
      return -fail(STCD_ERR_INVALID, "bad halo");
    if ((d->src_sy[s] > 1 || d->src_sx[s] > 1) && (d->src_ey[s] || d->src_ex[s]))
      return -fail(STCD_ERR_INVALID, "strided sources take one box per tap (halo must be 0)");
  }
  const int ho = d->hg * d->osy, wo = d->wg * d->osx;
  const int out_imgs = (d->pair ? 2 : d->img_mult);
  if (d->fold_cs) {
    // all osy*osx phases in one GEMM phase, or the osx horizontal phases in each of osy GEMM phases (oy = 0 .. osy-1, ox = 0)
    const int P = d->osy * d->osx;
    const bool all_folded = d->n_phase == 1 && d->cout == P * d->fold_cs;
    bool x_folded = d->osx > 1 && d->n_phase == d->osy && d->cout == d->osx * d->fold_cs;
    for (int ph = 0; ph < d->n_phase && x_folded; ++ph) x_folded = (d->phase[ph].ox == 0 && d->phase[ph].oy >= 0 && d->phase[ph].oy < d->osy);
    if (P < 2 || !(all_folded || x_folded) || d->fold_cs % 16 || d->fold_cout < 8 || d->fold_cout > d->fold_cs || (d->fold_cout % 8))
      return -fail(STCD_ERR_INVALID, "phase folding: need one GEMM phase with cout == osy*osx*fold_cs, or osy GEMM phases (ox = 0) with "
                   "cout == osx*fold_cs; fold_cs %% 16 == 0, fold_cout %% 8 == 0 "
                   "(got osy=%d osx=%d n_phase=%d cout=%d fold_cs=%d fold_cout=%d)", d->osy, d->osx, d->n_phase, d->cout, d->fold_cs, d->fold_cout);
    if (d->out0 < 0 || d->out0_s2d || d->out_raw >= 0 || d->res >= 0 || d->out_pool >= 0 || d->out_diff >= 0 || d->out_ext >= 0 || d->scale2)
      return -fail(STCD_ERR_INVALID, "phase folding supports the affine + ReLU + out0 epilogue only");
  }
  auto check_out = [&](int id, int hh, int ww, int coff, int mult, const char* name) -> int {
    if (id < 0) return 0;
    if (!valid_tensor(plan, id)) return fail(STCD_ERR_INVALID, "bad %s tensor %d", name, id);
    const Tensor& t = plan->tensors[id];
    if (t.h != hh || t.w != ww || (plan->split ? t.c / 2 : t.c) < coff + (d->fold_cs ? d->fold_cout : d->cout) || t.mult != mult)
      return fail(STCD_ERR_INVALID, "%s tensor %d is [%d*chunk,%d,%d,%d], op writes [%d*chunk,%d,%d,%d+%d]", name, id,
                  t.mult, t.h, t.w, t.c, mult, hh, ww, coff, d->cout);
    return 0;
  };
  const bool bf16_out = d->out0 >= 0 || d->out_raw >= 0 || d->out_pool >= 0 || d->out_diff >= 0 || d->res >= 0;
  if (bf16_out && (d->cout % 8)) return -fail(STCD_ERR_INVALID, "bf16 outputs need cout %% 8 == 0 (cout=%d)", d->cout);
  if (d->out0_coff % 8) return -fail(STCD_ERR_INVALID, "out0_coff must be a multiple of 8");
  if (d->out0_s2d) {
    if (d->out0 < 0 || d->out0_coff || (ho % 2) || (wo % 2) || !valid_tensor(plan, d->out0))
      return -fail(STCD_ERR_INVALID, "space-to-depth out0 needs a tensor, even output dims and no channel offset");
    const Tensor& t = plan->tensors[d->out0];
    // split precision: hi of parity class k at k*cout, lo at 4*cout + k*cout
    if (t.h != ho / 2 || t.w != wo / 2 || t.c != (plan->split ? 8 : 4) * d->cout || t.mult != out_imgs)
      return -fail(STCD_ERR_INVALID, "space-to-depth out0 tensor is [%d*chunk,%d,%d,%d], op writes [%d*chunk,%d,%d,%d*%d]", t.mult, t.h, t.w,
                   t.c, out_imgs, ho / 2, wo / 2, plan->split ? 8 : 4, d->cout);
  } else if (check_out(d->out0, ho, wo, d->out0_coff, out_imgs, "out0")) return -STCD_ERR_INVALID;
  if (check_out(d->out_raw, ho, wo, 0, out_imgs, "out_raw")) return -STCD_ERR_INVALID;
  if (check_out(d->res, ho, wo, 0, out_imgs, "res")) return -STCD_ERR_INVALID;
  if (d->out_pool >= 0) {
    if (d->osy != 1 || d->osx != 1 || d->n_phase != 1 || (ho % 2) || (wo % 2))
      return -fail(STCD_ERR_INVALID, "fused 2x2 max-pool needs a stride-1 single-phase op with even output dims");
    if (check_out(d->out_pool, ho / 2, wo / 2, 0, out_imgs, "out_pool")) return -STCD_ERR_INVALID;
  }
  if (check_out(d->out_diff, ho, wo, 0, 1, "out_diff")) return -STCD_ERR_INVALID;
  if (d->out_ext >= 0 && (d->img_mult != 1 || d->pair)) return -fail(STCD_ERR_INVALID, "external outputs need img_mult=1");
  if (d->n_chunks < 1 || d->n_taps < 1) return -fail(STCD_ERR_INVALID, "empty K-program");
  int blocks_total = 0;
  for (int ph = 0; ph < d->n_phase; ++ph) {
    const stcd_phase& f = d->phase[ph];
    if (f.chunk_begin < 0 || f.chunk_count < 1 || f.chunk_count > stcd::kMaxChunks || f.chunk_begin + f.chunk_count > d->n_chunks)
      return -fail(STCD_ERR_INVALID, "phase %d chunk slice [%d,+%d) out of range", ph, f.chunk_begin, f.chunk_count);
    if (f.oy < 0 || f.oy >= d->osy || f.ox < 0 || f.ox >= d->osx) return -fail(STCD_ERR_INVALID, "phase %d offsets out of range", ph);
    if (f.n_blocks < 1 || f.n_blocks > stcd::kMaxTaps || f.w_block != blocks_total)
      return -fail(STCD_ERR_INVALID, "phase %d: n_blocks %d / w_block %d (expected %d)", ph, f.n_blocks, f.w_block, blocks_total);
    int taps_seen = 0;
    const int tap0 = d->chunks[f.chunk_begin].tap_begin;
    for (int i = 0; i < f.chunk_count; ++i) {
      const stcd_chunk& e = d->chunks[f.chunk_begin + i];
      if (e.src < 0 || e.src >= d->n_src) return -fail(STCD_ERR_INVALID, "chunk %d: src %d", i, e.src);
      const Tensor& t = plan->tensors[d->src[e.src]];
      // a chunk may overhang the tensor's last 8-channel group: TMA zero-fills the missing group
      // a chunk may overhang the tensor by one 8-channel group (TMA zero-fills it) or run into the next parity class
      // of a space-to-depth tensor (those K rows carry zero weights)
      if (e.c0 < 0 || (e.c0 % 8) || e.c0 >= t.c || e.c0 + d->kc > t.c + 8)
        return -fail(STCD_ERR_INVALID, "chunk %d: channels [%d,+%d) of %d", i, e.c0, d->kc, t.c);
      const int top = (d->pair ? 1 : d->img_mult - 1) * plan->chunk + plan->chunk - 1 + e.n_off;
      if (e.n_off < 0 || top >= t.mult * plan->chunk) return -fail(STCD_ERR_INVALID, "chunk %d: image offset %d overruns source", i, e.n_off);
      if (e.n_taps < 1 || e.tap_begin != tap0 + taps_seen || e.tap_begin + e.n_taps > d->n_taps)
        return -fail(STCD_ERR_INVALID, "chunk %d: taps [%d,+%d) not contiguous", i, e.tap_begin, e.n_taps);
      for (int k = 0; k < e.n_taps; ++k) {
        const stcd_tap& tp = d->taps[e.tap_begin + k];
        if (tp.ty < 0 || tp.ty > d->src_ey[e.src] || tp.tx < 0 || tp.tx > d->src_ex[e.src])
          return -fail(STCD_ERR_INVALID, "chunk %d tap %d: (%d,%d) outside the halo (%d,%d)", i, k, tp.ty, tp.tx,
                       d->src_ey[e.src], d->src_ex[e.src]);
      }
      taps_seen += e.n_taps;
    }
    if (taps_seen != f.n_blocks) return -fail(STCD_ERR_INVALID, "phase %d: %d taps but n_blocks %d", ph, taps_seen, f.n_blocks);
    blocks_total += f.n_blocks;
  }
  const int64_t need = (int64_t)(d->cout_pad / d->n_tile) * blocks_total * d->n_tile * d->kc;
  if (d->w_elems != need) return -fail(STCD_ERR_INVALID, "weights: %lld elements, expected %lld", (long long)d->w_elems, (long long)need);

  ConvOp op;
  op.d = *d;
  op.mt = mt;
  op.weights.assign(d->weights, d->weights + d->w_elems);
  op.chunks.assign(d->chunks, d->chunks + d->n_chunks);
  op.taps.assign(d->taps, d->taps + d->n_taps);
  op.scale.assign(d->scale, d->scale + d->cout_pad);
  op.shift.assign(d->shift, d->shift + d->cout_pad);
  if (d->scale2) {
    op.scale2.assign(d->scale2, d->scale2 + d->cout_pad);
    op.shift2.assign(d->shift2, d->shift2 + d->cout_pad);
  }
  op.d.weights = nullptr;
  op.d.chunks = nullptr;
  op.d.taps = nullptr;
  op.d.scale = op.d.shift = op.d.scale2 = op.d.shift2 = nullptr;
  if (d->out_ext >= 0) {
    plan->n_ext = std::max(plan->n_ext, d->out_ext + 1);
    if ((int)plan->ext_elems.size() < plan->n_ext) plan->ext_elems.resize(plan->n_ext, 0);
    plan->ext_elems[d->out_ext] = (size_t)d->cout * ho * wo;
  }
  plan->convs.push_back(std::move(op));
  plan->ops.push_back({0, (int)plan->convs.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_add_ecam_head(stcd_plan* plan, const stcd_ecam_desc* d) {
  if (!plan || !d) return -fail(STCD_ERR_STATE, "plan/desc is NULL");
  if (plan->finalized) return -fail(STCD_ERR_STATE, "plan already finalized");
  if (d->c < 8 || d->c > 64 || (d->c % 8) || d->n_class < 1 || d->n_class > 4 || d->r < 1 || d->r > 16 || d->r1 < 1 || d->r1 > 16)
    return -fail(STCD_ERR_INVALID, "ecam head: c=%d n_class=%d r=%d r1=%d out of range", d->c, d->n_class, d->r, d->r1);
  if (!d->ca_fc1 || !d->ca_fc2 || !d->ca1_fc1 || !d->ca1_fc2 || !d->w_final || !d->b_final || d->out_ext < 0)
    return -fail(STCD_ERR_INVALID, "ecam head: NULL weights / bad out_ext");
  int h = 0, w = 0;
  for (int k = 0; k < 4; ++k) {
    if (!valid_tensor(plan, d->src[k])) return -fail(STCD_ERR_INVALID, "ecam head: bad src tensor %d", d->src[k]);
    const Tensor& t = plan->tensors[d->src[k]];
    if (t.mult != 1 || t.c != (plan->split ? 2 : 1) * d->c || (k && (t.h != h || t.w != w)))
      return -fail(STCD_ERR_INVALID, "ecam head: src %d is [%d*chunk,%d,%d,%d], need [chunk,%d,%d,%d]", k, t.mult, t.h, t.w, t.c, h, w, d->c);
    h = t.h;
    w = t.w;
  }
  EcamOp e;
  e.d = *d;
  const int c4 = 4 * d->c;
  const float* parts[6] = {d->ca_fc1, d->ca_fc2, d->ca1_fc1, d->ca1_fc2, d->w_final, d->b_final};
  const size_t sizes[6] = {(size_t)d->r * c4, (size_t)c4 * d->r, (size_t)d->r1 * d->c, (size_t)d->c * d->r1, (size_t)d->n_class * c4, (size_t)d->n_class};
  for (int i = 0; i < 6; ++i) e.w.insert(e.w.end(), parts[i], parts[i] + sizes[i]);
  e.d.ca_fc1 = e.d.ca_fc2 = e.d.ca1_fc1 = e.d.ca1_fc2 = e.d.w_final = e.d.b_final = nullptr;
  e.hw = h * w;
  plan->n_ext = std::max(plan->n_ext, d->out_ext + 1);
  if ((int)plan->ext_elems.size() < plan->n_ext) plan->ext_elems.resize(plan->n_ext, 0);
  plan->ext_elems[d->out_ext] = (size_t)d->n_class * h * w;
  plan->ecams.push_back(std::move(e));
  plan->ops.push_back({2, (int)plan->ecams.size() - 1});
  return (int)plan->ops.size() - 1;
}

int stcd_plan_finalize(stcd_plan* plan) {
  if (plan && plan->device < 0)
    return fail(STCD_ERR_NO_DEVICE, "validation plan (device -1): descriptors were checked, nothing can run -- libstcd_b200 has no CPU fallback");
  if (!plan) return fail(STCD_ERR_STATE, "plan is NULL");
  if (plan->finalized) return fail(STCD_ERR_STATE, "plan already finalized");
  DeviceGuard dev_guard(plan->device);   // the caller's current device is restored on return
  // ---- activation workspace
  size_t off = 0;
  for (Tensor& t : plan->tensors) {
    t.offset = off;
    off += round_up(t.bytes, 1024);
  }
  plan->workspace_bytes = std::max<size_t>(off, 1024);
  CUDA_TRY(cudaMalloc(&plan->workspace, plan->workspace_bytes));
  CUDA_TRY(cudaMemset(plan->workspace, 0, plan->workspace_bytes));
  for (Tensor& t : plan->tensors) t.ptr = plan->workspace + t.offset;
  // ---- constant arena
  size_t aoff = 0;
  for (ConvOp& op : plan->convs) {
    op.w_off = aoff;
    aoff += round_up(op.weights.size() * 2, 1024);
    op.c_off = aoff;
    aoff += round_up(op.chunks.size() * sizeof(stcd_chunk), 256);
    op.t_off = aoff;
    aoff += round_up(op.taps.size() * sizeof(stcd_tap), 256);
    op.s_off = aoff;
    aoff += round_up((size_t)op.d.cout_pad * 4 * 4, 256);
  }
  plan->arena_bytes = std::max<size_t>(aoff, 1024);
  CUDA_TRY(cudaMalloc(&plan->arena, plan->arena_bytes));
  std::vector<uint8_t> host(plan->arena_bytes, 0);
  for (ConvOp& op : plan->convs) {
    memcpy(host.data() + op.w_off, op.weights.data(), op.weights.size() * 2);
    memcpy(host.data() + op.c_off, op.chunks.data(), op.chunks.size() * sizeof(stcd_chunk));
    memcpy(host.data() + op.t_off, op.taps.data(), op.taps.size() * sizeof(stcd_tap));
    const size_t n = op.d.cout_pad;
    memcpy(host.data() + op.s_off, op.scale.data(), n * 4);
    memcpy(host.data() + op.s_off + n * 4, op.shift.data(), n * 4);
    if (!op.scale2.empty()) {
      memcpy(host.data() + op.s_off + n * 8, op.scale2.data(), n * 4);
      memcpy(host.data() + op.s_off + n * 12, op.shift2.data(), n * 4);
    }
  }
  CUDA_TRY(cudaMemcpy(plan->arena, host.data(), plan->arena_bytes, cudaMemcpyHostToDevice));

  static_assert(sizeof(stcd_chunk) == sizeof(stcd::Chunk), "chunk layout");
  static_assert(sizeof(stcd_tap) == sizeof(stcd::Tap), "tap layout");
  const size_t kSmemMax = 227 * 1024 - 12 * 1024;  // dynamic budget: static tables + barriers live beside it
  int n_kernels = 0;
  static std::vector<stcd::ConvKernelEntry> all_kernels;     // the translation units' tables, concatenated once
  if (all_kernels.empty()) {
    using TableFn = const stcd::ConvKernelEntry* (*)(int*);
    for (TableFn fn : {stcd::conv_kernel_table_a, stcd::conv_kernel_table_b, stcd::conv_kernel_table_c, stcd::conv_kernel_table_d,
                       stcd::conv_kernel_table_e, stcd::conv_kernel_table_f}) {
      int n = 0;
      const stcd::ConvKernelEntry* t = fn(&n);
      all_kernels.insert(all_kernels.end(), t, t + n);
    }
  }
  n_kernels = (int)all_kernels.size();
  const stcd::ConvKernelEntry* kernels = all_kernels.data();
  for (int i = 0; i < n_kernels; ++i)
  {
    CUDA_TRY(cudaFuncSetAttribute(kernels[i].fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
    // one shared-memory carve-out for every instance: consecutive launches never reconfigure the SM
    CUDA_TRY(cudaFuncSetAttribute(kernels[i].fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  }
  // Per-CTA dynamic shared-memory budget for `o` resident CTAs per SM: the SM's capacity split o ways, minus the
  // kernel's STATIC shared memory (tables, barriers, affine vectors) and the 1 KB the driver reserves per CTA.  Sizing
  // against a fixed constant instead let occupancy-2 plans ask for a few KB too much and silently run one CTA per SM.
  size_t static_smem = 0;
  for (int i = 0; i < n_kernels; ++i) {
    cudaFuncAttributes fa;
    CUDA_TRY(cudaFuncGetAttributes(&fa, kernels[i].fn));
    static_smem = std::max(static_smem, fa.sharedSizeBytes);
  }
  int smem_per_sm = 233472;
  CUDA_TRY(cudaDeviceGetAttribute(&smem_per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, plan->device));
  auto cta_budget = [&](int o) -> size_t {
    const size_t share = (size_t)smem_per_sm / o;
    const size_t fixed = static_smem + 1024 + 256;
    return std::min(kSmemMax, share > fixed ? share - fixed : 0);
  };
  plan->pdl = env_int("STCD_PDL", 1);
  // Opt-in (STCD_GRAPH=1).  Measured on B200 (round 2, gpurun_out/gab_*): replaying the captured chunk is NOT faster than the
  // programmatic-dependent-launch chain the plain path already issues -- SiamUnet_diff at 8 pairs: 26.7 k pairs/s plain vs
  // 14.4 k through the graph, ChangeGNNV1: 2 239 vs 1 847 (1 300 in another run), SNUNet / SegCD: equal (profiles/r2_graph_ab.txt).  The small nets are bound by the device-side
  // fill / drain of each kernel (4-11 us from the end of one layer to the first MMA of the next), not by host launch cost.
  plan->graph_mode = env_int("STCD_GRAPH", 0);
  const int force_generic = env_int("STCD_FORCE_GENERIC", 0);
  int n_sm = 148;
  CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, plan->device));

  const int force_occ_env = env_int("STCD_FORCE_OCC", 0);
  const int min_stages_occ2 = std::max(2, env_int("STCD_MIN_STAGES_OCC2", 2));  // two CTAs per SM with 2 A stages each beat one CTA with 8
  const int force_stream = env_int("STCD_FORCE_WSTREAM", 0);
  // One conv op -> tensor maps, shared-memory plan, kernel instance, grid.  mt_override > 0 forces the number of M sub-tiles per CTA
  // pass (the autotuner below re-runs it per candidate); 0 = the heuristics.
  // tune_flags: bit 0 flips the folded-layer issue-loop choice, bit 1 forbids the eight-epilogue-warp instance, bit 2 plans for ONE
  // CTA per SM where two would fit (deeper rings, and the eight-epilogue-warp instances become eligible).
  auto configure = [&](ConvOp& op, int mt_override, int tune_flags) -> int {
    const int force_occ = (tune_flags & 4) ? 1 : force_occ_env;
    const stcd_conv_desc& d = op.d;
    memset(&op.tm, 0, sizeof(op.tm));
    stcd::ConvParams& p = op.p;
    memset(&p, 0, sizeof(p));
    size_t a_sub = 0;
    const bool xf = d.xf_cs > 0;
    const int tile_w = xf ? stcd::kXfTileW : stcd::kTileW, tile_h = xf ? stcd::kXfTileH : stcd::kTileH;
    const int tile_step_x = xf ? stcd::kXfStep : stcd::kTileW;      // output columns per tile
    for (int s = 0; s < d.n_src; ++s) {
      const Tensor& t = plan->tensors[d.src[s]];
      int r = encode_act_map(&op.tm.src[s], t.ptr, t.mult * plan->chunk, t.h, t.w, t.c, d.kc, d.src_sx[s], d.src_sy[s],
                             d.src_ex[s], d.src_ey[s], tile_w, tile_h);
      if (r) return r;
      p.src_sy[s] = d.src_sy[s];
      p.src_sx[s] = d.src_sx[s];
      p.src_merged[s] = (d.src_sx[s] == 1 && d.src_sy[s] == 1) ? 1 : 0;
      p.src_pw[s] = tile_w + d.src_ex[s];
      p.src_ph[s] = tile_h + d.src_ey[s];
      a_sub = std::max(a_sub, (size_t)(d.kc / 8) * p.src_pw[s] * p.src_ph[s] * 16);
    }
    p.hg = d.hg;
    p.wg = d.wg;
    p.tiles_x = (d.wg + tile_step_x - 1) / tile_step_x;
    p.tiles_y = (d.hg + tile_h - 1) / tile_h;
    p.xf_cs = d.xf_cs;
    p.n_ntiles = d.cout_pad / d.n_tile;
    p.osy = d.osy;
    p.osx = d.osx;
    p.ho = d.hg * d.osy;
    p.wo = d.wg * d.osx;
    p.n_phase = d.n_phase;
    p.n_src = d.n_src;
    int max_blocks = 0, blocks_total = 0;
    for (int ph = 0; ph < d.n_phase; ++ph) {
      p.phase[ph] = {d.phase[ph].chunk_begin, d.phase[ph].chunk_count, d.phase[ph].oy, d.phase[ph].ox, d.phase[ph].w_block,
                     d.phase[ph].n_blocks, d.phase[ph].chunk_count > 0 ? op.chunks[d.phase[ph].chunk_begin].tap_begin : 0};
      max_blocks = std::max(max_blocks, d.phase[ph].n_blocks);
      blocks_total += d.phase[ph].n_blocks;
    }
    p.blocks_per_ntile = blocks_total;
    p.chunks = reinterpret_cast<const stcd::Chunk*>(plan->arena + op.c_off);
    p.taps = reinterpret_cast<const stcd::Tap*>(plan->arena + op.t_off);
    p.wpack = plan->arena + op.w_off;
    p.kc = d.kc;
    p.n_tile = d.n_tile;
    p.cout = d.cout;
    p.wblk_bytes = (uint32_t)d.n_tile * d.kc * 2;
    p.a_sub_bytes = (uint32_t)round_up(a_sub, 128);
    p.tab_bytes = (uint32_t)round_up((size_t)max_blocks * (d.kc / 16) * 8, 128);
    const size_t w_all = (size_t)max_blocks * p.wblk_bytes;
    const int groups = d.n_phase * p.n_ntiles;
    // ---- M tiles per CTA pass (sub-tiles sharing every weight block) and the shared-memory plan.
    // base: 1 image, or the (T1, T2) pair.  More sub-tiles = other images of the chunk: when the
    // weights do not fit in shared memory they are re-streamed from L2 for every pass, so the widest
    // pass that fits TMEM (2 accumulator sets) and shared memory wins; weight-stationary layers
    // keep the base width (more, smaller tiles balance better over the SMs).
    const int base_mt = d.pair ? 2 : 1;
    const int base_imgs = (d.pair ? 1 : d.img_mult) * plan->chunk;
    int occ = 0;
    auto try_plan = [&](int mt) -> bool {
      const int g = mt / base_mt;
      if (base_imgs % g) return false;
      if (2 * mt * d.n_tile > 512) return false;
      if (d.out_ext >= 0 && mt > 2) return false;
      p.mt = mt;
      p.a_stage_bytes = mt * p.a_sub_bytes;
      p.acc_cols = mt * d.n_tile;
      uint32_t cols = 32;
      while (cols < 2 * p.acc_cols) cols <<= 1;
      p.tmem_cols = cols;
      occ = 0;
      for (int o = 2; o >= 1 && !occ; --o) {
        if (force_occ && o != force_occ) continue;
        if (cols * o > 512) continue;
        if (cta_budget(o) < 256 + p.tab_bytes + 2 * (size_t)p.a_stage_bytes) continue;
        const size_t budget = cta_budget(o) - 256 - p.tab_bytes;
        const int min_stages = (o == 2) ? min_stages_occ2 : 2;
        if (!force_stream && w_all + (size_t)min_stages * p.a_stage_bytes <= budget) {
          occ = o;
          p.w_resident = 1;
          p.w_stages = 0;
          p.a_stages = (int)std::min<size_t>(stcd::kMaxAStages, (budget - round_up(w_all, 128)) / p.a_stage_bytes);
        } else if (o == 1) {
          const size_t a_min = 2 * (size_t)p.a_stage_bytes;
          if (a_min + 2 * (size_t)p.wblk_bytes > budget) return false;
          occ = 1;
          p.w_resident = 0;
          p.w_stages = (int)std::min<size_t>(std::min<size_t>(stcd::kMaxWStages, (size_t)max_blocks),
                                             std::max<size_t>(2, (budget - a_min - (size_t)p.a_stage_bytes) / p.wblk_bytes));
          p.a_stages = (int)std::min<size_t>(stcd::kMaxAStages,
                                             (budget - round_up((size_t)p.w_stages * p.wblk_bytes, 128)) / p.a_stage_bytes);
          if (p.a_stages < 2) return false;
        }
      }
      return occ != 0;
    };
    {
      const int force_mt = mt_override > 0 ? mt_override : env_int("STCD_FORCE_MT", 0);
      bool ok = false;
      if (force_mt && force_mt % base_mt == 0) ok = try_plan(force_mt);
      if (!ok) {
        ok = try_plan(base_mt);
        if (ok && p.w_resident && !force_mt && d.n_phase == 1 && d.phase[0].chunk_count >= 3) {
          // deep-K weight-stationary layers: wider passes amortise the per-chunk pipeline costs,
          // as long as the weights stay resident
          for (int mt = 4; mt > base_mt; mt >>= 1) {
            const int passes = p.tiles_x * p.tiles_y * (base_imgs / (mt / base_mt));
            if (passes < 2 * n_sm / groups) continue;
            if (try_plan(mt) && p.w_resident) break;
            ok = try_plan(base_mt);
          }
        } else if (ok && !p.w_resident && !force_mt) {
          // weights streamed per pass: widen while it fits and every SM still gets >= 2 passes
          for (int mt = 4; mt > base_mt; mt >>= 1) {
            const int passes = p.tiles_x * p.tiles_y * (base_imgs / (mt / base_mt));
            if (passes < 2 * n_sm / groups) continue;
            if (try_plan(mt)) break;
            ok = try_plan(base_mt);
          }
        }
      }
      if (!ok) occ = 0;
    }
    // ---- regular phases: per-MMA operand offsets into the constant bank (fast issue path)
    for (int ph = 0; ph < d.n_phase; ++ph) {
      const stcd_phase& f = d.phase[ph];
      const stcd_chunk& c0 = op.chunks[f.chunk_begin];
      const int ksteps = d.kc / 16;
      bool regular = c0.n_taps * ksteps <= stcd::kFastMma && !env_int("STCD_NO_FAST", 0);
      const int pw = p.src_pw[c0.src], phh = p.src_ph[c0.src];
      for (int i = 0; i < f.chunk_count && regular; ++i) {
        const stcd_chunk& c = op.chunks[f.chunk_begin + i];
        if (c.n_taps != c0.n_taps || p.src_pw[c.src] != pw || p.src_ph[c.src] != phh) regular = false;
        for (int k = 0; k < c.n_taps && regular; ++k)
          if (op.taps[c.tap_begin + k].ty != op.taps[c0.tap_begin + k].ty || op.taps[c.tap_begin + k].tx != op.taps[c0.tap_begin + k].tx)
            regular = false;
      }
      p.f_regular[ph] = regular ? 1 : 0;
      if (!regular) continue;
      p.f_nmma[ph] = c0.n_taps * ksteps;
      p.f_a_hi[ph] = (xf ? 8u : ((uint32_t)pw & 0x3FFF)) | (1u << 14);     // SBO: the next 8 pixels of M (XF: 128 B throughout)
      p.f_a_lo_lbo[ph] = ((uint32_t)(pw * phh) & 0x3FFF) << 16;
      p.f_b_chunk16[ph] = (uint32_t)c0.n_taps * (p.wblk_bytes >> 4);
      for (int k = 0; k < c0.n_taps; ++k)
        for (int ks = 0; ks < ksteps; ++ks) {
          const uint32_t a = (uint32_t)(op.taps[c0.tap_begin + k].ty * pw + op.taps[c0.tap_begin + k].tx) + (uint32_t)ks * 2u * pw * phh;
          const uint32_t b = (uint32_t)k * (p.wblk_bytes >> 4) + (uint32_t)ks * 2u * d.n_tile;
          if (a > 0xFFFFu || b > 0xFFFFu) return fail(STCD_ERR_INVALID, "fast-path offset overflow");
          p.f_off[ph][k * ksteps + ks] = a | (b << 16);
        }
    }
    op.mt = p.mt;
    op.occ = occ;
    {
      const int g = op.mt / base_mt;
      p.n_img = base_imgs / g;
      p.n_tiles = p.tiles_x * p.tiles_y * p.n_img;
      for (int m = 0; m < op.mt; ++m)
        p.m_off[m] = d.pair ? (m & 1) * plan->chunk + (m >> 1) * p.n_img : m * p.n_img;
    }
    if (!occ) return fail(STCD_ERR_INVALID, "conv op: no shared-memory plan (forced occupancy %d)", force_occ);
    const size_t w_region = round_up(p.w_resident ? w_all : (size_t)p.w_stages * p.wblk_bytes, 128);
    // ---- residual ring: a dedicated warp fetches the residual by TMA in blocks of `res_rb` channels of the MS sub-tiles the
    // epilogue finishes together (slot <= 16 KB), up to kMaxRSlots blocks ahead, when >= 2 slots (32 KB when there is room)
    // fit beside >= 2 A stages; else the epilogue loads the residual itself
    p.res_slots = 0;
    p.split = plan->split;
    if (d.res >= 0 && d.n_phase == 1 && d.osy == 1 && d.osx == 1 && !plan->split && env_int("STCD_RES_SMEM", 1)) {
      const Tensor& tr = plan->tensors[d.res];
      const int ms = d.pair ? 2 : 1;
      p.res_ch = xf ? d.xf_cs : d.n_tile;
      int rb = 64 / ms;                                   // 16 KB slots: 64 channels of one stream, 32 of a Siamese pair
      while (rb > 16 && rb > p.res_ch) rb >>= 1;
      p.res_rb = rb;
      const size_t sub = (size_t)rb * tile_h * tile_w * 2;                         // [res_rb / 8][tile rows][tile px][8] bf16
      const size_t slot = sub * ms;
      const size_t fixed = 256 + p.tab_bytes + w_region;
      const size_t budget = cta_budget(occ);
      if (tr.h == p.ho && tr.w == p.wo) {
        // four blocks in flight (32-64 KB) cover the DRAM latency; more would take the room of the activation stages, which
        // matter more (eight 8 KB slots instead of four cost SNUNet's conv0_x.conv2 three of its five A stages: 190 -> 237 us)
        for (int r = 4; r >= 2 && !p.res_slots; --r) {
          const int a_min = std::min(p.a_stages, r >= 3 ? 3 : 2);
          if (fixed + (size_t)a_min * p.a_stage_bytes + r * slot > budget) continue;
          p.res_slots = r;
          p.res_slot_bytes = (uint32_t)slot;
          p.res_sub_bytes = (uint32_t)sub;
          p.a_stages = (int)std::min<size_t>(p.a_stages, (budget - fixed - r * slot) / p.a_stage_bytes);
        }
      }
      if (p.res_slots) {
        int r = encode_act_map(&op.tm.res, tr.ptr, tr.mult * plan->chunk, tr.h, tr.w, tr.c, p.res_rb, 1, 1, 0, 0, tile_w, tile_h);
        if (r) return r;
      }
    }
    op.smem = p.tab_bytes + w_region + (size_t)p.a_stages * p.a_stage_bytes + (size_t)p.res_slots * p.res_slot_bytes + 128;
    if (op.smem > kSmemMax) return fail(STCD_ERR_INVALID, "conv op needs %zu B of shared memory", op.smem);
    const int ctas = std::max(1, (n_sm * occ) / groups);
    op.grid = dim3((unsigned)std::min(p.n_tiles, ctas), (unsigned)p.n_ntiles, (unsigned)d.n_phase);
    p.dbg = env_int("STCD_DBG", 0);
    p.xf_fast = (xf && d.n_phase == 1 && d.phase[0].chunk_count >= env_int("STCD_XF_FAST_MIN", 4)) ? 1 : 0;
    if (xf && d.n_phase == 1 && (tune_flags & 1)) p.xf_fast ^= 1;
    p.reverse = (env_int("STCD_SERPENTINE", 1) && ((&op - &plan->convs[0]) & 1)) ? 1 : 0;
    if (env_int("STCD_TRACE", 0) && !op.trace) {
      const size_t nb = (size_t)op.grid.x * op.grid.y * op.grid.z * 16 * sizeof(long long);
      CUDA_TRY(cudaMalloc(&op.trace, nb));
      CUDA_TRY(cudaMemset(op.trace, 0, nb));
      p.trace = op.trace;
    }
    const float* sc = reinterpret_cast<const float*>(plan->arena + op.s_off);
    p.scale = sc;
    p.shift = sc + d.cout_pad;
    if (!op.scale2.empty()) {
      p.scale2 = sc + 2 * d.cout_pad;
      p.shift2 = sc + 3 * d.cout_pad;
    }
    p.relu = d.relu;
    p.act_pre = d.act_pre;
    p.act_alpha = d.act_alpha;
    // epilogue features -> kernel instance (specialised when one exists, else the generic one)
    op.epi = (d.out_raw >= 0 ? stcd::E_RAW : 0u) | (!op.scale2.empty() ? stcd::E_AFF2 : 0u) | (d.res >= 0 ? stcd::E_RES : 0u) |
             (d.relu ? stcd::E_RELU : 0u) | (d.out0 >= 0 ? stcd::E_OUT0 : 0u) | (d.out_pool >= 0 ? stcd::E_POOL : 0u) |
             (d.out_diff >= 0 ? stcd::E_DIFF : 0u) | (d.out_ext >= 0 ? stcd::E_F32 : 0u) |
             ((d.relu >= 2 || d.act_pre) ? stcd::E_ACTX : 0u) | (p.res_slots ? stcd::E_RSM : 0u) | (xf ? stcd::E_XF : 0u);
    op.fn = nullptr;
    op.threads = stcd::kConvThreads;
    // plans that run one CTA per SM anyway take the eight-epilogue-warp instance when there is one (>= 2 column steps to share)
    const bool want8 = !(tune_flags & 2) && occ == 1 && (xf ? (d.xf_cs >= 32 && env_int("STCD_XF_EPI8", 1) != 0) : d.n_tile >= 32) && env_int("STCD_EPI8", 1) != 0;
    for (int i = 0; i < n_kernels && !force_generic && !plan->split; ++i)     // split precision lives in the generic instances
      if (kernels[i].mt == op.mt && kernels[i].ms == (d.pair ? 2 : 1) && kernels[i].epi == op.epi && (kernels[i].ne == 4 || want8)) {
        if (op.fn && kernels[i].ne == 4) continue;       // an eight-warp instance found earlier wins
        op.fn = kernels[i].fn;
        op.threads = kernels[i].ne == 8 ? stcd::kConvThreads8 : stcd::kConvThreads;
        if (kernels[i].ne == 8) break;
      }
    for (int i = 0; i < n_kernels && !op.fn; ++i)
      if (kernels[i].mt == op.mt && kernels[i].ms == (d.pair ? 2 : 1) && kernels[i].epi == (stcd::E_GENERIC | (xf ? stcd::E_XF : 0u))) op.fn = kernels[i].fn;
    if (!op.fn) return fail(STCD_ERR_INVALID, "no conv kernel instance for mt=%d", op.mt);
    if (d.res >= 0) {
      p.res = (const __nv_bfloat16*)plan->tensors[d.res].ptr;
      p.res_c8 = plan->tensors[d.res].c / 8;
    }
    if (d.out0 >= 0) {
      p.out0 = (__nv_bfloat16*)plan->tensors[d.out0].ptr;
      p.out0_c8 = plan->tensors[d.out0].c / 8;
      p.out0_coff = d.out0_coff;
      p.out0_s2d = d.out0_s2d;
      p.fold_cs = d.fold_cs;
      p.fold_cout = d.fold_cout;
    }
    if (d.out_raw >= 0) {
      p.out_raw = (__nv_bfloat16*)plan->tensors[d.out_raw].ptr;
      p.out_raw_c8 = plan->tensors[d.out_raw].c / 8;
    }
    if (d.out_pool >= 0) {
      p.out_pool = (__nv_bfloat16*)plan->tensors[d.out_pool].ptr;
      p.out_pool_c8 = plan->tensors[d.out_pool].c / 8;
    }
    if (d.out_diff >= 0) {
      p.out_diff = (__nv_bfloat16*)plan->tensors[d.out_diff].ptr;
      p.out_diff_c8 = plan->tensors[d.out_diff].c / 8;
    }
    return STCD_OK;
  };
  for (ConvOp& op : plan->convs) {
    const int r = configure(op, 0, 0);
    if (r) return r;
  }
  // ---- Autotune the M sub-tiles per CTA pass, then the folded-layer issue loop and the epilogue width (STCD_AUTOTUNE=0: off).  How many images share a weight block in one pass
  // trades weight reuse and per-tile overheads against tile count, TMEM columns and occupancy, and no static rule gets every layer
  // right: with the heuristic's choice forced to 2 or 4 instead, SNUNet's `conv1_x.conv2` / `conv4_0` run 14-19 % faster at 2,
  // `conv0_0.conv1` 17 % and `conv1_x.conv1` / `Up1_x` 6-7 % faster at 4, while `conv0_x.conv2` and `Up1_x` lose 25-38 % at the other
  // setting (round 2, per-op A/B on one box).  So each op is timed on the plan's own workspace with every admissible count (the data
  // is whatever the workspace holds: the kernels' time does not depend on values) and keeps the fastest; a candidate must win by
  // 4 % to displace the heuristic.  Results do not depend on the choice: a sub-tile's MMAs and epilogue are the same sequence.
  if (env_int("STCD_AUTOTUNE", 1) && !env_int("STCD_FORCE_MT", 0) && !env_int("STCD_TRACE", 0)) {
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    cudaStream_t st = nullptr;
    auto time_op = [&](const ConvOp& op, float* ms_out) -> int {
      float best = 1e30f;
      for (int rep = 0; rep < 4; ++rep) {               // first launch = warm-up
        CUDA_TRY(cudaEventRecord(e0, st));
        const int r = launch_conv(plan, op, plan->chunk, nullptr, st);
        if (r) return r;
        CUDA_TRY(cudaEventRecord(e1, st));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0) best = std::min(best, ms);
      }
      *ms_out = best;
      return STCD_OK;
    };
    for (ConvOp& op : plan->convs) {
      if (op.d.out_ext >= 0) continue;                  // writes a caller-owned buffer that does not exist yet
      const int mt0 = op.mt;
      float t0 = 0.f;
      int r = time_op(op, &t0);
      if (r) return r;
      int best_mt = 0, best_flags = 0;                  // 0 / 0 = the heuristics' own choice
      float best_t = t0 * 0.96f;
      const int base_mt = op.d.pair ? 2 : 1;
      for (int mt = base_mt; mt <= 4; mt <<= 1) {
        if (mt == mt0) continue;
        if (configure(op, mt, 0) != STCD_OK || op.mt != mt) continue;      // not admissible: the heuristics answered instead
        float t = 0.f;
        r = time_op(op, &t);
        if (r) return r;
        if (t < best_t) {
          best_t = t;
          best_mt = mt;
        }
      }
      // with the pass width settled: one CTA per SM where two were planned, four epilogue warps where eight were taken, and the
      // folded-layer issue loop the other way round
      for (int flag = 4; flag >= 1; flag >>= 1) {       // occupancy first: it decides whether eight epilogue warps are on the table
        if (configure(op, best_mt, best_flags) != STCD_OK) break;
        if (flag == 4 && op.occ != 2) continue;
        if (flag == 1 && !(op.d.xf_cs > 0 && op.d.n_phase == 1)) continue;
        if (flag == 2 && op.threads != stcd::kConvThreads8) continue;
        if (configure(op, best_mt, best_flags | flag) != STCD_OK) continue;
        float t = 0.f;
        r = time_op(op, &t);
        if (r) return r;
        if (t < best_t) {
          best_t = t;
          best_flags |= flag;
        }
      }
      r = configure(op, best_mt, best_flags);
      if (r) return r;
      if (env_int("STCD_AUTOTUNE_LOG", 0))
        fprintf(stderr, "autotune conv %3d  mt %d -> %d flags %d (%.1f us -> %.1f us)\n", (int)(&op - &plan->convs[0]), mt0, op.mt, best_flags, t0 * 1e3f,
                ((best_mt || best_flags) ? best_t : t0) * 1e3f);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CUDA_TRY(cudaDeviceSynchronize());
  }
  for (GraphOp& g : plan->graphs) {
    const Tensor& ts = plan->tensors[g.src];
    const size_t B = (size_t)ts.mult * plan->chunk, N = (size_t)ts.h * ts.w, M = N / (g.r * g.r);
    CUDA_TRY(cudaMalloc(&g.xf, B * g.c * N * sizeof(float)));
    if (g.r > 1) CUDA_TRY(cudaMalloc(&g.yf, B * g.c * M * sizeof(float)));
    const bool knn_pipe = env_int("STCD_KNN_MMA", 1) != 0 && g.k * g.dilation <= 27 && M <= (size_t)stcd::kKnnM;
    if (knn_pipe) {
      CUDA_TRY(cudaMalloc(&g.xp, knn_planes_bytes((int)B, g.c, (int)N)));
      CUDA_TRY(cudaMemset(g.xp, 0, knn_planes_bytes((int)B, g.c, (int)N)));      // padding rows / groups stay zero for good
      CUDA_TRY(cudaMalloc(&g.xsq, knn_sq_bytes((int)B, (int)N)));
      CUDA_TRY(cudaMemset(g.xsq, 0, knn_sq_bytes((int)B, (int)N)));
      if (g.r > 1) {
        CUDA_TRY(cudaMalloc(&g.yp, knn_planes_bytes((int)B, g.c, (int)M)));
        CUDA_TRY(cudaMemset(g.yp, 0, knn_planes_bytes((int)B, g.c, (int)M)));
        CUDA_TRY(cudaMalloc(&g.ysq, knn_sq_bytes((int)B, (int)M)));
        CUDA_TRY(cudaMemset(g.ysq, 0, knn_sq_bytes((int)B, (int)M)));
      }
    } else {
      CUDA_TRY(cudaMalloc(&g.xn, B * g.c * N * sizeof(float)));
      if (g.r > 1) CUDA_TRY(cudaMalloc(&g.yn, B * g.c * M * sizeof(float)));
    }
    CUDA_TRY(cudaMalloc(&g.idx, B * N * g.k * sizeof(long long)));
    if (!g.relpos.empty()) {
      CUDA_TRY(cudaMalloc(&g.relpos_dev, g.relpos.size() * sizeof(float)));
      CUDA_TRY(cudaMemcpy(g.relpos_dev, g.relpos.data(), g.relpos.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
  }
  // the 3-stream head instances stage 58 KB: dynamic shared memory above the 48 KB default
  CUDA_TRY(cudaFuncSetAttribute(stcd::segcd_head_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  for (ChanAttnOp& k : plan->chan_attns) {
    CUDA_TRY(cudaMalloc(&k.w_dev, k.w.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.w_dev, k.w.data(), k.w.size() * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&k.psum, (size_t)plan->chunk * k.ranges * k.c_tot * sizeof(float)));
    CUDA_TRY(cudaMalloc(&k.pmax, (size_t)plan->chunk * k.ranges * k.c_tot * sizeof(float)));
    CUDA_TRY(cudaMalloc(&k.gate, (size_t)plan->chunk * k.c_tot * sizeof(float)));
  }
  for (GlGateOp& k : plan->gl_gates) {
    const Tensor& ts = plan->tensors[k.src];
    const size_t B = (size_t)ts.mult * plan->chunk;
    CUDA_TRY(cudaMalloc(&k.w_dev, k.w.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.w_dev, k.w.data(), k.w.size() * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&k.psum, B * k.ranges * k.c * sizeof(float)));
    CUDA_TRY(cudaMalloc(&k.pmax, B * k.ranges * k.c * sizeof(float)));
    CUDA_TRY(cudaMalloc(&k.stats, B * ts.h * ts.w * sizeof(float2)));
  }
  for (VffmOp& k : plan->vffms) {
    const Tensor& ts = plan->tensors[k.mixed];
    const size_t B = (size_t)ts.mult * plan->chunk;
    CUDA_TRY(cudaMalloc(&k.w_dev, k.w.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.w_dev, k.w.data(), k.w.size() * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&k.psum, B * k.ranges * k.c * sizeof(float)));
    CUDA_TRY(cudaMalloc(&k.pmax, B * k.ranges * k.c * sizeof(float)));
  }
  for (SpatialGateOp& k : plan->spatial_gates) {
    const Tensor& ts = plan->tensors[k.src];
    CUDA_TRY(cudaMalloc(&k.w_dev, k.w.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.w_dev, k.w.data(), k.w.size() * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&k.stats, (size_t)ts.mult * plan->chunk * ts.h * ts.w * sizeof(float2)));
  }
  for (BitOp& k : plan->bits) {
    CUDA_TRY(cudaMalloc(&k.w_dev, k.w.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.w_dev, k.w.data(), k.w.size() * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&k.tokens, (size_t)2 * plan->chunk * stcd::kBitL * stcd::kBitC * sizeof(float)));
    CUDA_TRY(cudaMalloc(&k.coef, (size_t)2 * plan->chunk * k.d.n_dec * stcd::kBitCoef * sizeof(float)));
    CUDA_TRY(cudaMalloc(&k.tok_mixed, (size_t)plan->chunk * 2 * stcd::kBitL * stcd::kBitC * sizeof(float)));
    CUDA_TRY(cudaFuncSetAttribute(stcd::bit_token_mixer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.mixer_smem));
    CUDA_TRY(cudaFuncSetAttribute(stcd::bit_coef_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.coef_smem));
  }
  for (GateOp& k : plan->gates) {
    const Tensor& ts = plan->tensors[k.src];
    CUDA_TRY(cudaMalloc(&k.w_dev, k.w.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.w_dev, k.w.data(), k.w.size() * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&k.partial, (size_t)ts.mult * plan->chunk * k.ranges * k.c * sizeof(float)));
  }
  for (LayerNormOp& k : plan->lns) {
    CUDA_TRY(cudaMalloc(&k.gb_dev, k.gb.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.gb_dev, k.gb.data(), k.gb.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  for (DWConvOp& k : plan->dws) {
    CUDA_TRY(cudaMalloc(&k.wb_dev, k.wb.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.wb_dev, k.wb.data(), k.wb.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  for (SegHeadOp& k : plan->heads) {
    CUDA_TRY(cudaMalloc(&k.w_dev, k.w.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(k.w_dev, k.w.data(), k.w.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  for (EcamOp& e : plan->ecams) {
    const stcd_ecam_desc& d = e.d;
    const int c4 = 4 * d.c;
    CUDA_TRY(cudaMalloc(&e.w_dev, e.w.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(e.w_dev, e.w.data(), e.w.size() * sizeof(float), cudaMemcpyHostToDevice));
    stcd::EcamParams& q = e.p;
    memset(&q, 0, sizeof(q));
    for (int k = 0; k < 4; ++k) q.src[k] = (const __nv_bfloat16*)plan->tensors[d.src[k]].ptr;
    q.c = d.c;
    q.split = plan->split;
    q.hw = e.hw;
    q.n_img = plan->chunk;
    q.n_class = d.n_class;
    q.r = d.r;
    q.r1 = d.r1;
    q.ranges = std::max(1, std::min(16, e.hw / 4096));
    CUDA_TRY(cudaMalloc(&e.partial, (size_t)plan->chunk * q.ranges * 2 * 5 * d.c * sizeof(float)));
    q.partial = e.partial;
    const float* wp = e.w_dev;
    q.ca_fc1 = wp;
    wp += (size_t)d.r * c4;
    q.ca_fc2 = wp;
    wp += (size_t)c4 * d.r;
    q.ca1_fc1 = wp;
    wp += (size_t)d.r1 * d.c;
    q.ca1_fc2 = wp;
    wp += (size_t)d.c * d.r1;
    q.w_final = wp;
    wp += (size_t)d.n_class * c4;
    q.b_final = wp;
  }
  plan->finalized = true;
  return STCD_OK;
}

int stcd_plan_tensor_copy(stcd_plan* plan, int tensor_id, void* host, int64_t bytes, int to_device) {
  if (!plan || !plan->finalized) return fail(STCD_ERR_STATE, "plan not finalized");
  if (!valid_tensor(plan, tensor_id) || !host) return fail(STCD_ERR_INVALID, "bad tensor id %d / NULL host buffer", tensor_id);
  const Tensor& t = plan->tensors[tensor_id];
  if (bytes != (int64_t)t.bytes) return fail(STCD_ERR_INVALID, "tensor %d has %zu bytes, got %lld", tensor_id, t.bytes, (long long)bytes);
  DeviceGuard dev_guard(plan->device);   // the caller's current device is restored on return
  CUDA_TRY(cudaDeviceSynchronize());
  if (to_device)
    CUDA_TRY(cudaMemcpy(t.ptr, host, t.bytes, cudaMemcpyHostToDevice));
  else
    CUDA_TRY(cudaMemcpy(host, t.ptr, t.bytes, cudaMemcpyDeviceToHost));
  return STCD_OK;
}

int64_t stcd_plan_read_trace(stcd_plan* plan, int op_index, int64_t* host, int64_t max_words, int32_t* info) {
  if (!plan || !plan->finalized || op_index < 0 || op_index >= (int)plan->ops.size() || plan->ops[op_index].kind != 0) return -1;
  const ConvOp& op = plan->convs[plan->ops[op_index].idx];
  if (info) {
    info[0] = op.grid.x; info[1] = op.grid.y * op.grid.z; info[2] = (int)op.smem; info[3] = op.p.a_stages; info[4] = op.p.w_stages;
    info[5] = op.p.w_resident; info[6] = op.p.tmem_cols; info[7] = op.p.n_tiles; info[8] = op.p.a_stage_bytes; info[9] = op.p.wblk_bytes;
  }
  if (!op.trace || !host) return 0;
  const int64_t n = std::min<int64_t>(max_words, (int64_t)op.grid.x * op.grid.y * op.grid.z * 16);
  cudaDeviceSynchronize();
  if (cudaMemcpy(host, op.trace, n * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return n;
}

int64_t stcd_plan_workspace_bytes(const stcd_plan* plan) {
  return plan ? (int64_t)(plan->workspace_bytes + plan->arena_bytes) : 0;
}

int64_t stcd_plan_launches(const stcd_plan* plan, int n_pairs) {
  if (!plan || n_pairs < 1) return 0;
  const int64_t chunks = (n_pairs + plan->chunk - 1) / plan->chunk;
  int64_t per_chunk = (int64_t)plan->ops.size() + (int64_t)plan->ecams.size();  // an ECAM head op is two kernels
  per_chunk += (int64_t)plan->gates.size();                                    // a channel gate is two kernels
  for (const ChanAttnOp& k : plan->chan_attns) per_chunk += 2 * k.n_src;      // stats + apply per segment, one FC kernel
  per_chunk += (int64_t)plan->spatial_gates.size();                            // statistics + apply
  per_chunk += 2 * (int64_t)plan->gl_gates.size() + (int64_t)plan->vffms.size();  // 3 kernels / 2 kernels
  per_chunk += 3 * (int64_t)plan->bits.size();                                 // tokenizer + mixer + coefficients + decoder
  for (const GraphOp& g : plan->graphs) per_chunk += 3 + (g.r > 1 ? 2 : 0);     // unpack, [pool], norm, [norm y], kNN, max-relative
  return chunks * per_chunk;
}

// One chunk through a cached CUDA graph when this exact (inputs, outputs, n_valid) has been seen before, else plain launches.
static int run_chunk_graphed(stcd_plan* plan, const void* x1, const void* x2, int nv, float* const* outs, int n_outs, cudaStream_t st) {
  if (!plan->graph_mode) return run_chunk(plan, x1, x2, nv, outs, st);
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
    cudaGetLastError();                       // the caller is capturing its own graph: just record the launches into it
    return run_chunk(plan, x1, x2, nv, outs, st);
  }
  stcd_plan::GraphEntry* e = nullptr;
  for (auto& g : plan->graph_cache) {
    if (g.x1 != x1 || g.x2 != x2 || g.n_valid != nv || (int)g.outs.size() != n_outs) continue;
    bool same = true;
    for (int k = 0; k < n_outs && same; ++k) same = (g.outs[k] == outs[k]);
    if (same) {
      e = &g;
      break;
    }
  }
  const uint64_t now = ++plan->graph_clock;
  if (e && e->exec) {
    e->last_use = now;
    CUDA_TRY(cudaGraphLaunch(e->exec, st));
    return STCD_OK;
  }
  if (!e) {                                   // first sighting: remember the key (evict the least recently used), launch plainly
    if (plan->graph_cache.size() >= kGraphCacheSize) {
      size_t lru = 0;
      for (size_t i = 1; i < plan->graph_cache.size(); ++i)
        if (plan->graph_cache[i].last_use < plan->graph_cache[lru].last_use) lru = i;
      if (plan->graph_cache[lru].exec) cudaGraphExecDestroy(plan->graph_cache[lru].exec);
      plan->graph_cache.erase(plan->graph_cache.begin() + lru);
    }
    stcd_plan::GraphEntry g;
    g.x1 = x1;
    g.x2 = x2;
    g.n_valid = nv;
    g.outs.assign(outs, outs + n_outs);
    g.seen = 1;
    g.last_use = now;
    plan->graph_cache.push_back(g);
    return run_chunk(plan, x1, x2, nv, outs, st);
  }
  // second sighting: capture the launch list on the plan's own stream, instantiate, replay on the caller's stream
  e->last_use = now;
  e->seen++;
  if (!plan->s_capture && cudaStreamCreateWithFlags(&plan->s_capture, cudaStreamNonBlocking) != cudaSuccess) {
    cudaGetLastError();
    plan->graph_mode = 0;
    return run_chunk(plan, x1, x2, nv, outs, st);
  }
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  bool ok = cudaStreamBeginCapture(plan->s_capture, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
  if (ok) {
    const int r = run_chunk(plan, x1, x2, nv, outs, plan->s_capture);
    const cudaError_t ce = cudaStreamEndCapture(plan->s_capture, &graph);
    ok = (r == STCD_OK) && ce == cudaSuccess && graph != nullptr;
  }
  if (ok) ok = cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
  if (graph) cudaGraphDestroy(graph);
  if (!ok) {                                  // never again for this plan; plain launches are always correct
    cudaGetLastError();
    if (exec) cudaGraphExecDestroy(exec);
    plan->graph_mode = 0;
    return run_chunk(plan, x1, x2, nv, outs, st);
  }
  e->exec = exec;
  CUDA_TRY(cudaGraphLaunch(exec, st));
  return STCD_OK;
}

static int forward_any(stcd_plan* plan, const void* x1, const void* x2, int u8, int n_pairs, float* const* outs, int n_outs,
                       void* stream) {
  if (!plan || !plan->finalized) return fail(STCD_ERR_STATE, "plan not finalized");
  if (!x1 || !x2 || n_pairs < 0) return fail(STCD_ERR_INVALID, "bad inputs");
  if (plan->in_u8 != u8) return fail(STCD_ERR_INVALID, "plan takes %s inputs", plan->in_u8 ? "uint8 HWC (stcd_forward_u8)" : "fp32 NCHW (stcd_forward)");
  if (n_outs != plan->n_ext || (n_outs > 0 && !outs)) return fail(STCD_ERR_INVALID, "plan has %d external outputs, got %d", plan->n_ext, n_outs);
  DeviceGuard dev_guard(plan->device);   // the caller's current device is restored on return
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t in_bytes = (size_t)plan->in_c * plan->in_h * plan->in_w * (u8 ? 1 : sizeof(float));
  std::vector<float*> o(n_outs);
  for (int start = 0; start < n_pairs; start += plan->chunk) {
    const int nv = std::min(plan->chunk, n_pairs - start);
    for (int k = 0; k < n_outs; ++k) o[k] = outs[k] ? outs[k] + (size_t)start * plan->ext_elems[k] : nullptr;
    int r = run_chunk_graphed(plan, static_cast<const uint8_t*>(x1) + (size_t)start * in_bytes,
                              static_cast<const uint8_t*>(x2) + (size_t)start * in_bytes, nv, o.data(), n_outs, st);
    if (r) return r;
  }
  return STCD_OK;
}

int stcd_forward(stcd_plan* plan, const float* x1, const float* x2, int n_pairs, float* const* outs, int n_outs,
                 void* stream) {
  return forward_any(plan, x1, x2, 0, n_pairs, outs, n_outs, stream);
}

int stcd_forward_u8(stcd_plan* plan, const uint8_t* x1, const uint8_t* x2, int n_pairs, float* const* outs, int n_outs,
                    void* stream) {
  return forward_any(plan, x1, x2, 1, n_pairs, outs, n_outs, stream);
}

int stcd_forward_profile(stcd_plan* plan, const float* x1, const float* x2, int n_pairs, float* const* outs, int n_outs,
                         void* stream, float* op_ms, int n_ops) {
  if (!plan || !plan->finalized) return fail(STCD_ERR_STATE, "plan not finalized");
  if (!x1 || !x2 || n_pairs < 0 || !op_ms) return fail(STCD_ERR_INVALID, "bad inputs");
  if (n_ops != (int)plan->ops.size()) return fail(STCD_ERR_INVALID, "plan has %zu ops, got %d", plan->ops.size(), n_ops);
  if (n_outs != plan->n_ext || (n_outs > 0 && !outs)) return fail(STCD_ERR_INVALID, "plan has %d external outputs, got %d", plan->n_ext, n_outs);
  DeviceGuard dev_guard(plan->device);   // the caller's current device is restored on return
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t in_bytes = (size_t)plan->in_c * plan->in_h * plan->in_w * (plan->in_u8 ? 1 : sizeof(float));
  const uint8_t* b1 = reinterpret_cast<const uint8_t*>(x1);
  const uint8_t* b2 = reinterpret_cast<const uint8_t*>(x2);
  std::vector<cudaEvent_t> ev(n_ops + 1);
  for (auto& e : ev) CUDA_TRY(cudaEventCreate(&e));
  for (int i = 0; i < n_ops; ++i) op_ms[i] = 0.f;
  std::vector<float*> o(n_outs);
  int rc = STCD_OK;
  for (int start = 0; start < n_pairs && rc == STCD_OK; start += plan->chunk) {
    const int nv = std::min(plan->chunk, n_pairs - start);
    for (int k = 0; k < n_outs; ++k) o[k] = outs[k] ? outs[k] + (size_t)start * plan->ext_elems[k] : nullptr;
    rc = run_chunk(plan, b1 + (size_t)start * in_bytes, b2 + (size_t)start * in_bytes, nv, o.data(), st, ev.data());
    if (rc) break;
    if (cudaStreamSynchronize(st) != cudaSuccess) {
      rc = fail(STCD_ERR_CUDA, "stream sync failed: %s", cudaGetErrorString(cudaGetLastError()));
      break;
    }
    for (int i = 0; i < n_ops; ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      op_ms[i] += ms;
    }
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return rc;
}

static int forward_host_any(stcd_plan* plan, const void* x1v, const void* x2v, int u8, int n_pairs, float* const* outs_host,
                            int n_outs) {
  if (!plan || !plan->finalized) return fail(STCD_ERR_STATE, "plan not finalized");
  if (!x1v || !x2v || n_pairs < 0) return fail(STCD_ERR_INVALID, "bad inputs");
  if (plan->in_u8 != u8) return fail(STCD_ERR_INVALID, "plan takes %s inputs", plan->in_u8 ? "uint8 HWC (stcd_forward_host_u8)" : "fp32 NCHW (stcd_forward_host)");
  const uint8_t* x1h = static_cast<const uint8_t*>(x1v);
  const uint8_t* x2h = static_cast<const uint8_t*>(x2v);
  if (n_outs != plan->n_ext || (n_outs > 0 && !outs_host)) return fail(STCD_ERR_INVALID, "plan has %d external outputs, got %d", plan->n_ext, n_outs);
  DeviceGuard dev_guard(plan->device);   // the caller's current device is restored on return
  const size_t in_elems = (size_t)plan->in_c * plan->in_h * plan->in_w * (u8 ? 1 : sizeof(float));   // bytes per image
  const size_t in_bytes = in_elems * plan->chunk;
  if (!plan->s_copy) {
    CUDA_TRY(cudaStreamCreateWithFlags(&plan->s_copy, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&plan->s_comp, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&plan->s_d2h, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
      CUDA_TRY(cudaEventCreateWithFlags(&plan->ev_h2d[b], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&plan->ev_comp[b], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&plan->ev_d2h[b], cudaEventDisableTiming));
      for (int s = 0; s < 2; ++s) CUDA_TRY(cudaMalloc(&plan->stage_in[b][s], in_bytes));
      plan->stage_out[b].assign(plan->n_ext, nullptr);
      for (int k = 0; k < plan->n_ext; ++k)
        CUDA_TRY(cudaMalloc(&plan->stage_out[b][k], plan->ext_elems[k] * plan->chunk * sizeof(float)));
    }
  }
  int it = 0;
  for (int start = 0; start < n_pairs; start += plan->chunk, ++it) {
    const int b = it & 1;
    const int nv = std::min(plan->chunk, n_pairs - start);
    if (it >= 2) CUDA_TRY(cudaStreamWaitEvent(plan->s_copy, plan->ev_comp[b], 0));  // staging buffer consumed
    CUDA_TRY(cudaMemcpyAsync(plan->stage_in[b][0], x1h + (size_t)start * in_elems, in_elems * nv, cudaMemcpyHostToDevice,
                             plan->s_copy));
    CUDA_TRY(cudaMemcpyAsync(plan->stage_in[b][1], x2h + (size_t)start * in_elems, in_elems * nv, cudaMemcpyHostToDevice,
                             plan->s_copy));
    CUDA_TRY(cudaEventRecord(plan->ev_h2d[b], plan->s_copy));
    CUDA_TRY(cudaStreamWaitEvent(plan->s_comp, plan->ev_h2d[b], 0));
    if (it >= 2) CUDA_TRY(cudaStreamWaitEvent(plan->s_comp, plan->ev_d2h[b], 0));  // output staging drained
    int r = run_chunk(plan, plan->stage_in[b][0], plan->stage_in[b][1], nv, plan->stage_out[b].data(), plan->s_comp);
    if (r) return r;
    CUDA_TRY(cudaEventRecord(plan->ev_comp[b], plan->s_comp));
    CUDA_TRY(cudaStreamWaitEvent(plan->s_d2h, plan->ev_comp[b], 0));
    for (int k = 0; k < n_outs; ++k) {
      if (!outs_host[k]) continue;
      CUDA_TRY(cudaMemcpyAsync(outs_host[k] + (size_t)start * plan->ext_elems[k], plan->stage_out[b][k],
                               plan->ext_elems[k] * nv * sizeof(float), cudaMemcpyDeviceToHost, plan->s_d2h));
    }
    CUDA_TRY(cudaEventRecord(plan->ev_d2h[b], plan->s_d2h));
  }
  CUDA_TRY(cudaStreamSynchronize(plan->s_copy));
  CUDA_TRY(cudaStreamSynchronize(plan->s_comp));
  CUDA_TRY(cudaStreamSynchronize(plan->s_d2h));
  return STCD_OK;
}

int stcd_forward_host(stcd_plan* plan, const float* x1h, const float* x2h, int n_pairs, float* const* outs_host, int n_outs) {
  return forward_host_any(plan, x1h, x2h, 0, n_pairs, outs_host, n_outs);
}

int stcd_forward_host_u8(stcd_plan* plan, const uint8_t* x1h, const uint8_t* x2h, int n_pairs, float* const* outs_host,
                         int n_outs) {
  return forward_host_any(plan, x1h, x2h, 1, n_pairs, outs_host, n_outs);
}

int stcd_confusion_add_batch(const void* pred, int pred_kind, float thr, const void* label, int label_kind,
                             int64_t n_img, int64_t pix, int num_class, int64_t* cm_dev, uint8_t* pred_out,
                             void* stream) {
  if (!pred || !label || !cm_dev) return fail(STCD_ERR_INVALID, "NULL pointer");
  if (n_img < 0 || pix < 0) return fail(STCD_ERR_INVALID, "negative size");
  if (num_class < 2 || num_class > 32) return fail(STCD_ERR_INVALID, "num_class %d not in [2, 32]", num_class);
  if (pred_kind < STCD_PRED_ARGMAX2 || pred_kind > STCD_PRED_U8_GE1) return fail(STCD_ERR_INVALID, "pred_kind %d", pred_kind);
  if (pred_kind == STCD_PRED_U8_GE1 && num_class != 2) return fail(STCD_ERR_INVALID, "raw mask predictions need num_class == 2");
  if (label_kind < STCD_LABEL_I64 || label_kind > STCD_LABEL_U8_GE1) return fail(STCD_ERR_INVALID, "label_kind %d", label_kind);
  if (num_class != 2 && pred_kind <= STCD_PRED_RAW_GE) return fail(STCD_ERR_INVALID, "binarising kinds need num_class == 2");
  if (n_img == 0 || pix == 0) return STCD_OK;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(STCD_ERR_NO_DEVICE, "no CUDA device visible: libstcd_b200 has no CPU fallback");
  }
  DeviceGuard dev_guard(device_of(cm_dev));   // launch where the buffers live
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* cm = reinterpret_cast<unsigned long long*>(cm_dev);
  const size_t ne = (size_t)n_img * pix;
  const bool aligned = ((reinterpret_cast<uintptr_t>(pred) | reinterpret_cast<uintptr_t>(label) |
                         reinterpret_cast<uintptr_t>(pred_out)) & 15) == 0;
  const int vec = (aligned && (pix % 4 == 0)) ? 1 : 0;
  const size_t work = vec ? ne / 4 : ne;
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((work + 255) / 256, 148 * 8));

#define STCD_CM2(PK, LK)                                                                                      \
  stcd::confusion2_kernel<PK, LK><<<blocks, 256, 0, st>>>(pred, label, (size_t)n_img, (size_t)pix, thr, vec, cm, pred_out)
#define STCD_CMK(PK, LK) \
  stcd::confusionK_kernel<PK, LK><<<blocks, 256, 0, st>>>(pred, label, (size_t)n_img, (size_t)pix, num_class, cm)
#define STCD_DISPATCH_L(M, PK)                                      \
  switch (label_kind) {                                             \
    case STCD_LABEL_I64: M(PK, STCD_LABEL_I64); break;              \
    case STCD_LABEL_U8: M(PK, STCD_LABEL_U8); break;                \
    case STCD_LABEL_U8_GE1: M(PK, STCD_LABEL_U8_GE1); break;        \
    default: M(PK, STCD_LABEL_I32); break;                          \
  }
  if (num_class == 2) {
    switch (pred_kind) {
      case STCD_PRED_ARGMAX2: STCD_DISPATCH_L(STCD_CM2, STCD_PRED_ARGMAX2); break;
      case STCD_PRED_SIGMOID_GT: STCD_DISPATCH_L(STCD_CM2, STCD_PRED_SIGMOID_GT); break;
      case STCD_PRED_RAW_GE: STCD_DISPATCH_L(STCD_CM2, STCD_PRED_RAW_GE); break;
      case STCD_PRED_U8: STCD_DISPATCH_L(STCD_CM2, STCD_PRED_U8); break;
      case STCD_PRED_I32: STCD_DISPATCH_L(STCD_CM2, STCD_PRED_I32); break;
      case STCD_PRED_U8_GE1: STCD_DISPATCH_L(STCD_CM2, STCD_PRED_U8_GE1); break;
      default: STCD_DISPATCH_L(STCD_CM2, STCD_PRED_I64); break;
    }
  } else {
    switch (pred_kind) {
      case STCD_PRED_U8: STCD_DISPATCH_L(STCD_CMK, STCD_PRED_U8); break;
      case STCD_PRED_I32: STCD_DISPATCH_L(STCD_CMK, STCD_PRED_I32); break;
      default: STCD_DISPATCH_L(STCD_CMK, STCD_PRED_I64); break;
    }
  }
  CUDA_TRY(cudaGetLastError());
  return STCD_OK;
}

int stcd_binarise_mask(const float* logits, int pred_kind, float thr, int64_t n_img, int64_t pix, int on_value, uint8_t* mask,
                       void* stream) {
  if (!logits || !mask) return fail(STCD_ERR_INVALID, "NULL pointer");
  if (pred_kind < STCD_PRED_ARGMAX2 || pred_kind > STCD_PRED_RAW_GE) return fail(STCD_ERR_INVALID, "pred_kind %d does not binarise logits", pred_kind);
  if (n_img < 0 || pix < 0 || on_value < 1 || on_value > 255) return fail(STCD_ERR_INVALID, "bad sizes / on_value");
  if (n_img == 0 || pix == 0) return STCD_OK;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(STCD_ERR_NO_DEVICE, "no CUDA device visible: libstcd_b200 has no CPU fallback");
  }
  DeviceGuard dev_guard(device_of(mask));   // launch where the buffers live
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t ne = (size_t)n_img * pix;
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((ne + 255) / 256, 148 * 16));
  switch (pred_kind) {
    case STCD_PRED_ARGMAX2: stcd::binarise_mask_kernel<STCD_PRED_ARGMAX2><<<blocks, 256, 0, st>>>(logits, n_img, pix, thr, on_value, mask); break;
    case STCD_PRED_SIGMOID_GT: stcd::binarise_mask_kernel<STCD_PRED_SIGMOID_GT><<<blocks, 256, 0, st>>>(logits, n_img, pix, thr, on_value, mask); break;
    default: stcd::binarise_mask_kernel<STCD_PRED_RAW_GE><<<blocks, 256, 0, st>>>(logits, n_img, pix, thr, on_value, mask); break;
  }
  CUDA_TRY(cudaGetLastError());
  return STCD_OK;
}

int stcd_knn_graph(const float* x, const float* y, const float* relpos, int B, int C, int N, int M, int k, int dilation,
                   int64_t* nn_idx, float* scratch, void* stream) {
  if (!x || !nn_idx || !scratch) return fail(STCD_ERR_INVALID, "NULL pointer");
  if (B < 0 || C < 1 || N < 1 || M < 1 || k < 1 || dilation < 1) return fail(STCD_ERR_INVALID, "bad sizes B=%d C=%d N=%d M=%d k=%d d=%d", B, C, N, M, k, dilation);
  if (!y && M != N) return fail(STCD_ERR_INVALID, "y is NULL (y := x) but M=%d != N=%d", M, N);
  if (M > stcd::kKnnM) return fail(STCD_ERR_INVALID, "M=%d > %d keys (ViG stages have at most 256 after the reduce-ratio pooling)", M, stcd::kKnnM);
  if (k * dilation > M) return fail(STCD_ERR_INVALID, "k*dilation=%d > M=%d", k * dilation, M);
  if (B == 0) return STCD_OK;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(STCD_ERR_NO_DEVICE, "no CUDA device visible: libstcd_b200 has no CPU fallback");
  }
  DeviceGuard dev_guard(device_of(nn_idx));   // launch where the buffers live
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (env_int("STCD_KNN_MMA", 1) != 0 && k * dilation <= 27) {
    // tensor-core path: the plane workspace (6 bytes per value, more than `scratch` holds) is taken from and returned to the
    // stream-ordered pool around the two kernels
    const size_t xb = knn_planes_bytes(B, C, N), xs = knn_sq_bytes(B, N), yb = y ? knn_planes_bytes(B, C, M) : 0, ys = y ? knn_sq_bytes(B, M) : 0;
    uint8_t* ws = nullptr;
    CUDA_TRY(cudaMallocAsync(&ws, xb + xs + yb + ys, st));
    CUDA_TRY(cudaMemsetAsync(ws, 0, xb + xs + yb + ys, st));
    int r = launch_knn_pipe(x, y, relpos, B, C, N, M, k, dilation, reinterpret_cast<__nv_bfloat16*>(ws), reinterpret_cast<float*>(ws + xb),
                            y ? reinterpret_cast<__nv_bfloat16*>(ws + xb + xs) : nullptr, y ? reinterpret_cast<float*>(ws + xb + xs + yb) : nullptr,
                            reinterpret_cast<long long*>(nn_idx), st);
    cudaFreeAsync(ws, st);
    return r;
  }
  float* xn = scratch;
  float* yn = y ? scratch + (size_t)B * C * N : scratch;
  auto ng = [](int B_, int n_) { return (unsigned)std::max(1, std::min(B_ * ((n_ + 31) / 32), 148 * 16)); };
  stcd::normalize_nodes_kernel<<<ng(B, N), 256, 0, st>>>(x, xn, B, C, N);
  if (y) stcd::normalize_nodes_kernel<<<ng(B, M), 256, 0, st>>>(y, yn, B, C, M);
  return launch_knn(xn, yn, relpos, B, C, N, M, k, dilation, reinterpret_cast<long long*>(nn_idx), st);
}

int stcd_max_relative(const float* x, const float* y, const int64_t* nn_idx, int B, int C, int N, int M, int k, int interleave,
                      float* out, void* stream) {
  if (!x || !nn_idx || !out) return fail(STCD_ERR_INVALID, "NULL pointer");
  if (B < 0 || C < 1 || N < 1 || M < 1 || k < 1) return fail(STCD_ERR_INVALID, "bad sizes");
  if (!y && M != N) return fail(STCD_ERR_INVALID, "y is NULL (y := x) but M=%d != N=%d", M, N);
  if (B == 0) return STCD_OK;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(STCD_ERR_NO_DEVICE, "no CUDA device visible: libstcd_b200 has no CPU fallback");
  }
  DeviceGuard dev_guard(device_of(out));   // launch where the buffers live
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t total = (size_t)B * C * N;
  stcd::max_relative_kernel<<<(unsigned)std::min<size_t>((total + 255) / 256, 148 * 16), 256, 0, st>>>(
      x, y ? y : x, reinterpret_cast<const long long*>(nn_idx), B, C, N, M, k, interleave, out);
  CUDA_TRY(cudaGetLastError());
  return STCD_OK;
}

}  // extern "C"
