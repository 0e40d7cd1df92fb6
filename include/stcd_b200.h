/*
 * stcd_b200.h — C-ABI of libstcd_b200.so: B200 (sm_100a) bi-temporal change-detection
 * inference + confusion-matrix evaluation.
 *
 * The reference (VCISwang/STCD) has no FFI of its own; the boundary it exposes is Python:
 *   net_G(x1, x2)                       models/SiamUnet_diff.py:94, models/SNUNet.py:116,
 *                                       segmentation_models_pytorch/decoders/unet/model.py:316
 *   define_G(args, ...)                 models/networks.py:138-215
 *   SegmentationMetric.addBatch(p, l)   train_stcd.py:572-588
 * Each entry point below names the reference call it stands in for.  Plain pointers and sizes
 * only — no torch types.  All `const void*` / `void*` data pointers are DEVICE pointers unless a
 * function says "host"; `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *
 * Error convention: every int-returning function returns STCD_OK (0) or a negative/positive
 * error code; stcd_last_error() gives a thread-local message (reference: Python exceptions,
 * models/networks.py:214 NotImplementedError, train_stcd.py:587 assert).
 *
 * Threading: a plan is not re-entrant (one forward in flight per plan); distinct plans are
 * independent.  All work is enqueued on the caller's stream.
 */
#ifndef STCD_B200_H_
#define STCD_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STCD_ABI_VERSION 21

enum stcd_status {
  STCD_OK = 0,
  STCD_ERR_INVALID = 1,   /* bad argument / shape (reference: assert / ValueError) */
  STCD_ERR_CUDA = 2,      /* a CUDA runtime / driver call failed */
  STCD_ERR_NO_DEVICE = 3, /* no sm_100 device visible: the product path has NO CPU fallback */
  STCD_ERR_STATE = 4      /* plan used before finalize / after destroy */
};

enum stcd_dtype { STCD_BF16 = 0, STCD_F32 = 1 };

typedef struct stcd_plan stcd_plan;

/* ------------------------------------------------------------------------------------------ */
/* library                                                                                    */
const char* stcd_last_error(void);
int stcd_abi_version(void);
/* number of visible CUDA devices with compute capability 10.x; 0 on a CPU-only host */
int stcd_device_count(void);

/* ------------------------------------------------------------------------------------------ */
/* plan construction: the host side (Python mirror of the reference modules) lowers a         */
/* reference nn.Module (its state_dict) into a list of fused ops on NHWC bf16 tensors.         */
/* The batch is processed in chunks of `chunk_pairs` image pairs so that inter-layer           */
/* activations stay resident in the 126 MB L2.                                                 */

/* device = -1 creates a VALIDATION plan: every stcd_plan_add_* call checks and records its descriptor exactly as on a
 * device, stcd_plan_finalize returns STCD_ERR_NO_DEVICE (host-side tests of the lowering run without a GPU).
 *
 * precision: STCD_PRECISION_BF16 or STCD_PRECISION_SPLIT, for every op of the plan.  Split precision is the tolerance class
 * the north star calls "tf32": logits within 1e-3 of the fp32 reference; the reference itself computes in fp32,
 * models/SNUNet.py:116-152.  In a split plan every tensor stores 2x its logical channels, a multiple of 16
 * (stcd_plan_add_tensor refuses any other count): a hi plane bf16(v) in channel groups [0, c8/2) and a lo plane
 * bf16(v - hi) in [c8/2, c8).  A conv's K-program (built by the host) reads each logical source as the three segments
 * (hi, lo, hi) against the weights (Whi, Whi, Wlo); its epilogue writes both planes of out0 / out_raw / out_pool / out_diff
 * and reads the residual as hi + lo.  A space-to-depth out0 stores 8*cout channels: hi of parity class k at k*cout, lo at
 * 4*cout + k*cout; fold_cs and xf_cs are refused.  The other ops read hi + lo, compute in fp32 and write hi = bf16(v),
 * lo = bf16(v - hi); their comments give the layouts as "split plan:" lines.  Graph conv, channel attention, spatial gate,
 * global-local gate, CSAM gate, VFFM, seg head and the uint8 input pack have no split form and are refused. */
enum stcd_precision { STCD_PRECISION_BF16 = 0, STCD_PRECISION_SPLIT = 1 };
int stcd_plan_create(int device, int chunk_pairs, int precision, stcd_plan** out);
void stcd_plan_destroy(stcd_plan* plan);

/* Declare an activation tensor of img_mult*chunk_pairs images, bf16 [img][c/8][h][w][8].
 * split plan: c is a multiple of 16 (two planes of 8-channel groups).  Returns id >= 0, or <0. */
int stcd_plan_add_tensor(stcd_plan* plan, int img_mult, int h, int w, int c, int dtype);

/* Activation tensors are stored channel-chunked: bf16 [img][c/8][h][w][8] ("NC8HW8"), so that a
 * TMA box {8 ch, box_w px, box_h px, kc/8 chunks} lands in shared memory as the un-swizzled
 * K-major core-matrix layout tcgen05.mma consumes, and a filter tap is just a byte offset into
 * the box: a 3x3 conv reads its (16+2)x(8+2) halo ONCE per K-chunk instead of once per tap.
 *
 * One A-stage load of the implicit GEMM: channels [c0, c0+kc) of source `src` (index into
 * stcd_conv_desc.src) over the pixel box whose origin is (ty*src_sy + by, tx*src_sx + bx) of image
 * (n + n_off) for the tile at tile-pixel (ty, tx).  Out-of-bounds pixels read as 0 (= zero
 * padding, nn.Conv2d padding=1: SiamUnet_diff.py:18).  The chunk feeds `n_taps` filter taps
 * (stcd_tap entries [tap_begin, tap_begin + n_taps)). */
typedef struct stcd_chunk {
  int16_t src, c0;
  int16_t by, bx;
  int32_t n_off;
  int16_t tap_begin, n_taps;
} stcd_chunk;

/* One filter tap inside a chunk's box: tile pixel (i, j) reads box pixel (i + ty, j + tx).
 * Weight blocks are consumed in tap order: tap t of a phase multiplies weight block t. */
typedef struct stcd_tap {
  int16_t ty, tx;
} stcd_tap;

/* One output phase: tile pixel (i, j) -> output pixel (i*osy + oy, j*osx + ox). A stride-1
 * conv has one phase; ConvTranspose2d(stride=2) (SiamUnet_diff.py:52) has four. */
typedef struct stcd_phase {
  int32_t chunk_begin, chunk_count; /* slice of the chunk array */
  int32_t oy, ox;
  int32_t w_block;                  /* first weight block of this phase (per N tile) */
  int32_t n_blocks;                 /* = number of taps summed over the phase's chunks */
} stcd_phase;

#define STCD_MAX_SRC 6
#define STCD_MAX_PHASE 4
#define STCD_TILE_H 16
#define STCD_TILE_W 8

typedef struct stcd_conv_desc {
  /* A operand (activations): virtual concat of up to 6 sources (torch.cat, SNUNet.py:142) */
  int32_t n_src;
  int32_t src[STCD_MAX_SRC];      /* tensor ids */
  int32_t src_sy[STCD_MAX_SRC];   /* per-source input coordinate stride (2 for a stride-2 conv) */
  int32_t src_sx[STCD_MAX_SRC];
  int32_t src_ey[STCD_MAX_SRC];   /* per-source halo: box = (16 + ey) x (8 + ex) pixels (0 if stride > 1) */
  int32_t src_ex[STCD_MAX_SRC];
  /* tile grid */
  int32_t hg, wg;                 /* tile-pixel grid (= output dims / osy, osx) */
  int32_t img_mult;               /* images in the grid = img_mult * chunk_pairs */
  int32_t pair;                   /* 1: each CTA also accumulates image n + chunk_pairs (Siamese pair) */
  /* B operand (weights), packed by the host in consumption order:
   * bf16 [n_tiles][total blocks][kc/8][n_tile][8]  (block = one tap of one chunk) */
  const uint16_t* weights;        /* HOST pointer, copied at add time */
  int64_t w_elems;
  int32_t kc;                     /* channels per chunk: a multiple of 16 in [16, 128] (64 / 32 / 16, or e.g. 80 for 80-, 160-, 400-channel maps) */
  int32_t n_tile;                 /* GEMM N per CTA (multiple of 16, <= 256) */
  int32_t cout;                   /* real output channels */
  int32_t cout_pad;               /* padded to a multiple of n_tile */
  int32_t n_phase;
  stcd_phase phase[STCD_MAX_PHASE];
  const stcd_chunk* chunks;       /* HOST pointer */
  int32_t n_chunks;
  const stcd_tap* taps;           /* HOST pointer */
  int32_t n_taps;
  int32_t osy, osx;               /* output coordinate stride */
  /* epilogue: v = acc*scale + shift; [out_raw <- v]; [v = v*scale2 + shift2]; [v += res];
   * [v = relu(v)]; out0 <- v; out_pool <- maxpool2x2(v); out_diff <- |v(n) - v(n+chunk)| */
  const float* scale;             /* HOST, [cout_pad] */
  const float* shift;             /* HOST, [cout_pad] */
  const float* scale2;            /* HOST or NULL */
  const float* shift2;            /* HOST or NULL */
  int32_t relu;                   /* activation: 0 none, 1 ReLU, 2 GELU (erf form, nn.GELU()), 3 PReLU with one slope act_alpha */
  int32_t res;                    /* tensor id or -1 */
  int32_t out0, out0_coff;        /* tensor id or -1; channel offset inside out0 */
  int32_t out_raw;                /* tensor id or -1 */
  int32_t out_pool;               /* tensor id or -1 */
  int32_t out_diff;               /* tensor id or -1 (needs pair=1) */
  int32_t out_ext;                /* index into stcd_forward's outs[] for fp32 NCHW logits, or -1 */
  /* 1: out0 is stored space-to-depth, a [ho/2][wo/2] tensor of 4*cout channels: output pixel (y, x),
   * channel c -> pixel (y/2, x/2), channel ((y%2)*2 + x%2)*cout + c.  Feature maps read only by
   * stride-2 convs (torchvision BasicBlock conv1/downsample, models/resnet.py:59-60) and by the Unet
   * decoder's skip path (decoders/unet/decoder.py:36-40) are stored this way so that every consumer is
   * a stride-1 halo load over one parity class. */
  int32_t out0_s2d;
  /* Phase folding for up-sampling ops (ConvTranspose2d stride 2: SNUNet.py:38, SiamUnet_diff.py:52; nearest x2 +
   * conv: decoders/unet/decoder.py:36-40): fold_cs > 0 folds the osy*osx output phases into GEMM N.  The op then
   * has ONE phase entry, cout = osy*osx*fold_cs columns, and column p*fold_cs + c (c < fold_cout) is channel c of
   * output pixel (i*osy + p/osx, j*osx + p%osx): the A operand is fetched once for all phases and N grows from
   * cout to 4*cout, which is what Cout <= 32 layers need (an SS-mode MMA costs the same for any N <= 64).
   * Only the affine + ReLU + out0 epilogue is available in this mode.  fold_cs % 16 == 0.
   * Alternatively the op has osy phase entries (oy = 0 .. osy-1, ox = 0) of cout = osx*fold_cs columns each: only the
   * horizontal phases are folded (column block p -> output pixel (i*osy + oy, j*osx + p)). */
  int32_t fold_cs, fold_cout;
  /* act_pre = 1: the activation is applied BEFORE the second affine (conv -> PReLU/ReLU -> BatchNorm, the order of
   * ChangeFormer.py:1138-1157 conv_diff / make_prediction) instead of at the end of the epilogue; needs scale2/shift2. */
  int32_t act_pre;
  float act_alpha;
  /* Horizontal tap folding of a stride-1 3x3 conv with few output channels (nn.Conv2d(k=3, padding=1): SNUNet.py:17-26,
   * SiamUnet_diff.py:18-48; ConvTranspose2d(k=3, s=1, p=1) decoder "convs": SiamUnet_diff.py:54-90).  xf_cs > 0: the K-program
   * holds ONE tap per filter row (dy = -1, 0, +1; dx = 0; no horizontal halo) whose weight block stacks the row's three
   * filter columns, n_tile = cout_pad = 3*xf_cs (xf_cs = cout rounded up to 16): column b*xf_cs + c of the accumulator at
   * input position x is tap (dy, b - 1)'s contribution to channel c of output x - (b - 1); the epilogue sums the three
   * blocks across neighbouring pixels.  Tiles are 8 x 16 input positions with 14 output columns (the library's choice;
   * hg / wg stay the output dims).  Single phase, stride-1 sources, osy = osx = 1, no space-to-depth / folded store. */
  int32_t xf_cs;
} stcd_conv_desc;

/* returns op index >= 0, or <0 */
int stcd_plan_add_conv(stcd_plan* plan, const stcd_conv_desc* desc);

/* x1, x2 (fp32 NCHW [n_pairs, cin, h, w], the reference's input layout: data/dataset.py:196-203)
 * -> bf16 [2*chunk][2][h][w][8] (cin <= 8 real channels, 16 stored) with the T1 images first, then
 * the T2 images.
 * split plan: dst has 16 stored channels, [0, 8) = bf16(x), [8, 16) = bf16(x - bf16(x)); cin <= 8. */
int stcd_plan_add_input_pack(stcd_plan* plan, int dst_tensor, int cin);

/* Space-to-depth variant for the 7x7 stride-2 ResNet stem (smp/encoders/resnet.py:50): x1, x2 fp32 NCHW
 * [n_pairs, cin, 2h, 2w] -> bf16 [2*chunk][2][h][w][8] with channel (py*2 + px)*cin + c holding
 * x[c][2y + py][2x + px] (4*cin <= 16); the stem then runs as a 4x4 stride-1 conv.
 * split plan: dst stores 32 channels, the hi plane in [0, 16) (channel (py*2 + px)*cin + c), the lo plane in [16, 32). */
int stcd_plan_add_input_pack_s2d(stcd_plan* plan, int dst_tensor, int cin);

/* uint8 input pipeline (SURVEY.md §8(f)-1; reference: data/dataset.py:196-203, ToTensor + Normalize on the host).
 * Same as stcd_plan_add_input_pack / _s2d, but the plan's inputs become uint8 HWC images [n_pairs, H, W, cin] and
 * the pack kernel evaluates ((u / 255) - mean[c]) / std[c] in fp32 (IEEE ops, the reference's expression) before
 * the bf16 rounding: bit-identical to packing the host-normalised fp32 tensor, at a quarter of the PCIe bytes.
 * A plan built with this op is run with stcd_forward_u8 / stcd_forward_host_u8.  mean, std: HOST float[cin].
 * Refused in a split plan. */
int stcd_plan_add_input_pack_u8(stcd_plan* plan, int dst_tensor, int cin, int s2d, const float* mean, const float* std_);

/* nn.MaxPool2d(kernel_size=3, stride=2, padding=1) (smp/encoders/resnet.py:51) over a feature map stored
 * space-to-depth (src: [h][w] pixels x 4c channels = the (2h x 2w) map) -> dst [h][w] x c channels.
 * split plan: src stores 8c channels (hi of parity class k at k*c, lo at 4c + k*c), dst 2c; the max over hi + lo selects the
 *   winning (hi, lo) pair (first maximum in the kernel's window order). */
int stcd_plan_add_maxpool_s2d(stcd_plan* plan, int src_tensor, int dst_tensor, int c);

/* dst = |src[T1 images] - src[T2 images]| (torch.abs(f1 - f2), FFCTLCD.forward, decoders/unet/model.py:412): src holds
 * both temporal streams (mult 2), dst one stream with the same [h][w][c] (any layout: elementwise).
 * split plan (subdiff too): every tensor stores hi and lo planes. */
int stcd_plan_add_absdiff(stcd_plan* plan, int src_tensor, int dst_tensor);
/* the signed variant dst = (add) + src[T1] - src[T2] (DTCDSCN: decoder(...) + e_x - e_y, models/DTCDSCN.py:294-300);
 * add_or_neg: a one-stream tensor of dst's shape, or -1 */
int stcd_plan_add_subdiff(stcd_plan* plan, int src_tensor, int add_or_neg, int dst_tensor);

/* Squeeze-and-excitation gates of DTCDSCN on plan tensors (models/DTCDSCN.py): g = sigmoid(w2 relu(w1 mean_hw(src))),
 * w1 HOST fp32 [hid][c], w2 HOST fp32 [c][hid] (bias-free: SELayer :14-19, SCSEBlock.channel_excitation :153-158).
 *   mode 0 (SEBasicBlock tail, :93-109):  dst = relu(src * g + res)        res_or_neg: tensor id or -1
 *   mode 1 (DecoderBlock, :129-135):       dst = src * (1 + g + sigmoid(ws . src_pixel))   ws HOST fp32 [c] (spatial_se :160-162)
 * dst_s2d_or_neg >= 0 also writes the space-to-depth copy.  c <= 512, hid <= 32.
 * split plan: src, res, dst store 2c channels; the space-to-depth copy 8c (hi of parity class k at k*c, lo at 4c + k*c). */
int stcd_plan_add_channel_gate(stcd_plan* plan, int src_tensor, int res_or_neg, int dst_tensor, int dst_s2d_or_neg, int c, int hid,
                               const float* w1, const float* w2, const float* ws_or_null, int mode);

/* BIT's token path on a 32-channel plan tensor holding both streams (models/networks.py:359-394,414-428; blocks in
 * models/help_funcs.py): semantic tokens -> + learned positions -> transformer encoder over the pair's 2L tokens -> transformer
 * decoder (every pixel queries its image's L tokens).  c = 32, token_len = 4, heads = 8, mlp = 64 (the registered BIT keys).
 * enc / dec: HOST fp32, one packed row per layer:
 *   enc row: ln1_g[c] ln1_b[c] Wqkv[3*inner_enc][c] Wout[c][inner_enc] bout[c] ln2_g[c] ln2_b[c] W1[mlp][c] b1[mlp] W2[c][mlp] b2[c]
 *   dec row: ln1_g[c] ln1_b[c] Wq[inner_dec][c] Wk[..][c] Wv[..][c] Wout^T[inner_dec][c] bout[c] ln2_g[c] ln2_b[c]
 *            W1^T[c][mlp] b1[mlp] W2^T[mlp][c] b2[c]
 * (torch Linear layouts [out][in]; the decoder's to_out and feed-forward weights transposed).
 * split plan: src and dst store 64 channels (2 x 32); the token path itself is fp32 in both precisions. */
typedef struct {
  int32_t c, token_len, heads, mlp;
  int32_t n_enc, n_dec, inner_enc, inner_dec;
  int32_t softmax;                 /* Cross_Attention(softmax=...) of the decoder, help_funcs.py:101-104 */
  const float* conv_a;             /* [token_len][c]      conv_a.weight, networks.py:324 */
  const float* pos;                /* [2*token_len][c]    pos_embedding, :337 */
  const float* enc;
  const float* dec;
} stcd_bit_desc;
int stcd_plan_add_bit_transformer(stcd_plan* plan, int src_tensor, int dst_tensor, const stcd_bit_desc* desc);

/* DSIFN's channel attention over a virtual concat (models/DSIFN.py:24-36 and `x = self.caK(x) * x`, :140,154,166,178):
 * dst[1*chunk, h, w, sum(src_c)] = cat(srcs) * sigmoid(fc2(relu(fc1(avgpool))) + fc2(relu(fc1(maxpool)))).
 * src i = stream src_streams[i] (0 / 1) of plan tensor src_tensors[i], its first src_c[i] channels (multiples of 8); n_src <= 4.
 * fc1 HOST fp32 [hid][C], fc2 HOST fp32 [C][hid] (bias-free 1x1 convs); C <= 2048, hid <= 256. */
int stcd_plan_add_channel_attention(stcd_plan* plan, const int* src_tensors, const int* src_streams, const int* src_c, int n_src,
                                    int dst_tensor, int hid, const float* fc1, const float* fc2);

/* DSIFN's spatial attention followed by its BatchNorm (models/DSIFN.py:39-51 and `x = bn_saK(saK(x) * x)`, :131-132 ...):
 * dst = (src * sigmoid(conv7x7([mean_c src, max_c src]))) * scale + shift.  w HOST fp32 [2][7][7], scale / shift HOST fp32 [c]. */
int stcd_plan_add_spatial_gate(stcd_plan* plan, int src_tensor, int dst_tensor, int c, const float* w, const float* scale,
                               const float* shift);

/* ChangeGNNV2's Global_Local, global branch (models/ChangeVIG.py:377-385): dst = sigmoid(ch[c] * sp[pixel]) * src,
 * ch = relu(BN(grouped (2,1) conv over [avgpool; maxpool])), sp = relu(conv5x5([mean_c, max_c]) + b).
 * prm HOST fp32: w_avg[c] | w_max[c] | scale[c] | shift[c] (conv bias and BatchNorm folded) | w_sp[2][5][5] | b_sp.  c <= 512. */
int stcd_plan_add_global_local_gate(stcd_plan* plan, int src_tensor, int dst_tensor, int c, const float* prm);

/* VIG_V20_2's csam_V20 (models/ChangeVIG.py:956-994): dst = bt((sigmoid(ch[c]) + sigmoid(sp[pixel])) * src),
 * ch = liner2(relu(liner1(gelu(BN(grouped (2,1) conv over [avgpool; maxpool]))))), sp = conv3x3(relu(conv3x3([mean_c, max_c]))).
 * prm HOST fp32: w_avg[c] | w_max[c] | scale[c] | shift[c] | liner1[hid][c] | liner2^T[hid][c] | liner2 bias[c] | bt scale[c] |
 * bt shift[c] | conv2_1[2][3][3] | conv2_2[3][3].  c <= 512, hid <= 128. */
int stcd_plan_add_csam_gate(stcd_plan* plan, int src_tensor, int dst_tensor, int c, int hid, const float* prm);

/* ChangeGNNV2's VFFM (models/ChangeVIG.py:452-460): dst = 2 low wei + 2 high (1 - wei),
 * wei = sigmoid(MLP_avg(avgpool(mixed)) + MLP_max(maxpool(mixed)) + local), mixed = low + high (a plan tensor), local = the
 * local_att branch (a plan tensor).  All tensors [chunk, h, w, c] with exactly c channels.  prm HOST fp32: avg branch then max
 * branch, each  W1[inter][c] | s1[inter] | t1[inter] | W2^T[inter][c] | s2[c] | t2[c]  (conv biases and BatchNorms folded).
 * c <= 512, inter <= 128. */
int stcd_plan_add_vffm(stcd_plan* plan, int low_tensor, int high_tensor, int mixed_tensor, int local_tensor, int dst_tensor, int c,
                       int inter, const float* prm);

/* dst = sum of n <= 5 plan tensors of identical shape (Dblock.forward: x + d1 + d2 + d3 + d4, models/DTCDSCN.py:65-71).
 * split plan: every tensor stores hi and lo planes. */
int stcd_plan_add_sum(stcd_plan* plan, const int* src_tensors, int n, int dst_tensor);

/* SegCD's tail (segmentation_models_pytorch/decoders/unet/model.py:321-330) as one op over the decoder
 * output `src` (bf16, both temporal streams: mult = 2, c channels): with head = Conv2d(c, 1, 3, padding=1)
 * (base/heads.py:5-10), m1 = head(d1), m2 = head(d2), change = min(head(|d1 - d2|), |m1 - m2|).
 * weight: HOST fp32 [9][c] (tap-major ky*3 + kx), copied at add time.  External outputs out_ext,
 * out_ext + 1, out_ext + 2 = m1, m2, change (fp32 NCHW [n, 1, h, w]).  c in {8, 16, 24, 32}. */
typedef struct stcd_seghead_desc {
  int32_t src;
  int32_t c;
  const float* weight;
  float bias;
  int32_t out_ext;
  /* FFCTLCD (decoders/unet/model.py:407-423): >= 0 names a single-stream tensor [chunk][c/8][h][w][8] holding
   * decoder(|f1 - f2|); the feature-level branch is then head(that) instead of head(|d1 - d2|).  -1: SegCD. */
  int32_t diff_src;
} stcd_seghead_desc;
int stcd_plan_add_seg_head(stcd_plan* plan, const stcd_seghead_desc* desc);

/* The graph half of a ViG Grapher block on a plan tensor (gcn_lib DyGraphConv2d up to MRConv2d's aggregation; see
 * stcd_knn_graph / stcd_max_relative below for the semantics): y = avg_pool2d(x, r) if r > 1 else x, dense dilated kNN
 * graph of x over y with the relative-position bias, dst = bf16(max_k (y_j - x_i)).  src, dst: bf16 [imgs][c/8][h][w][8]
 * with the same image multiplicity; relative_pos: HOST fp32 [h*w][h*w/r^2] or NULL, copied at add time. */
int stcd_plan_add_graph_conv(stcd_plan* plan, int src_tensor, int dst_tensor, int c, int k, int dilation, int r,
                             const float* relative_pos);

/* F.interpolate(x, scale_factor=scale, mode="bilinear", align_corners=False) between two plan tensors
 * (ChangeVIG.py:246-262); dst is [scale*h][scale*w], first c channels.
 * split plan: src and dst store 2c channels. */
int stcd_plan_add_bilinear_up(stcd_plan* plan, int src_tensor, int dst_tensor, int c, int scale);

/* MiT / ChangeFormer encoder ops between plan tensors (models/ChangeFormer.py).
 * layernorm: nn.LayerNorm(c, eps) over the channels of every pixel / token (:226,475,480); dst_s2d_or_neg >= 0 also
 *   writes the space-to-depth copy ([h/2][w/2], 4c channels) a following stride-2 patch-embedding conv reads.
 *   gamma, beta: HOST fp32 [c].
 * sr_attention: softmax(q k^T * scale) v per head (:338-358); q, dst [imgs][h][w][c], kv [imgs][hk][wk][2c] with
 *   k = channels [0, c), v = [c, 2c); hk*wk <= 64 keys, c / heads in {64, 80}.
 * dwconv3x3: depth-wise 3x3 (padding 1) + bias, then GELU if gelu != 0 (:283-289,512-523); weight HOST fp32 [c][9].
 * split plan:
 *   layernorm: src and dst store 2c channels; the space-to-depth copy stores 8c: hi of parity class k, channel ch at k*c + ch,
 *     lo at 4c + k*c + ch.
 *   sr_attention: q and dst store 2c, kv 4c (k hi [0, c), v hi [c, 2c), k lo [2c, 3c), v lo [3c, 4c)); exactly 64 keys.
 *     S = Qhi Khi^T + Qlo Khi^T + Qhi Klo^T, fp32 softmax, P split into hi + lo, O = Phi Vhi + Plo Vhi + Phi Vlo, normalised
 *     by the fp32 row sum.
 *   dwconv3x3: src and dst store 2c channels. */
int stcd_plan_add_layernorm(stcd_plan* plan, int src_tensor, int dst_tensor, int dst_s2d_or_neg, int c, const float* gamma,
                            const float* beta, float eps);
int stcd_plan_add_sr_attention(stcd_plan* plan, int q_tensor, int kv_tensor, int dst_tensor, int c, int heads, float scale);
int stcd_plan_add_dwconv3x3(stcd_plan* plan, int src_tensor, int dst_tensor, int c, const float* weight, const float* bias,
                            int gelu);

/* SNUNet's ECAM tail (models/SNUNet.py:144-149: two ChannelAttention blocks :46-59 + conv_final)
 * over four activation tensors of `c` channels each, as one fused op writing external output
 * `out_ext` (fp32 NCHW [n, n_class, h, w]).  All weight pointers are HOST fp32, copied at add time:
 * ca_fc1 [r][4c], ca_fc2 [4c][r], ca1_fc1 [r1][c], ca1_fc2 [c][r1], w_final [n_class][4c],
 * b_final [n_class].  Limits: c % 8 == 0, c <= 64, r, r1 <= 16, n_class <= 4.
 * split plan: each source stores 2c channels (hi plane, lo plane) and is read as hi + lo. */
typedef struct stcd_ecam_desc {
  int32_t src[4];
  int32_t c, n_class, r, r1;
  const float* ca_fc1;
  const float* ca_fc2;
  const float* ca1_fc1;
  const float* ca1_fc2;
  const float* w_final;
  const float* b_final;
  int32_t out_ext;
} stcd_ecam_desc;
int stcd_plan_add_ecam_head(stcd_plan* plan, const stcd_ecam_desc* desc);

/* allocate the workspace, upload weights, encode TMA descriptors */
int stcd_plan_finalize(stcd_plan* plan);

/* Diagnostics / layer-wise parity tests: synchronous copy between a HOST buffer and activation
 * tensor `tensor_id` (bf16 [img_mult*chunk][c/8][h][w][8]); to_device != 0 writes the tensor.
 * `bytes` must equal the tensor's size. */
int stcd_plan_tensor_copy(stcd_plan* plan, int tensor_id, void* host, int64_t bytes, int to_device);

/* Diagnostics: launch geometry of conv op `op_index` (info[0..9] = grid.x, grid.y, dynamic smem,
 * A stages, W stages, W resident, TMEM columns, tiles, A stage bytes, W block bytes) and, when the
 * plan was finalized with STCD_TRACE=1 in the environment, 16 clock stamps per CTA of its last
 * launch.  Returns the number of int64 words written to `host`, or -1. */
int64_t stcd_plan_read_trace(stcd_plan* plan, int op_index, int64_t* host, int64_t max_words, int32_t* info);

/* bytes of device memory the plan owns (workspace + weights) */
int64_t stcd_plan_workspace_bytes(const stcd_plan* plan);
/* number of kernels one stcd_forward of n_pairs launches (for bench.py's gpu_launches) */
int64_t stcd_plan_launches(const stcd_plan* plan, int n_pairs);

/* ------------------------------------------------------------------------------------------ */
/* reference-facing entry points                                                               */

/* Replaces net_G(x1, x2) (SiamUnet_diff.py:94-181 etc.).  x1, x2: device fp32 NCHW
 * [n_pairs, cin, H, W]; outs[k]: device fp32 NCHW buffers for the plan's external outputs
 * (outs[n_outs-1] = full-resolution logits, like the reference's list-valued forwards). */
int stcd_forward(stcd_plan* plan, const float* x1, const float* x2, int n_pairs,
                 float* const* outs, int n_outs, void* stream);

/* stcd_forward with every op bracketed by CUDA events (a measurement pass, not the product
 * path): op_ms[i] receives the device time of op i summed over the chunks; n_ops must equal the
 * number of ops added to the plan. Synchronises the stream. */
int stcd_forward_profile(stcd_plan* plan, const float* x1, const float* x2, int n_pairs,
                         float* const* outs, int n_outs, void* stream, float* op_ms, int n_ops);

/* Same, HOST (ideally pinned) buffers: H2D of each chunk overlaps the previous chunk's compute,
 * logits are copied back. Blocks until the results are in `outs_host`. */
int stcd_forward_host(stcd_plan* plan, const float* x1_host, const float* x2_host, int n_pairs,
                      float* const* outs_host, int n_outs);

/* stcd_forward / stcd_forward_host for plans whose input op is stcd_plan_add_input_pack_u8:
 * x1, x2 are uint8 HWC [n_pairs, H, W, cin] (device / host). */
int stcd_forward_u8(stcd_plan* plan, const uint8_t* x1, const uint8_t* x2, int n_pairs, float* const* outs, int n_outs,
                    void* stream);
int stcd_forward_host_u8(stcd_plan* plan, const uint8_t* x1_host, const uint8_t* x2_host, int n_pairs,
                         float* const* outs_host, int n_outs);

/* Replaces `pred = argmax / sigmoid>thr / raw>=thr` + SegmentationMetric.addBatch
 * (train_stcd.py:477,483,572-588; models/evaluator.py:108-113). cm_dev: int64[num_class^2]
 * device accumulator, rows = ground truth, cols = prediction (train_stcd.py:576). */
enum stcd_pred_kind {
  STCD_PRED_ARGMAX2 = 0,    /* logits fp32 [n,2,h,w]  -> (l1 > l0)   (torch.argmax ties -> 0) */
  STCD_PRED_SIGMOID_GT = 1, /* logits fp32 [n,1,h,w]  -> sigmoid(x) > thr   (train_stcd.py:477,483) */
  STCD_PRED_RAW_GE = 2,     /* logits fp32 [n,1,h,w]  -> x >= thr           (evaluator.py:111) */
  STCD_PRED_U8 = 3,         /* class ids uint8 */
  STCD_PRED_I32 = 4,        /* class ids int32 (pred.int(), train_stcd.py:483) */
  STCD_PRED_I64 = 5,        /* class ids int64 */
  STCD_PRED_U8_GE1 = 6      /* raw uint8 mask image ({0, 255} pseudo-label PNG): >= 1 -> class 1 */
};
/* STCD_LABEL_U8_GE1: raw uint8 label image, binarised on the fly like the reference's loader (label[label >= 1] = 1,
 * data/dataset.py:206-210): a {0, 255} PNG mask goes straight to the evaluator. */
enum stcd_label_kind { STCD_LABEL_I64 = 0, STCD_LABEL_U8 = 1, STCD_LABEL_I32 = 2, STCD_LABEL_U8_GE1 = 3 };

int stcd_confusion_add_batch(const void* pred, int pred_kind, float thr, const void* label,
                             int label_kind, int64_t n_img, int64_t pix_per_img, int num_class,
                             int64_t* cm_dev, uint8_t* pred_out_or_null, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* ViG Grapher graph ops (ChangeVIG path).  The reference imports them from `gcn_lib`              */
/* (models/pyramid_vig.py:17; call sites models/ChangeVIG.py:61-63), a module that is not in its    */
/* tree: semantics follow upstream vig_pytorch/gcn_lib (SURVEY.md App. D).  Layouts are the         */
/* reference's: node features fp32 [B][C][N] (= [B, C, N, 1]), neighbour tables int64.              */

/* Replaces DenseDilatedKnnGraph(k, dilation)(x, y, relative_pos) (gcn_lib/torch_edge.py): L2-normalise the
 * nodes over channels, dist = |x_i|^2 - 2 x_i.y_j + |y_j|^2 (+ relative_pos[i][j]), take the k*dilation nearest
 * y-nodes of every x-node in ascending distance (ties: smaller index) and keep every dilation-th.
 * x [B][C][N]; y [B][C][M] or NULL (y := x, M must equal N); relative_pos [N][M] or NULL; M <= 256, k*dilation <= M.
 * nn_idx_out: int64 [B][N][k] = edge_index[0] (edge_index[1] is the centre index n).
 * scratch: device fp32 [B * C * (N + M)] (the L2-normalised copies of x and y; B * C * N when y is NULL) -- used by the fp32
 * kernel (k * dilation > 27); the tensor-core kernel takes its plane workspace from the stream-ordered memory pool. */
int stcd_knn_graph(const float* x, const float* y_or_null, const float* relative_pos_or_null, int B, int C, int N,
                   int M, int k, int dilation, int64_t* nn_idx_out, float* scratch, void* stream);

/* Replaces the aggregation of MRConv2d.forward (gcn_lib/torch_vertex.py): m = max_k (y_j - x_i).
 * interleave = 0: out fp32 [B][C][N] = m.  interleave = 1: out fp32 [B][2C][N], channel 2c = x_c, 2c + 1 = m_c
 * (the channel-interleaved tensor MRConv2d feeds to its grouped 1x1 conv). */
int stcd_max_relative(const float* x, const float* y_or_null, const int64_t* nn_idx, int B, int C, int N, int M,
                      int k, int interleave, float* out, void* stream);

/* Pseudo-label write path (SURVEY.md §8(f)-2; train_stcd.py:155-196, train_pse_cd.py:145): binarise fp32 logits
 * [n][1 or 2][pix] with `pred_kind` (ARGMAX2 / SIGMOID_GT / RAW_GE) and write the uint8 mask image the script saves
 * as PNG: `on_value` (255, train_stcd.py:185) where the change class wins, else 0. */
int stcd_binarise_mask(const float* logits, int pred_kind, float thr, int64_t n_img, int64_t pix_per_img,
                       int on_value, uint8_t* mask_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STCD_B200_H_ */
