"""Lowering of reference modules to the fused-op program libstcd_b200 executes.

A *program* is a list of ops over bf16 activation tensors (logical NHWC here; stored
channel-chunked [img][c/8][h][w][8] on the device) holding ``mult * chunk`` images (``mult`` = 2
for tensors that carry both temporal streams: T1 images first, then T2 images).  The only
compute op is the implicit-GEMM convolution (``ConvSpec``): its A operand is described by a
K-program (list of ``Chunk``: which source tensor, which channel block, which pixel box, and
the filter taps that read that box),
its B operand is a host-packed bf16 weight matrix, and its epilogue carries the folded
BatchNorm, ReLU, residual add, Siamese ``|f1 - f2|`` and 2x2 max-pool.

Everything here is pure host logic (numpy/torch on CPU): it is what ``tests/`` checks against
the reference without a GPU (through ``oracle/emulate.py``), and what ``plan.py`` hands to the
C-ABI on the GPU box.
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

TILE_H, TILE_W = 16, 8
MAX_SRC = 6
MAX_CHUNKS, MAX_TAPS = 128, 512


def _bf16_bits(x: torch.Tensor) -> np.ndarray:
    """fp32 tensor -> uint16 bit patterns of its round-to-nearest-even bf16 value."""
    return x.detach().to(torch.float32).contiguous().to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def bf16_bits_to_f32(bits: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(bits.view(np.int16).copy()).view(torch.bfloat16).to(torch.float32)


@dataclass
class TensorSpec:
    name: str
    mult: int  # images = mult * chunk
    h: int
    w: int
    c: int


@dataclass
class Chunk:
    """One A-stage load: channels [c0, c0+kc) of source `src` over the box whose origin is
    (ty*sy + by, tx*sx + bx) for the tile at tile-pixel (ty, tx); feeds taps [tap_begin, +n_taps)."""
    src: int
    c0: int
    by: int
    bx: int
    stream: int   # image offset in units of `chunk` (0: same image, 1: the T2 partner)
    tap_begin: int
    n_taps: int


@dataclass
class Phase:
    chunk_begin: int
    chunk_count: int
    oy: int
    ox: int
    w_block: int
    n_blocks: int


@dataclass
class ConvSpec:
    name: str
    srcs: List[str]
    src_sy: List[int]
    src_sx: List[int]
    src_ey: List[int]
    src_ex: List[int]
    hg: int
    wg: int
    img_mult: int
    pair: bool
    weights: np.ndarray          # uint16 [n_ntiles, total blocks, kc/8, n_tile, 8] (bf16 bits)
    kc: int
    n_tile: int
    cout: int
    cout_pad: int
    phases: List[Phase]
    chunks: List[Chunk]
    taps: List[Tuple[int, int]]  # (ty, tx) inside the chunk's box; tap t of a phase <-> weight block t
    osy: int
    osx: int
    scale: np.ndarray            # float32 [cout_pad]
    shift: np.ndarray
    scale2: Optional[np.ndarray] = None
    shift2: Optional[np.ndarray] = None
    relu: bool = False
    res: Optional[str] = None
    out0: Optional[str] = None
    out0_coff: int = 0
    out_raw: Optional[str] = None
    out_pool: Optional[str] = None
    out_diff: Optional[str] = None
    out_ext: int = -1
    macs_per_pair: int = 0       # reference-equivalent MACs (for the roofline), per image pair
    out0_s2d: bool = False       # out0 is stored space-to-depth: pixel (y, x), channel c ->
    #                              pixel (y//2, x//2), channel ((y%2)*2 + x%2) * cout + c
    fold_cs: int = 0             # > 0: output phases are folded into GEMM N: column p*fold_cs + c of GEMM phase (oy, ox) is
    fold_cout: int = 0           # channel c (< fold_cout) of output pixel (i*osy + oy + p//osx, j*osx + ox + p%osx);
    #                              all osy*osx phases in ONE GEMM phase (oy = ox = 0), or the osx horizontal ones per row parity
    # activation: 0 none, 1 ReLU, 2 GELU (erf), 3 PReLU with one slope `act_alpha`.  act_pre: the activation sits
    # BEFORE the second affine (conv -> PReLU -> BN, ChangeFormer.py:1138-1148) instead of at the end of the epilogue
    act_kind: int = 0
    act_alpha: float = 0.0
    act_pre: bool = False
    # > 0: horizontal tap folding of a stride-1 3x3 conv (csrc/conv_ws.cuh, E_XF): one tap per filter row whose weight block
    # stacks the row's three filter columns, n_tile = cout_pad = 3 * xf_cs; the epilogue sums the column blocks across
    # neighbouring pixels.  `cout` stays the real channel count.
    xf_cs: int = 0
    # split precision: every bf16 output is written as (hi, lo) planes (lo plane at channel offset = half the tensor's stored
    # channels) and the residual is read as hi + lo; the K-program already holds the (hi, lo, hi) x (Whi, Whi, Wlo) segments
    split: bool = False

    def weight_block(self, nt: int, block: int) -> torch.Tensor:
        """fp32 [n_tile, kc] view of one packed weight block (for the emulator)."""
        w = bf16_bits_to_f32(self.weights[nt, block])            # [kc/8, n_tile, 8]
        return w.permute(1, 0, 2).reshape(self.n_tile, self.kc)


@dataclass
class InputPackSpec:
    name: str
    dst: str
    cin: int
    s2d: bool = False            # space-to-depth: dst is [h/2, w/2] with channel (py*2 + px)*cin + c (split: lo plane at 16 + that)
    # (mean, std) per channel: the plan's inputs are uint8 HWC images and the pack kernel applies the reference
    # loader's ToTensor + Normalize (data/dataset.py:196-203) before the bf16 rounding; None: fp32 NCHW inputs
    u8_norm: Optional[Tuple[Tuple[float, ...], Tuple[float, ...]]] = None
    split: bool = False          # split precision: channels [0, 8) hold bf16(x), [8, 16) hold bf16(x - bf16(x))


class SegTaps(list):
    """Per-segment tap lists of one phase: element i is the list of (dy, dx, W[cout, c_real_i]) taps
    that read segment i (an ordinary list of (dy, dx, W[cout, cin_total]) applies to every segment)."""


@dataclass
class MaxPoolS2DSpec:
    """nn.MaxPool2d(kernel_size=3, stride=2, padding=1) (torchvision ResNet stem;
    segmentation_models_pytorch/encoders/resnet.py:51) reading a space-to-depth tensor
    [n, h/2, w/2, 4c] and writing the pooled [n, h/2, w/2, c]."""
    name: str
    src: str
    dst: str
    c: int
    split: bool = False          # split precision: src holds hi of class k at k*c and lo at 4c + k*c; the max over hi + lo picks a pair


@dataclass
class GraphConvSpec:
    """The graph half of a ViG Grapher block (gcn_lib DyGraphConv2d up to MRConv2d's aggregation, SURVEY App. D):
    y = avg_pool2d(x, r) if r > 1 else x; dense dilated kNN graph of x over y (k neighbours, every dilation-th of
    the k*dilation nearest, + relative-position bias); dst = max_k (y_j - x_i), bf16.  src/dst: [imgs, h, w, c]."""
    name: str
    src: str
    dst: str
    c: int
    k: int
    dilation: int
    r: int
    relpos: Optional[np.ndarray]     # float32 [h*w, h*w / r^2] or None
    macs_per_pair: int = 0


@dataclass
class LayerNormSpec:
    """nn.LayerNorm(c, eps) over the channels of every pixel / token (ChangeFormer.py:226,475,480; biased variance,
    fp32 statistics), bf16 in -> bf16 out.  dst_s2d: optional second copy stored space-to-depth ([h/2, w/2, 4c]) for a
    following stride-2 patch-embedding conv."""
    name: str
    src: str
    dst: str
    c: int
    gamma: np.ndarray
    beta: np.ndarray
    eps: float
    dst_s2d: Optional[str] = None
    split: bool = False          # split precision: reads hi + lo, writes both planes of dst (and of dst_s2d: lo of class k at 4c + k*c)


@dataclass
class AttentionSpec:
    """Spatial-reduction attention of a MiT block (ChangeFormer.py:338-358): softmax(q k^T * scale) v per head.
    q: [imgs, h, w, c] (head hd = channels [hd*d, (hd+1)*d)); kv: [imgs, hk, wk, 2c] (k = channels [0, c), v = [c, 2c));
    dst: [imgs, h, w, c].  fp32 scores / softmax on bf16 operands."""
    name: str
    q: str
    kv: str
    dst: str
    c: int
    heads: int
    scale: float
    macs_per_pair: int = 0
    split: bool = False          # split precision: S = QhKh + QlKh + QhKl, O = PhVh + PlVh + PhVl (P split after the fp32 softmax)


@dataclass
class DWConvSpec:
    """Depth-wise 3x3 conv (padding 1) + bias, then an optional GELU: Mlp.dwconv + act (ChangeFormer.py:283-289,512-523)."""
    name: str
    src: str
    dst: str
    c: int
    weight: np.ndarray           # float32 [c][9]
    bias: np.ndarray             # float32 [c]
    gelu: bool = True
    macs_per_pair: int = 0
    split: bool = False          # split precision: reads hi + lo, writes both planes


@dataclass
class BilinearUpSpec:
    """F.interpolate(x, scale_factor=scale, mode="bilinear", align_corners=False) (ChangeVIG.py:246-262: `resize` and
    `F.interpolate(_c4, scale_factor=2, mode="bilinear")`) on a bf16 tensor; dst is [imgs, scale*h, scale*w, c]."""
    name: str
    src: str
    dst: str
    c: int
    scale: int
    split: bool = False          # split precision: reads hi + lo, writes both planes


@dataclass
class AbsDiffSpec:
    """dst = |src[T1 images] - src[T2 images]| (torch.abs(f1 - f2), smp FFCTLCD.forward, decoders/unet/model.py:412):
    src holds both streams (mult 2), dst one (mult 1); any layout (elementwise), first c channels."""
    name: str
    src: str
    dst: str
    c: int
    signed: bool = False         # True: (add +) src[T1] - src[T2], no abs (DTCDSCN: decoder(..) + e_x - e_y, models/DTCDSCN.py:294-300)
    add: Optional[str] = None
    split: bool = False          # split precision: reads hi + lo, writes both planes


@dataclass
class ChannelGateSpec:
    """Squeeze-and-excitation gates of DTCDSCN (models/DTCDSCN.py): g = sigmoid(w2 relu(w1 mean_hw(src))).
    mode 0 (SEBasicBlock tail :93-109): dst = relu(src * g + res); mode 1 (DecoderBlock :129-135 with SCSEBlock :144-173):
    dst = src * (1 + g + sigmoid(ws . src_pixel)).  dst_s2d: optional space-to-depth copy."""
    name: str
    src: str
    dst: str
    c: int
    w1: np.ndarray               # float32 [hid][c]
    w2: np.ndarray               # float32 [c][hid]
    mode: int = 0
    res: Optional[str] = None
    ws: Optional[np.ndarray] = None   # float32 [c]
    dst_s2d: Optional[str] = None
    split: bool = False          # split precision: reads src / res as hi + lo, writes both planes (dst_s2d: lo of class k at 4c + k*c)


@dataclass
class BitTransformerSpec:
    """BIT's token path on a 32-channel feature map (models/networks.py:359-394,405-428; blocks in models/help_funcs.py):
    semantic tokens (softmax over pixels of a 1x1 conv, :359-367), + learned positions, transformer encoder over the 2L
    tokens of the pair, transformer decoder where every pixel queries its image's L tokens; src and dst hold both streams.

    enc / dec are flat fp32 arrays, one row per layer (``bit_pack_enc`` / ``bit_pack_dec`` give the layouts)."""
    name: str
    src: str
    dst: str
    c: int                       # 32
    token_len: int               # 4
    heads: int                   # 8
    inner_enc: int               # heads * dim_head
    inner_dec: int               # heads * decoder_dim_head
    mlp: int                     # 64
    conv_a: np.ndarray           # float32 [token_len, c]
    pos: np.ndarray              # float32 [2 * token_len, c]
    enc: np.ndarray              # float32 [n_enc, bit_enc_size]
    dec: np.ndarray              # float32 [n_dec, bit_dec_size]
    softmax: bool = True
    macs_per_pair: int = 0
    split: bool = False          # split precision: the map is read as hi + lo and written as both planes (the token path is fp32)


def bit_enc_fields(c: int, inner: int, mlp: int):
    """(name, shape) of one encoder layer's packed parameters, in order (torch layouts: Linear weight = [out, in])."""
    return [("ln1_g", (c,)), ("ln1_b", (c,)), ("wqkv", (3 * inner, c)), ("wout", (c, inner)), ("bout", (c,)),
            ("ln2_g", (c,)), ("ln2_b", (c,)), ("w1", (mlp, c)), ("b1", (mlp,)), ("w2", (c, mlp)), ("b2", (c,))]


def bit_dec_fields(c: int, inner: int, mlp: int):
    """One decoder layer; to_out and the feed-forward weights are stored TRANSPOSED ([in, out]): the kernels read rows."""
    return [("ln1_g", (c,)), ("ln1_b", (c,)), ("wq", (inner, c)), ("wk", (inner, c)), ("wv", (inner, c)), ("woutt", (inner, c)),
            ("bout", (c,)), ("ln2_g", (c,)), ("ln2_b", (c,)), ("w1t", (c, mlp)), ("b1", (mlp,)), ("w2t", (mlp, c)), ("b2", (c,))]


def bit_pack(fields, values: Dict[str, torch.Tensor]) -> np.ndarray:
    out = []
    for name, shape in fields:
        v = values[name].detach().to(torch.float32).reshape(-1).numpy()
        if v.size != int(np.prod(shape)):
            raise ValueError(f"BIT packing: {name} has {v.size} elements, layout wants {shape}")
        out.append(v)
    return np.concatenate(out).astype(np.float32)


def bit_unpack(fields, row: np.ndarray) -> Dict[str, torch.Tensor]:
    out, o = {}, 0
    for name, shape in fields:
        n = int(np.prod(shape))
        out[name] = torch.from_numpy(np.ascontiguousarray(row[o: o + n])).reshape(shape)
        o += n
    assert o == row.size
    return out


@dataclass
class ChannelAttentionSpec:
    """dst = cat(srcs) * ca(cat(srcs)), ca = sigmoid(fc2(relu(fc1(avgpool))) + fc2(relu(fc1(maxpool)))) (ChannelAttention,
    models/DSIFN.py:24-36; `x = self.caK(x) * x`, :140,154,166,178).  The concat is virtual on the input side; dst is the
    materialised, scaled concat [chunk, h, w, sum(c)] the next conv reads."""
    name: str
    srcs: List[Tuple[str, int, int]]     # (tensor, stream, channels)
    dst: str
    fc1: np.ndarray                      # float32 [hid][C]
    fc2: np.ndarray                      # float32 [C][hid]


@dataclass
class SpatialGateSpec:
    """dst = bn(sa(x) * x), sa = sigmoid(conv7x7([mean_c x, max_c x])) (SpatialAttention, models/DSIFN.py:39-51; :131-132 ...)."""
    name: str
    src: str
    dst: str
    c: int
    w: np.ndarray                        # float32 [2][7][7]
    scale: np.ndarray                    # float32 [c]  folded BatchNorm
    shift: np.ndarray


@dataclass
class GlobalLocalGateSpec:
    """Global branch of ChangeGNNV2's Global_Local (models/ChangeVIG.py:377-385): dst = sigmoid(ch[c] * sp[pixel]) * src,
    ch = relu((w_avg avg + w_max max) * scale + shift) (grouped (2,1) conv, bias + BN folded), sp = relu(conv5x5([mean, max]) + b)."""
    name: str
    src: str
    dst: str
    c: int
    w_avg: np.ndarray            # float32 [c]
    w_max: np.ndarray
    scale: np.ndarray
    shift: np.ndarray
    w_sp: np.ndarray             # float32 [2][5][5]
    b_sp: float

    def packed(self) -> np.ndarray:
        return np.concatenate([self.w_avg, self.w_max, self.scale, self.shift, self.w_sp.reshape(-1), [self.b_sp]]).astype(np.float32)


@dataclass
class CsamGateSpec:
    """csam_V20 (models/ChangeVIG.py:956-994): dst = bt((sigmoid(ch[c]) + sigmoid(sp[pixel])) * src); ch = liner2(relu(liner1(gelu(
    (w_avg avg + w_max max) * scale + shift)))), sp = conv3x3(relu(conv3x3([mean, max]))) (both bias-free)."""
    name: str
    src: str
    dst: str
    c: int
    w_avg: np.ndarray            # float32 [c]
    w_max: np.ndarray
    scale: np.ndarray            # conv1_1 bias + batch_normal1 folded
    shift: np.ndarray
    l1: np.ndarray               # float32 [hid][c]
    l2: np.ndarray               # float32 [c][hid]
    b2: np.ndarray               # float32 [c]
    bt_scale: np.ndarray
    bt_shift: np.ndarray
    w21: np.ndarray              # float32 [2][3][3]
    w22: np.ndarray              # float32 [3][3]

    def packed(self) -> np.ndarray:
        return np.concatenate([self.w_avg, self.w_max, self.scale, self.shift, self.l1.reshape(-1), np.ascontiguousarray(self.l2.T).reshape(-1),
                               self.b2, self.bt_scale, self.bt_shift, self.w21.reshape(-1), self.w22.reshape(-1)]).astype(np.float32)


@dataclass
class VffmSpec:
    """VFFM (models/ChangeVIG.py:452-460): dst = 2 low wei + 2 high (1 - wei), wei = sigmoid(MLP_avg(avgpool(mixed)) +
    MLP_max(maxpool(mixed)) + local).  branches: (avg, max), each dict(w1 [inter][c], s1, t1, w2 [c][inter], s2, t2) with the
    conv biases and BatchNorms folded into scale / shift."""
    name: str
    low: str
    high: str
    mixed: str
    local: str
    dst: str
    c: int
    inter: int
    branches: Tuple[Dict[str, np.ndarray], Dict[str, np.ndarray]]

    def packed(self) -> np.ndarray:
        out = []
        for b in self.branches:
            out += [b["w1"].reshape(-1), b["s1"], b["t1"], np.ascontiguousarray(b["w2"].T).reshape(-1), b["s2"], b["t2"]]
        return np.concatenate(out).astype(np.float32)


@dataclass
class SumSpec:
    """dst = sum of up to five tensors (Dblock.forward, models/DTCDSCN.py:65-71)."""
    name: str
    srcs: List[str]
    dst: str
    split: bool = False          # split precision: the fp32 sum of hi + lo values, written as both planes


@dataclass
class SegHeadSpec:
    """SegCD's tail (segmentation_models_pytorch/decoders/unet/model.py:321-330) as ONE op over the
    decoder output d (both temporal streams, c channels): m1 = head(d1), m2 = head(d2),
    change = min(head(|d1 - d2|), |m1 - m2|) with head = Conv2d(c, 1, 3, padding=1)
    (base/heads.py:5-10).  External outputs out_ext, out_ext+1, out_ext+2 = m1, m2, change."""
    name: str
    src: str
    c: int
    weight: np.ndarray           # float32 [9][c]  (tap-major: ky*3 + kx)
    bias: float
    out_ext: int = 0
    macs_per_pair: int = 0
    # FFCTLCD (model.py:407-423): the feature-level branch is head(decoder(|f1 - f2|)): its decoder output arrives as
    # a separate single-stream tensor instead of |d1 - d2| computed from `src`
    diff_src: Optional[str] = None


@dataclass
class ExtOutput:
    name: str
    channels: int
    h: int
    w: int


@dataclass
class Program:
    model: str
    in_channels: int
    h: int
    w: int
    tensors: Dict[str, TensorSpec] = field(default_factory=dict)
    ops: List[object] = field(default_factory=list)
    ext: List[ExtOutput] = field(default_factory=list)
    # constant tensors (e.g. a positional embedding added as a residual): name -> fp32 [h, w, c], replicated over
    # the images of the tensor when the plan is built
    consts: Dict[str, torch.Tensor] = field(default_factory=dict)
    # "bf16": activations are single bf16 values (north star: logits within 2e-2).
    # "split": the precision path the reference API calls tf32 (north star: logits within 1e-3).  Every activation and weight
    # is carried as a (hi, lo) PAIR of bf16 values -- hi = bf16(v), lo = bf16(v - hi): 16 mantissa bits, against tf32's 11 --
    # and every product as hi*hi + lo*hi + hi*lo in fp32 accumulators (the lo*lo term is below 2**-16 relative).  Plain
    # kind::tf32 MMAs do NOT meet 1e-3 on these nets (measured with tf32-rounded operands on the oracle, logit std 0.42:
    # max error 3.7e-3); the split form does (~6e-5), on the same bf16 tensor-core path: a tensor holds its hi plane in
    # channels [0, C) and its lo plane in [C, 2C), a conv reads (hi, lo, hi) as three K segments with weights (Whi, Whi, Wlo)
    # -- 3 bf16 MMAs per product where kind::tf32 would spend the time of 2, at the same 4 bytes per activation.
    precision: str = "bf16"

    @property
    def split(self) -> bool:
        return self.precision == "split"

    def tensor(self, name: str, mult: int, h: int, w: int, c: int) -> str:
        """Declare an activation tensor of `c` logical channels (split precision: 2c stored, hi plane then lo plane)."""
        if name in self.tensors:
            raise ValueError(f"duplicate tensor {name}")
        if c % 8:
            raise ValueError(f"tensor {name}: channels {c} must be a multiple of 8")
        self.tensors[name] = TensorSpec(name, mult, h, w, 2 * c if self.split else c)
        return name

    def half(self, name: str) -> int:
        """Logical channel count of a tensor (= the offset of its lo plane in split precision)."""
        t = self.tensors[name]
        return t.c // 2 if self.split else t.c

    def macs_per_pair(self) -> int:
        return sum(getattr(o, "macs_per_pair", 0) for o in self.ops)


# ------------------------------------------------------------------------------------------
# folding


def fold_bn(bias: Optional[torch.Tensor], bn: Optional[Dict[str, torch.Tensor]], cout: int, eps: float = 1e-5
            ) -> Tuple[np.ndarray, np.ndarray]:
    """Eval-mode BatchNorm2d after a biased conv as one affine: y = acc*scale + shift.

    scale = gamma / sqrt(var + eps); shift = beta + (bias - mean) * scale  (SURVEY App. A;
    reference: SiamUnet_diff.py:99 ``relu(bn11(conv11(x)))`` with running statistics).
    """
    b = torch.zeros(cout, dtype=torch.float64) if bias is None else bias.detach().to(torch.float64)
    if bn is None:
        return np.ones(cout, np.float32), b.to(torch.float32).numpy()
    g = bn["weight"].detach().to(torch.float64)
    beta = bn["bias"].detach().to(torch.float64)
    mean = bn["running_mean"].detach().to(torch.float64)
    var = bn["running_var"].detach().to(torch.float64)
    scale = g / torch.sqrt(var + eps)
    shift = beta + (b - mean) * scale
    return scale.to(torch.float32).numpy(), shift.to(torch.float32).numpy()


def bn_params(sd: Dict[str, torch.Tensor], prefix: str) -> Dict[str, torch.Tensor]:
    return {k: sd[f"{prefix}.{k}"] for k in ("weight", "bias", "running_mean", "running_var")}


def _pad_vec(v: np.ndarray, n: int, fill: float) -> np.ndarray:
    out = np.full(n, fill, np.float32)
    out[: v.shape[0]] = v
    return out


# ------------------------------------------------------------------------------------------
# K-program / weight packing


@dataclass
class Segment:
    """A channel segment of the virtual concat: channels [0, c_real) of `tensor` (whose storage
    may be padded to more channels) at temporal stream `stream`."""
    tensor: str
    c_real: int
    stream: int = 0
    sy: int = 1
    sx: int = 1
    c_off: int = 0          # first channel of the segment inside `tensor` (multiple of 8)
    c_store: int = -1       # stored width of the segment (default: the rest of the tensor)


FAST_MMA = 36        # stcd::kFastMma: taps x K-steps of one chunk that fit the issue path's constant-bank table


def choose_kc(c_list: Sequence[int], taps_per_chunk: int = 1, cap: int = 112) -> int:
    """Channels per A-stage chunk.  Stored channel counts are multiples of 8; a count that is an odd
    multiple of 8 is covered by a 16-channel chunk whose missing half TMA zero-fills.

    Powers of two first (64, 32, 16).  Channel counts like 80 / 160 / 400 / 800 (the ViG pyramid) only divide by 16 or 32: a
    400-channel 1x1 conv would run 25 one-MMA chunks and pay the per-chunk pipeline hand-off 25 times (measured 6-12x above
    the layer's floor), so any multiple of 16 up to 112 that divides every segment is taken instead (80 -> 5 K-steps per chunk)
    as long as the chunk's taps x K-steps still fit the fast issue path."""
    stored = [(c + 15) // 16 * 16 for c in c_list]
    best = next((kc for kc in (64, 32, 16) if kc <= max(cap, 16) and all(s % kc == 0 for s in stored)), None)
    if best is None:
        raise ValueError(f"channel counts {list(c_list)} are not multiples of 8")
    if best < 64:
        for kc in range(min(cap, 112) // 16 * 16, best, -16):
            if all(s % kc == 0 for s in stored) and taps_per_chunk * (kc // 16) <= FAST_MMA:
                return kc
    return best


NARROW_K_MMAS = int(os.environ.get("STCD_NARROW_K", "24"))       # measured: C4 +2.8 %, C5 +3 %, SegCD-R50 +3.5 % against 0


def choose_n_tile(cout: int, pair: bool, k_mmas: int = 1 << 30) -> Tuple[int, int]:
    """N per CTA: accumulators are double-buffered in TMEM (512 columns): 2 * (2 if pair else 1) * n_tile <= 512.

    Narrow-K ops (k_mmas = MMAs per tile <= NARROW_K_MMAS, e.g. the 1x1 convs of the ViG / MiT blocks) are bound by their epilogue,
    not by the tensor pipe: a pair op with N = 128 owns all 512 TMEM columns, i.e. ONE CTA and four epilogue warps per SM.  N = 64
    halves the accumulator, so two CTAs share the SM and twice as many epilogue warps drain it (and 320 outputs are 5 x 64 instead
    of 3 x 128 with 17 % padding)."""
    cp = (cout + 15) // 16 * 16
    limit = 128 if pair else 256
    if k_mmas <= NARROW_K_MMAS and cp > 64:
        cp = (cout + 63) // 64 * 64
        return 64, cp
    if cp <= limit:
        return cp, cp
    cp = (cout + 127) // 128 * 128
    return 128, cp


def _taps_to_gemm(
    prog: Program,
    name: str,
    segs: Sequence[Segment],
    phase_taps: Sequence[Tuple[int, int, List[Tuple[int, int, torch.Tensor]]]],
    cout: int,
    pair: bool,
    max_kc: int = 64,
    force_n_tile: int = 0,
):
    """Build the K-program and the packed weights.

    phase_taps: per phase (oy, ox, [(dy, dx, W[cout, cin_total])...]): dy/dx are input offsets in
    un-strided source pixels relative to (tile pixel * source stride); cin_total indexes the
    concatenated segments.

    Stride-1 sources load ONE box per (phase, channel chunk) that covers every tap of the phase
    (halo reuse); strided sources load one box per tap.
    """
    srcs: List[str] = []
    for s in segs:
        if s.tensor not in srcs:
            srcs.append(s.tensor)
    if len(srcs) > MAX_SRC:
        raise ValueError(f"{name}: {len(srcs)} sources > {MAX_SRC}")
    stored_c = [(prog.tensors[s.tensor].c - s.c_off) if s.c_store < 0 else s.c_store for s in segs]
    for s in segs:
        if s.c_off % 8:
            raise ValueError(f"{name}: segment channel offset {s.c_off} is not a multiple of 8")
    n_nt = 0
    sy = [1] * len(srcs)
    sx = [1] * len(srcs)
    for s in segs:
        sy[srcs.index(s.tensor)] = s.sy
        sx[srcs.index(s.tensor)] = s.sx

    # per phase, per segment: [(dy, dx, W[cout, c_real])]
    seg_phase_taps = [(oy, ox, _split_taps(name, segs, taps)) for (oy, ox, taps) in phase_taps]
    max_taps = max((len(t) for (_, _, staps) in seg_phase_taps for t in staps), default=1)
    # wide halos (dilated convs) take thinner chunks: the A stage is (tile + halo) * kc
    kc = choose_kc(stored_c, max(1, max_taps), cap=max_kc if max_kc < 64 else 112)
    k_mmas = max((sum(len(t) * -(-sc_ // 16) for sc_, t in zip(stored_c, staps)) for (_, _, staps) in seg_phase_taps), default=1)
    n_tile, cout_pad = (force_n_tile, force_n_tile) if force_n_tile else choose_n_tile(cout, pair, k_mmas)
    n_nt = cout_pad // n_tile
    # halo extents per source: max over phases and segments of the tap range (stride-1 sources only)
    ey = [0] * len(srcs)
    ex = [0] * len(srcs)
    for (_, _, staps) in seg_phase_taps:
        for s, taps in zip(segs, staps):
            i = srcs.index(s.tensor)
            if taps and sy[i] == 1 and sx[i] == 1:
                dys = [t[0] for t in taps]
                dxs = [t[1] for t in taps]
                ey[i] = max(ey[i], max(dys) - min(dys))
                ex[i] = max(ex[i], max(dxs) - min(dxs))
    phases: List[Phase] = []
    chunks: List[Chunk] = []
    tap_list: List[Tuple[int, int]] = []
    blocks: List[torch.Tensor] = []          # each [cout_pad, kc]
    for (oy, ox, staps) in seg_phase_taps:
        chunk_begin, w_block = len(chunks), len(blocks)
        for s, sc, taps in zip(segs, stored_c, staps):
            if not taps:
                continue
            si = srcs.index(s.tensor)
            halo = (sy[si] == 1 and sx[si] == 1)
            dy0 = min(t[0] for t in taps)
            dx0 = min(t[1] for t in taps)
            for w in taps:
                if w[2].shape[1] != s.c_real:
                    raise ValueError(f"{name}: tap weight has {w[2].shape[1]} channels, segment has {s.c_real}")
            for c0 in range(0, sc, kc):
                if c0 >= s.c_real:      # pure padding chunk: contributes nothing
                    continue

                def wblock(wtap):
                    blk = torch.zeros(cout_pad, kc, dtype=torch.float32)
                    n_real = min(kc, s.c_real - c0)
                    blk[:cout, :n_real] = wtap[:, c0: c0 + n_real]
                    return blk

                if halo:
                    chunks.append(Chunk(si, s.c_off + c0, dy0, dx0, s.stream, len(tap_list), len(taps)))
                    for (dy, dx, wtap) in taps:
                        tap_list.append((dy - dy0, dx - dx0))
                        blocks.append(wblock(wtap))
                else:
                    for (dy, dx, wtap) in taps:
                        chunks.append(Chunk(si, s.c_off + c0, dy, dx, s.stream, len(tap_list), 1))
                        tap_list.append((0, 0))
                        blocks.append(wblock(wtap))
        phases.append(Phase(chunk_begin, len(chunks) - chunk_begin, oy, ox, w_block, len(blocks) - w_block))
        if phases[-1].chunk_count > MAX_CHUNKS or phases[-1].n_blocks > MAX_TAPS:
            raise ValueError(f"{name}: K-program too long ({phases[-1].chunk_count} chunks, {phases[-1].n_blocks} taps)")
    wall = torch.stack(blocks, 0)                                    # [B, cout_pad, kc]
    wall = wall.reshape(len(blocks), n_nt, n_tile, kc // 8, 8)       # [B, nt, n, k8, 8]
    wall = wall.permute(1, 0, 3, 2, 4).contiguous()                  # [nt, B, k8, n, 8]
    return _bf16_bits(wall), kc, n_tile, cout_pad, phases, chunks, tap_list, srcs, sy, sx, ey, ex


def conv_taps(weight: torch.Tensor, pad: int, stride: int = 1) -> List[Tuple[int, int, List]]:
    """nn.Conv2d weight [cout, cin, kh, kw] -> one phase of taps (dy, dx, W[cout, cin])."""
    kh, kw = weight.shape[2], weight.shape[3]
    taps = [(ky - pad, kx - pad, weight[:, :, ky, kx].to(torch.float32)) for ky in range(kh) for kx in range(kw)]
    return [(0, 0, taps)]


def convT_as_conv_weight(weight_t: torch.Tensor) -> torch.Tensor:
    """ConvTranspose2d(stride=1) weight [cin, cout, k, k] -> equivalent Conv2d weight
    [cout, cin, k, k] (flip both spatial axes, swap channel axes); padding' = k - 1 - padding.
    Reference: the FC-Siam decoder "convs" are ConvTranspose2d(k=3, padding=1): SiamUnet_diff.py:54-90."""
    return weight_t.flip(2, 3).transpose(0, 1).contiguous()


def convT_phase_taps(weight_t: torch.Tensor, stride: int, pad: int) -> List[Tuple[int, int, List]]:
    """ConvTranspose2d weight [cin, cout, k, k], stride s -> s*s output phases.

    out[s*i + a] = sum over ky with (a + pad - ky) % s == 0 of in[i + (a + pad - ky)//s] * W[ky]
    (SiamUnet_diff.py:52 k3 s2 p1 op1; SNUNet.py:38 k2 s2; ChangeFormerBaseNetworks.py:101 k4 s2 p1).
    """
    k = weight_t.shape[2]
    out = []

    def axis(a):
        return [((a + pad - kk) // stride, kk) for kk in range(k) if (a + pad - kk) % stride == 0]

    for a in range(stride):
        for b in range(stride):
            taps = [(dy, dx, weight_t[:, :, ky, kx].transpose(0, 1).to(torch.float32))
                    for (dy, ky) in axis(a) for (dx, kx) in axis(b)]
            out.append((a, b, taps))
    return out


def s2d_segments(tensor: str, c: int, stream: int = 0) -> List[Segment]:
    """The four parity classes (py, px) of a space-to-depth tensor [n, h/2, w/2, 4c] as segments."""
    return [Segment(tensor, c, stream=stream, c_off=k * c, c_store=c) for k in range(4)]


def s2d_conv_taps(weight: torch.Tensor, pad: int, a: int = 0, b: int = 0) -> SegTaps:
    """Taps of a conv whose source is stored space-to-depth (see ``s2d_segments``) and whose output
    pixel (i, j) of the tile grid sits at full-resolution position (2i + a, 2j + b):
    out(i, j) = sum_k W[ky, kx] * src_full(2i + a + ky - pad, 2j + b + kx - pad).
    With a = b = 0 this is a stride-2 conv (torchvision BasicBlock conv1 / downsample,
    models/resnet.py:59-60); with (a, b) in {0,1}^2 the four output phases of a stride-1 conv at the
    source's full resolution (the skip half of smp's DecoderBlock.conv1, decoders/unet/decoder.py:35-40).
    Full-res row r = 2i + a + ky - pad belongs to parity class r % 2 at half-res row i + r // 2."""
    kh, kw = weight.shape[2], weight.shape[3]
    out = SegTaps([[] for _ in range(4)])
    for ky in range(kh):
        ry = a + ky - pad
        for kx in range(kw):
            rx = b + kx - pad
            out[(ry % 2) * 2 + (rx % 2)].append((ry // 2, rx // 2, weight[:, :, ky, kx].to(torch.float32)))
    return out


def up2_conv_taps(weight: torch.Tensor, pad: int, a: int, b: int) -> List[Tuple[int, int, torch.Tensor]]:
    """Taps of a conv over the NEAREST 2x up-sampling of a low-resolution source
    (F.interpolate(scale_factor=2, mode="nearest") + Conv2d, decoders/unet/decoder.py:36-40) for output
    phase (a, b): up(y) = src(y // 2), so taps that land on the same source pixel merge and their
    weights add (a 3x3 conv becomes 2x2 taps per phase: 4/9 of the MACs, and the up-sampled tensor is
    never materialised)."""
    kh, kw = weight.shape[2], weight.shape[3]
    merged: Dict[Tuple[int, int], torch.Tensor] = {}
    for ky in range(kh):
        dy = (a + ky - pad) // 2
        for kx in range(kw):
            dx = (b + kx - pad) // 2
            w = weight[:, :, ky, kx].to(torch.float32)
            merged[(dy, dx)] = merged[(dy, dx)] + w if (dy, dx) in merged else w.clone()
    return [(dy, dx, w) for (dy, dx), w in sorted(merged.items())]


XF_MAX_CS = int(os.environ.get("STCD_XF_MAX_CS", "64"))       # widest Cout (rounded up to 16) that takes horizontal tap folding; 0 disables
XF_MIN_W = 28


def xf_taps(name: str, segs: Sequence[Segment], phase_taps, cout: int, pair: bool, hg: int, wg: int):
    """Horizontal tap folding (ConvSpec.xf_cs): returns (single-phase SegTaps with one tap per filter row and [3*cs, c]
    weight blocks, cs) when the op is a stride-1 3x3 conv over stride-1 sources with Cout <= XF_MAX_CS, else None.

    An SS-mode tcgen05.mma M=128 K=16 costs ~45 cycles for N <= 64 and ~56 for N = 96 (A + B operand bytes over the
    128 B/clk shared-memory read): three taps per MMA instead of one cut the tensor-pipe cycles of a Cout-32 layer 2.4x
    (Cout 16: 3x); 14 of a tile's 16 columns are outputs, so the net gain is 2.1x / 2.6x."""
    cs = (cout + 15) // 16 * 16
    if not XF_MAX_CS or cs > XF_MAX_CS or len(phase_taps) != 1 or wg < XF_MIN_W or hg < 8:
        return None
    # Siamese-pair ops would need 2 x 2 x 3cs TMEM columns: one CTA per SM with four epilogue warps for twice the accumulator
    # reads -- measured 2x SLOWER than the tap-by-tap form (SNUNet conv0_0: 262 -> 525 us), and the pair layers of the
    # nets have too few input channels to profit anyway
    if pair:
        return None
    # Cost model (cycles per output pixel, measured MMA costs: tools/ubench/mma_n.cu).  The folded form reads 3x the accumulator
    # columns from TMEM (tools/ubench/tmem_read.cu: one 32-lane x 16-column load per 43 cycles and warp) and shuffles them --
    # an epilogue cost of ~24 * cs + 200 cycles per tile fits the measured crossovers -- so it only pays once the tile's MMAs
    # outlast that: e.g. Cout 32 from >= 48 input channels, Cout 16 from >= 32 (measured: SNUNet conv0_x.conv1, 128-224 input
    # channels, 907 -> 622 us; conv0_x.conv2, 32 input channels, 166 -> 222 us).
    k16 = sum((s.c_real + 15) // 16 for s in segs)
    cost_std = k16 * 9 * mma_cycles(cs) / 128.0
    cost_xf = max(k16 * 3 * mma_cycles(3 * cs), 24 * cs + 200) / 112.0
    if cost_xf >= cost_std:
        return None
    if any(s.sy != 1 or s.sx != 1 for s in segs):
        return None
    oy, ox, taps = phase_taps[0]
    per_seg = _split_taps(name, segs, taps)
    want = sorted((dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1))
    out = SegTaps([[] for _ in segs])
    for si, (s, t) in enumerate(zip(segs, per_seg)):
        if sorted((dy, dx) for (dy, dx, _) in t) != want:
            return None
        by_off = {(dy, dx): w for (dy, dx, w) in t}
        for dy in (-1, 0, 1):
            blk = torch.zeros(3 * cs, s.c_real, dtype=torch.float32)
            for b, dx in enumerate((-1, 0, 1)):
                blk[b * cs: b * cs + cout] = by_off[(dy, dx)]
            out[si].append((dy, 0, blk))
    return [(oy, ox, out)], cs


FOLD_X_MAX_N = int(os.environ.get("STCD_FOLD_X_MAX_N", "128"))   # widest GEMM N of a horizontally folded up-sampling op


def mma_cycles(n: int) -> int:
    """Measured cost of one SS-mode tcgen05.mma M=128 K=16 on B200 (tools/ubench/mma_rate.cu): for N <= 64 the
    4 KB A-operand read from shared memory, not the math, sets the pace."""
    return max(45, 32 + n // 4, n // 2)        # 45 (N <= 48), 48 (64), 56 (96), 64 (128), 96 (192), 128 (256)


def _split_taps(name: str, segs: Sequence[Segment], taps) -> List[list]:
    """One phase's taps as per-segment lists [(dy, dx, W[cout, c_real])]."""
    if isinstance(taps, SegTaps):
        if len(taps) != len(segs):
            raise ValueError(f"{name}: {len(taps)} tap lists for {len(segs)} segments")
        return [list(t) for t in taps]
    out, ci = [], 0
    for s in segs:
        out.append([(dy, dx, w[:, ci: ci + s.c_real]) for (dy, dx, w) in taps])
        ci += s.c_real
    for (_, _, w) in taps:
        if ci != w.shape[1]:
            raise ValueError(f"{name}: weight has {w.shape[1]} input channels, segments give {ci}")
    return out


def fold_phases_x(name: str, segs: Sequence[Segment], phase_taps, cout: int, osy: int, osx: int):
    """Fold only the osx HORIZONTAL output phases into GEMM N (one GEMM phase per output row parity).

    Column block px of row-parity phase oy owns output pixel (i*osy + oy, j*osx + px): a thread then holds the
    horizontally adjacent output pixels of its input pixel, and both halves of every 32-byte sector leave the SM
    together.  Per-phase launches wrote each sector half from different CTAs far apart in time: the up-sampling
    ops of SNUNet ran at 3 TB/s of store traffic (Up1_x: 263 us with the stores, 85 us without).
    Returns ([(oy, 0, SegTaps)] per row parity, cs)."""
    cs = (cout + 15) // 16 * 16
    per_phase = {(oy, ox): _split_taps(name, segs, taps) for (oy, ox, taps) in phase_taps}
    if sorted(per_phase) != [(a, b) for a in range(osy) for b in range(osx)]:
        raise ValueError(f"{name}: folding needs exactly one tap list per output phase")
    out = []
    for oy in range(osy):
        folded = SegTaps([[] for _ in segs])
        for si, s in enumerate(segs):
            merged: Dict[Tuple[int, int], torch.Tensor] = {}
            for ox in range(osx):
                for (dy, dx, w) in per_phase[(oy, ox)][si]:
                    blk = merged.setdefault((dy, dx), torch.zeros(osx * cs, s.c_real, dtype=torch.float32))
                    blk[ox * cs: ox * cs + cout] += w
            folded[si] = [(dy, dx, w) for (dy, dx), w in sorted(merged.items())]
        out.append((oy, 0, folded))
    return out, cs


def fold_phases(name: str, segs: Sequence[Segment], phase_taps, cout: int, osy: int, osx: int, pair: bool):
    """Fold the osy*osx output phases of an up-sampling op into the GEMM N dimension.

    Phase p = oy*osx + ox owns columns [p*cs, p*cs + cout) (cs = cout rounded up to 16).  Every distinct
    (segment, input offset) becomes ONE tap whose weight block holds each phase's weights for that offset (zeros
    for phases that do not read it): the A operand is fetched and multiplied once for all phases instead of
    once per phase, and N grows from cout to P*cs -- which is what small-cout layers need, since an SS-mode
    MMA costs the same 45 cycles for any N <= 64.  Returns (single-phase taps, cs, cost_folded, cost_unfolded)
    in modelled MMA cycles per tile, so the caller can keep the per-phase form when folding does not pay
    (wide layers, where the zero blocks cost more than the shared operand saves)."""
    P = osy * osx
    cs = (cout + 15) // 16 * 16
    per_phase = [(oy * osx + ox, _split_taps(name, segs, taps)) for (oy, ox, taps) in phase_taps]
    if sorted(p for p, _ in per_phase) != list(range(P)):
        raise ValueError(f"{name}: folding needs exactly one tap list per output phase")
    folded = SegTaps([[] for _ in segs])
    k16 = [(s.c_real + 15) // 16 for s in segs]
    cost_unf = 0
    for si, s in enumerate(segs):
        merged: Dict[Tuple[int, int], torch.Tensor] = {}
        for p, staps in per_phase:
            for (dy, dx, w) in staps[si]:
                blk = merged.setdefault((dy, dx), torch.zeros(P * cs, s.c_real, dtype=torch.float32))
                blk[p * cs: p * cs + cout] += w
            cost_unf += len(staps[si]) * k16[si]
        folded[si] = [(dy, dx, w) for (dy, dx), w in sorted(merged.items())]
    n_unf, pad_unf = choose_n_tile(cout, pair)
    n_f, pad_f = choose_n_tile(P * cs, pair)
    cost_unf *= mma_cycles(n_unf) * (pad_unf // n_unf)
    cost_f = sum(len(t) * k for t, k in zip(folded, k16)) * mma_cycles(n_f) * (pad_f // n_f)
    return [(0, 0, folded)], cs, cost_f, cost_unf


def _split_operands(prog: Program, name: str, segs: Sequence[Segment], phase_taps):
    """Split precision: a * w  ->  a_hi * w_hi + a_lo * w_hi + a_hi * w_lo as three K segments per logical segment.

    Segment s over tensor T (hi plane at channel s.c_off, lo plane at half(T) + s.c_off) becomes
    (hi plane, W_hi), (lo plane, W_hi), (hi plane, W_lo) with W_hi = bf16(W), W_lo = W - W_hi (rounded to bf16 by the
    weight packer).  Returns (segments, [(oy, ox, SegTaps)])."""
    out_segs: List[Segment] = []
    for s in segs:
        half = prog.half(s.tensor)
        store = (half - s.c_off) if s.c_store < 0 else s.c_store
        hi = Segment(s.tensor, s.c_real, s.stream, s.sy, s.sx, s.c_off, store)
        lo = Segment(s.tensor, s.c_real, s.stream, s.sy, s.sx, half + s.c_off, store)
        out_segs += [hi, lo, hi]
    out_taps = []
    for (oy, ox, taps) in phase_taps:
        per_seg = _split_taps(name, segs, taps)
        st = SegTaps()
        for t in per_seg:
            w_hi = [(dy, dx, w.to(torch.bfloat16).to(torch.float32)) for (dy, dx, w) in t]
            w_lo = [(dy, dx, w - wh) for (dy, dx, w), (_, _, wh) in zip(t, w_hi)]
            st += [w_hi, list(w_hi), w_lo]
        out_taps.append((oy, ox, st))
    return out_segs, out_taps


def add_conv(
    prog: Program,
    name: str,
    segs: Sequence[Segment],
    phase_taps,
    cout: int,
    hg: int,
    wg: int,
    img_mult: int,
    scale: np.ndarray,
    shift: np.ndarray,
    *,
    pair: bool = False,
    relu: bool = False,
    osy: int = 1,
    osx: int = 1,
    scale2: Optional[np.ndarray] = None,
    shift2: Optional[np.ndarray] = None,
    res: Optional[str] = None,
    out0: Optional[str] = None,
    out0_coff: int = 0,
    out_raw: Optional[str] = None,
    out_pool: Optional[str] = None,
    out_diff: Optional[str] = None,
    out_ext: int = -1,
    macs_per_pair: int = 0,
    out0_s2d: bool = False,
    fold: Optional[bool] = None,
    act: Optional[str] = None,
    act_alpha: float = 0.0,
    act_pre: bool = False,
    max_kc: int = 64,
) -> ConvSpec:
    if act is not None and relu:
        raise ValueError(f"{name}: give either relu=True or act=...")
    act_kind = 1 if relu else {None: 0, "relu": 1, "gelu": 2, "prelu": 3}[act]
    relu = act_kind != 0          # the epilogue's "has activation" switch
    if act_pre and scale2 is None:
        raise ValueError(f"{name}: act_pre needs the second affine")
    split = prog.split
    if split:
        fold = False                # folded / horizontally folded forms keep their specialised bf16 epilogues
        segs, phase_taps = _split_operands(prog, name, segs, phase_taps)
        parts = _k_partition(prog, name, segs, phase_taps, cout, pair, max_kc)
        if len(parts) > 1:
            plain = (res is None and out_raw is None and out_pool is None and out_diff is None and out_ext < 0 and scale2 is None
                     and out0 is not None and len(phase_taps) == 1 and osy == 1 and osx == 1)
            if not plain:
                raise NotImplementedError(f"{name}: the split K-program is too long and only single-phase affine + activation + out0 "
                                          "ops are partitioned along K")
            return _add_k_partitioned(prog, name, segs, phase_taps, parts, cout, hg, wg, img_mult, scale, shift, pair=pair,
                                      out0=out0, out0_coff=out0_coff, macs_per_pair=macs_per_pair, act_kind=act_kind,
                                      act_alpha=act_alpha, max_kc=max_kc)
    fold_cs = fold_cout = 0
    plain_out = (res is None and out_raw is None and out_pool is None and out_diff is None and out_ext < 0
                 and scale2 is None and not out0_s2d and out0 is not None)
    if fold is not False and osy * osx > 1 and len(phase_taps) == osy * osx and plain_out:
        f_taps, cs, cost_f, cost_unf = fold_phases(name, segs, phase_taps, cout, osy, osx, pair)
        # measured (SNUNet Up1_x, C=64): a folded N=256 tile is slower than four N=64 phases (one accumulator set,
        # occupancy 1); fold only while the whole op is one N <= 128 tile
        if fold or (cost_f < cost_unf and osy * osx * cs <= 128):
            P = osy * osx
            fold_cs, fold_cout = cs, cout
            sc = np.ones(P * cs, np.float32)
            sh = np.zeros(P * cs, np.float32)
            for p_ in range(P):
                sc[p_ * cs: p_ * cs + cout] = scale[:cout]
                sh[p_ * cs: p_ * cs + cout] = shift[:cout]
            phase_taps, cout, scale, shift = f_taps, P * cs, sc, sh
        elif osx > 1 and osx * cs <= FOLD_X_MAX_N:
            # not one tile: fold the horizontal phases only (stores of adjacent output pixels leave together)
            f_taps, cs = fold_phases_x(name, segs, phase_taps, cout, osy, osx)
            fold_cs, fold_cout = cs, cout
            sc = np.ones(osx * cs, np.float32)
            sh = np.zeros(osx * cs, np.float32)
            for p_ in range(osx):
                sc[p_ * cs: p_ * cs + cout] = scale[:cout]
                sh[p_ * cs: p_ * cs + cout] = shift[:cout]
            phase_taps, cout, scale, shift = f_taps, osx * cs, sc, sh
    elif fold:
        raise ValueError(f"{name}: phase folding needs an up-sampling op whose only output is out0")
    if res is not None and pair and cout <= 64:
        # Siamese-pair ops with a residual: a 64-channel chunk of both streams (2 x 23 KB per stage) leaves no room for the
        # residual ring beside resident 64 -> 64 weights (74 KB) -- the op fell back to per-thread residual loads and ran at
        # 0.39 of the HBM roof (SNUNet conv1_0.conv2: 354 -> 298 us).  32-channel chunks halve the stage; the MMAs per chunk
        # stay >= 18.  Wider layers stream their weights and lose with thinner chunks (conv2_0.conv2: 160 -> 248 us), so they keep 64.
        max_kc = min(max_kc, 32)
    xf_cs = 0
    if osy == 1 and osx == 1 and not out0_s2d and not fold_cs and act_kind in (0, 1) and not act_pre and not split:
        xf = xf_taps(name, segs, phase_taps, cout, pair, hg, wg)
        if xf is not None:
            xf_phase_taps, xf_cs = xf
    if xf_cs:
        wbits, kc, n_tile, cout_pad, phases, chunks, taps, srcs, sy, sx, ey, ex = _taps_to_gemm(
            prog, name, segs, xf_phase_taps, 3 * xf_cs, pair, max_kc, force_n_tile=3 * xf_cs)
    else:
        # a folded op keeps its column blocks in ONE N tile (the store pairs blocks of the same CTA)
        wbits, kc, n_tile, cout_pad, phases, chunks, taps, srcs, sy, sx, ey, ex = _taps_to_gemm(
            prog, name, segs, phase_taps, cout, pair, max_kc, force_n_tile=cout if fold_cs else 0)
    spec = ConvSpec(
        name=name, srcs=srcs, src_sy=sy, src_sx=sx, src_ey=ey, src_ex=ex, hg=hg, wg=wg, img_mult=img_mult, pair=pair,
        weights=wbits, kc=kc, n_tile=n_tile, cout=cout, cout_pad=cout_pad, phases=phases, chunks=chunks, taps=taps,
        osy=osy, osx=osx, scale=_pad_vec(scale, cout_pad, 1.0), shift=_pad_vec(shift, cout_pad, 0.0),
        scale2=None if scale2 is None else _pad_vec(scale2, cout_pad, 1.0),
        shift2=None if shift2 is None else _pad_vec(shift2, cout_pad, 0.0),
        relu=relu, res=res, out0=out0, out0_coff=out0_coff, out_raw=out_raw, out_pool=out_pool,
        out_diff=out_diff, out_ext=out_ext, macs_per_pair=macs_per_pair, out0_s2d=out0_s2d,
        fold_cs=fold_cs, fold_cout=fold_cout, act_kind=act_kind, act_alpha=float(act_alpha), act_pre=act_pre,
        xf_cs=xf_cs, split=split,
    )
    prog.ops.append(spec)
    return spec


def _k_program_len(prog: Program, name: str, segs: Sequence[Segment], taps, cout: int, pair: bool, max_kc: int,
                   res: bool) -> Tuple[int, int]:
    """(chunks, weight blocks) of ONE phase's K-program as ``_taps_to_gemm`` would build it (``taps``: that phase's SegTaps),
    with the chunk width ``add_conv`` picks for an op with (``res``) or without a residual."""
    if res and pair and cout <= 64:
        max_kc = min(max_kc, 32)
    stored_c = [(prog.tensors[s.tensor].c - s.c_off) if s.c_store < 0 else s.c_store for s in segs]
    per_seg = _split_taps(name, segs, taps)
    kc = choose_kc(stored_c, max(1, max((len(t) for t in per_seg), default=1)), cap=max_kc if max_kc < 64 else 112)
    n_chunks = n_blocks = 0
    for s, sc, t in zip(segs, stored_c, per_seg):
        if not t:
            continue
        k_blocks = sum(1 for c0 in range(0, sc, kc) if c0 < s.c_real)
        n_chunks += k_blocks * (1 if s.sy == 1 and s.sx == 1 else len(t))
        n_blocks += k_blocks * len(t)
    return n_chunks, n_blocks


def _k_partition(prog: Program, name: str, segs: Sequence[Segment], phase_taps, cout: int, pair: bool, max_kc: int) -> List[range]:
    """Split programs only: the segment ranges of the fewest launches whose K-programs fit the kernel's per-phase tables
    (MAX_CHUNKS / MAX_TAPS).  The split form triples every K-program, so a few ops that fit in bf16 (the 7x7 stride-4 patch
    embedding, 8x8 stride-8 spatial reduction) outgrow them.  Cuts fall on segment boundaries; the last launch reads the partial
    sum as its residual, so it is sized with the residual's chunk width.  One range = no partitioning."""
    whole = range(len(segs))
    if len(phase_taps) != 1:
        return [whole]
    taps = _split_taps(name, segs, phase_taps[0][2])

    def fits(lo: int, hi: int, res: bool) -> bool:
        n_c, n_b = _k_program_len(prog, name, segs[lo:hi], SegTaps(taps[lo:hi]), cout, pair, max_kc, res)
        return n_c <= MAX_CHUNKS and n_b <= MAX_TAPS

    if fits(0, len(segs), False):
        return [whole]
    parts: List[range] = []
    hi, res = len(segs), True          # packed from the back: the last launch is the one with the residual
    while hi > 0:
        lo = hi - 1
        if not fits(lo, hi, res):
            raise ValueError(f"{name}: one K segment alone exceeds the K-program tables")
        while lo > 0 and fits(lo - 1, hi, res):
            lo -= 1
        parts.insert(0, range(lo, hi))
        hi, res = lo, False
    return parts


def _add_k_partitioned(prog: Program, name: str, segs: Sequence[Segment], phase_taps, parts: List[range], cout: int, hg: int, wg: int,
                       img_mult: int, scale: np.ndarray, shift: np.ndarray, *, pair: bool, out0: str, out0_coff: int,
                       macs_per_pair: int, act_kind: int, act_alpha: float, max_kc: int) -> ConvSpec:
    """One split conv as len(parts) launches along K: launch i < last writes acc_i*scale (+ launch i-1's partial) to the split
    intermediate ``{name}.part{i}``; the last computes acc*scale + shift + partial, then the activation, into out0.  Each
    intermediate rounds to hi + lo (16 mantissa bits), like every other split activation."""
    oy, ox, taps = phase_taps[0]
    taps = _split_taps(name, segs, taps)
    t0 = prog.tensors[out0]
    mult = 2 if pair else img_mult
    zero = np.zeros_like(np.asarray(shift, np.float32))
    prev = None
    for i, r in enumerate(parts[:-1]):
        part = prog.tensor(f"{name}.part{i}", mult, t0.h, t0.w, cout)
        _emit_conv(prog, f"{name}.part{i}", [segs[j] for j in r], [(oy, ox, SegTaps(taps[j] for j in r))], cout, hg, wg, img_mult,
                   scale, zero, pair=pair, res=prev, out0=part, split=True, max_kc=max_kc)
        prev = part
    r = parts[-1]
    return _emit_conv(prog, name, [segs[j] for j in r], [(oy, ox, SegTaps(taps[j] for j in r))], cout, hg, wg, img_mult, scale, shift,
                      pair=pair, res=prev, out0=out0, out0_coff=out0_coff, macs_per_pair=macs_per_pair, act_kind=act_kind,
                      act_alpha=act_alpha, split=True, max_kc=max_kc)


def _emit_conv(prog: Program, name: str, segs, phase_taps, cout: int, hg: int, wg: int, img_mult: int, scale: np.ndarray,
               shift: np.ndarray, *, pair: bool, res: Optional[str], out0: str, split: bool, max_kc: int, out0_coff: int = 0,
               macs_per_pair: int = 0, act_kind: int = 0, act_alpha: float = 0.0) -> ConvSpec:
    """One launch of a K-partitioned split conv (single phase, out0 store, no folding)."""
    if res is not None and pair and cout <= 64:
        max_kc = min(max_kc, 32)
    wbits, kc, n_tile, cout_pad, phases, chunks, taps, srcs, sy, sx, ey, ex = _taps_to_gemm(prog, name, segs, phase_taps, cout, pair, max_kc)
    spec = ConvSpec(
        name=name, srcs=srcs, src_sy=sy, src_sx=sx, src_ey=ey, src_ex=ex, hg=hg, wg=wg, img_mult=img_mult, pair=pair,
        weights=wbits, kc=kc, n_tile=n_tile, cout=cout, cout_pad=cout_pad, phases=phases, chunks=chunks, taps=taps,
        osy=1, osx=1, scale=_pad_vec(scale, cout_pad, 1.0), shift=_pad_vec(shift, cout_pad, 0.0),
        relu=act_kind != 0, res=res, out0=out0, out0_coff=out0_coff, macs_per_pair=macs_per_pair, act_kind=act_kind,
        act_alpha=float(act_alpha), split=split)
    prog.ops.append(spec)
    return spec


# ------------------------------------------------------------------------------------------
# SNUNet ECAM tail (models/SNUNet.py:144-149) as ONE fused op over the four level-0 node outputs


@dataclass
class EcamHeadSpec:
    """out = conv_final( ca(cat(x)) * (cat(x) + ca1(sum(x)).repeat(4)) )  for x = srcs (each C channels).

    ca / ca1 are ``ChannelAttention`` blocks (models/SNUNet.py:46-59): sigmoid(fc2(relu(fc1(avgpool)))
    + fc2(relu(fc1(maxpool)))) with bias-free 1x1 convs.  Per image the whole tail collapses to a 1x1
    conv with per-image weights W'[k, c] = Wf[k, c] * ca[c] and bias b'[k] = bf[k] + sum_c W'[k, c] *
    ca1[c % C]: pass 1 reduces avg/max per (image, channel), pass 2 applies the per-image head.
    """
    name: str
    srcs: List[str]              # 4 tensors [chunk, h, w, C]
    c: int                       # channels per source (32)
    n_class: int
    ca_fc1: np.ndarray           # float32 [r, 4C]
    ca_fc2: np.ndarray           # float32 [4C, r]
    ca1_fc1: np.ndarray          # float32 [r1, C]
    ca1_fc2: np.ndarray          # float32 [C, r1]
    w_final: np.ndarray          # float32 [n_class, 4C]
    b_final: np.ndarray          # float32 [n_class]
    out_ext: int = 0
    macs_per_pair: int = 0
    split: bool = False          # split precision: each source holds (hi, lo) planes, read as hi + lo


# ------------------------------------------------------------------------------------------
# algorithmic HBM bytes (bench.py's roofline): every source read once + every output written once at its storage dtype


def op_bytes_per_pair(prog: Program, op) -> int:
    """Algorithmic bytes one image pair moves through op `op` (DESIGN.md §4: sources read once, outputs written once)."""
    T = prog.tensors
    if isinstance(op, InputPackSpec):
        t = T[op.dst]
        in_b = 1 if op.u8_norm is not None else 4
        return 2 * (op.cin * prog.h * prog.w * in_b + t.h * t.w * t.c * 2)
    if isinstance(op, MaxPoolS2DSpec):
        t = T[op.dst]
        return 2 * (4 * op.c + op.c) * t.h * t.w * 2 * (2 if op.split else 1)
    if isinstance(op, SegHeadSpec):
        t = T[op.src]
        return (2 + (op.diff_src is not None)) * op.c * t.h * t.w * 2 + 3 * t.h * t.w * 4
    if isinstance(op, AbsDiffSpec):
        t = T[op.dst]
        return (3 + (op.add is not None)) * op.c * t.h * t.w * 2 * (2 if op.split else 1)
    if isinstance(op, ChannelGateSpec):
        t = T[op.src]
        return t.mult * op.c * t.h * t.w * 2 * (3 + (op.mode == 1) + (op.res is not None) + (op.dst_s2d is not None)) * (2 if op.split else 1)
    if isinstance(op, SumSpec):
        t = T[op.dst]
        return t.mult * t.c * t.h * t.w * 2 * (len(op.srcs) + 1)
    if isinstance(op, ChannelAttentionSpec):
        t = T[op.dst]
        return t.c * t.h * t.w * 2 * 3                      # every segment read twice, the concat written once
    if isinstance(op, SpatialGateSpec):
        t = T[op.src]
        return t.mult * (op.c * t.h * t.w * 2 * 3 + t.h * t.w * 8 * 2)
    if isinstance(op, (GlobalLocalGateSpec, CsamGateSpec)):
        t = T[op.src]
        return t.mult * (op.c * t.h * t.w * 2 * 4 + t.h * t.w * 8 * 2)
    if isinstance(op, VffmSpec):
        t = T[op.low]
        return t.mult * op.c * t.h * t.w * 2 * 5
    if isinstance(op, BitTransformerSpec):
        t = T[op.src]
        return t.mult * op.c * t.h * t.w * 2 * 3 * (2 if op.split else 1)      # tokenizer read + decoder read + write
    if isinstance(op, EcamHeadSpec):
        t = T[op.srcs[0]]
        return 2 * 4 * op.c * t.h * t.w * 2 + op.n_class * t.h * t.w * 4
    if isinstance(op, GraphConvSpec):
        t = T[op.src]
        return t.mult * (2 * op.c * t.h * t.w * 2 + (0 if op.relpos is None else op.relpos.size * 4))
    if isinstance(op, LayerNormSpec):
        t = T[op.src]
        return t.mult * op.c * t.h * t.w * 2 * (2 if op.dst_s2d is None else 3) * (2 if op.split else 1)
    if isinstance(op, DWConvSpec):
        t = T[op.src]
        return t.mult * op.c * t.h * t.w * 2 * 2 * (2 if op.split else 1)
    if isinstance(op, AttentionSpec):
        tq, tk = T[op.q], T[op.kv]
        return tq.mult * (2 * op.c * tq.h * tq.w * 2 + 2 * op.c * tk.h * tk.w * 2) * (2 if op.split else 1)
    if isinstance(op, BilinearUpSpec):
        t = T[op.dst]
        return t.mult * (op.c * t.h * t.w * 2 + op.c * t.h * t.w * 2 // (op.scale * op.scale)) * (2 if op.split else 1)
    if isinstance(op, ConvSpec):
        imgs = 2 if op.pair else op.img_mult
        seen, byt = set(), 0
        for ck in op.chunks:
            key = (ck.src, ck.stream, ck.c0)
            if key in seen:
                continue
            seen.add(key)
            t = T[op.srcs[ck.src]]
            byt += t.h * t.w * min(op.kc, t.c - ck.c0) * 2 * imgs
        ho, wo = op.hg * op.osy, op.wg * op.osx
        cout = op.fold_cout if op.fold_cs else op.cout
        for o, f in ((op.out0, 1.0), (op.out_raw, 1.0), (op.res, 1.0), (op.out_pool, 0.25), (op.out_diff, 0.5 if op.pair else 1.0)):
            if o:
                byt += int(ho * wo * cout * 2 * imgs * f)
        if op.out_ext >= 0:
            byt += ho * wo * cout * 4 * imgs
        return byt
    return 0
