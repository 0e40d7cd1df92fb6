"""ChangeFormerV6 (MiT-style Siamese transformer encoder + multi-scale difference decoder) behind ``net_G(x1, x2)``.

Drop-in for ``models/ChangeFormer.py::ChangeFormerV6`` (registry key ``ChangeFormerV6``, models/networks.py:190-191):
same constructor arguments, the reference's parameter names (``Tenc_x2.block1.0.attn.q.weight`` ...
``TDec_x2.linear_c4.proj.weight`` ...: a reference ``state_dict`` loads), same return value: a list of five tensors
with the full-resolution logits last.  Eval mode (Dropout / DropPath are identities).

Lowering (both temporal images ride through every encoder launch):

* tokens ``[B, N, C]`` are pixels ``[B, H, W, C]``: every ``nn.Linear`` is a 1x1 conv of the implicit-GEMM kernel with the
  bias, GELU and the residual add in its epilogue;
* OverlapPatchEmbed (ChangeFormer.py:195-236): the 7x7 stride-4 conv on the image reads strided TMA boxes (one per tap),
  the 7x7 stride-2 convs read the previous stage's output stored space-to-depth (4x4 taps over parity classes);
* LayerNorm is one bandwidth kernel (fp32 statistics), optionally writing the space-to-depth copy as well;
* spatial-reduction attention (:298-358): ``sr`` is a stride-``sr`` conv (strided boxes), ``kv`` a 1x1 conv on the 64
  reduced tokens, and ``softmax(q k^T / sqrt(d)) v`` one kernel that keeps the 64 keys/values of a head in shared memory
  (the score matrix never exists in HBM);
* ``Mlp`` (:260-295): fc1 -> depth-wise 3x3 + bias + GELU (one bandwidth kernel) -> fc2 + residual;
* the decoder is ChangeGNNV1's (``changevig.lower_diff_decoder``).
"""
from __future__ import annotations

from typing import Dict, List

import numpy as np
import torch
import torch.nn as nn

from . import lowering as L
from .changevig import (_ConvLayer, _DecoderV1, _MLP, _ResidualBlock, _UpsampleConvLayer, lower_decoder_tail,
                        lower_diff_decoder)
from .module import PlannedModule

_DIMS = (64, 128, 320, 512)
_DEPTHS = (3, 3, 4, 3)
_HEADS = (1, 2, 4, 8)
_SRS = (8, 4, 2, 1)


class _OverlapPatchEmbed(nn.Module):
    def __init__(self, k: int, stride: int, cin: int, cout: int):
        super().__init__()
        self.proj = nn.Conv2d(cin, cout, kernel_size=k, stride=stride, padding=k // 2)
        self.norm = nn.LayerNorm(cout)


class _Attention(nn.Module):
    def __init__(self, dim: int, sr: int):
        super().__init__()
        self.q = nn.Linear(dim, dim, bias=True)
        self.kv = nn.Linear(dim, dim * 2, bias=True)
        self.proj = nn.Linear(dim, dim)
        if sr > 1:
            self.sr = nn.Conv2d(dim, dim, kernel_size=sr, stride=sr)
            self.norm = nn.LayerNorm(dim)


class _DWConv(nn.Module):
    def __init__(self, dim: int):
        super().__init__()
        self.dwconv = nn.Conv2d(dim, dim, 3, 1, 1, bias=True, groups=dim)


class _Mlp(nn.Module):
    def __init__(self, dim: int):
        super().__init__()
        self.fc1 = nn.Linear(dim, 4 * dim)
        self.dwconv = _DWConv(4 * dim)
        self.fc2 = nn.Linear(4 * dim, dim)


class _Block(nn.Module):
    def __init__(self, dim: int, sr: int):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.attn = _Attention(dim, sr)
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.mlp = _Mlp(dim)


class _EncoderTransformerV3(nn.Module):
    """models/ChangeFormer.py:1340-1432 (parameters only)."""

    def __init__(self, in_chans: int, depths=_DEPTHS, patch_k: int = 7, intra_patch: bool = False):
        super().__init__()
        self.patch_embed1 = _OverlapPatchEmbed(7, 4, in_chans, _DIMS[0])
        self.patch_embed2 = _OverlapPatchEmbed(patch_k, 2, _DIMS[0], _DIMS[1])
        self.patch_embed3 = _OverlapPatchEmbed(patch_k, 2, _DIMS[1], _DIMS[2])
        self.patch_embed4 = _OverlapPatchEmbed(patch_k, 2, _DIMS[2], _DIMS[3])
        for s in range(4):
            setattr(self, f"block{s + 1}", nn.ModuleList([_Block(_DIMS[s], _SRS[s]) for _ in range(depths[s])]))
            setattr(self, f"norm{s + 1}", nn.LayerNorm(_DIMS[s], eps=1e-6))
            if intra_patch and s < 3:
                # EncoderTransformer's "intra-patch encoder" blocks (ChangeFormer.py:51-58, 66-73, 81-88): constructed, never
                # called by forward_features (:141-185) -- parameters only
                setattr(self, f"patch_block{s + 1}", nn.ModuleList([_Block(_DIMS[s + 1], _SRS[s])]))
                setattr(self, f"pnorm{s + 1}", nn.LayerNorm(_DIMS[s + 1], eps=1e-6))


class ChangeFormerV6(PlannedModule):
    """models/ChangeFormer.py:1669-1701."""
    default_chunk_pairs = 32
    supports_precision_path = True

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False, embed_dim: int = 256):
        super().__init__()
        if decoder_softmax:
            raise NotImplementedError("stcd_b200.ChangeFormerV6 serves decoder_softmax=False (networks.py:191)")
        if input_nc > 8 or output_nc > 8 or embed_dim % 16:
            raise NotImplementedError("input_nc, output_nc <= 8 and embed_dim a multiple of 16")
        self.input_nc, self.output_nc = input_nc, output_nc
        self.embed_dims = list(_DIMS)
        self.depths = list(_DEPTHS)
        self.embedding_dim = embed_dim
        self.Tenc_x2 = _EncoderTransformerV3(input_nc)
        self.TDec_x2 = _DecoderV1(_DIMS, embed_dim, output_nc, head="linear_c")
        for m in self.Tenc_x2.modules():                    # EncoderTransformer_v3._init_weights, :1404-1418
            if isinstance(m, nn.Linear):
                nn.init.trunc_normal_(m.weight, std=.02)
                nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.Conv2d):
                fan_out = m.kernel_size[0] * m.kernel_size[1] * m.out_channels // m.groups
                m.weight.data.normal_(0, (2.0 / fan_out) ** 0.5)
                m.bias.data.zero_()

    def lower(self, h: int, w: int) -> L.Program:
        return lower_changeformer(self.state_dict(), self.input_nc, self.embedding_dim, self.output_nc, h, w, precision=self.plan_precision)

    @torch.no_grad()
    def forward(self, x1: torch.Tensor, x2: torch.Tensor):
        return self.plan_for(x1).forward(x1, x2)        # list of 5, full-resolution logits last

    def _wrap_outputs(self, outs):
        return list(outs)


# ------------------------------------------------------------------------------------------
def lower_changeformer(sd: Dict[str, torch.Tensor], in_ch: int, e: int, n_class: int, h: int, w: int, precision: str = "bf16") -> L.Program:
    """state_dict of the reference ChangeFormerV6 -> fused-op Program (eval mode).  precision "split": every op carries (hi, lo)
    bf16 planes (lowering.Program.precision); the split K-programs that outgrow the conv kernel's tables are cut along K."""
    if h % 256 or w % 256:
        # stage 1 reduces its keys by sr = 8 at 1/4 scale, ..., and every stage must leave an integer, even token grid
        raise ValueError(f"ChangeFormerV6 lowering needs H and W divisible by 256 (got {h}x{w}); the reference is built for 256")
    if (h // 32) * (w // 32) > 64:
        raise ValueError("the attention kernel keeps at most 64 reduced tokens per image (256x256 inputs, the reference's img_size)")
    sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
    p = L.Program(model="ChangeFormerV6", in_channels=in_ch, h=h, w=w, precision=precision)
    feats = lower_mit_encoder(p, sd, "Tenc_x2", in_ch, _DEPTHS, h, w)
    lower_diff_decoder(p, sd, feats, e, n_class, "TDec_x2", "TDec_x2.linear_c{k}")
    return p


def lower_mit_encoder(p: L.Program, sd: Dict[str, torch.Tensor], enc: str, in_ch: int, depths, h: int, w: int):
    """EncoderTransformer (ChangeFormer.py:23-193; patch embeds 7/s4 then 3/s2) == EncoderTransformer_v3 (:1342-1472; 7/s4 then 7/s2):
    the patch size is read off the weights.  Returns [(tensor, channels, h, w)] per stage, both streams."""
    ones = lambda c: np.ones(c, np.float32)  # noqa: E731
    npf = lambda t: t.numpy().astype(np.float32)  # noqa: E731

    def linear(name: str, pre: str, src: str, cin: int, cout: int, hh: int, ww: int, **kw) -> None:
        wt = sd[f"{pre}.weight"][:, :, None, None]
        L.add_conv(p, name, [L.Segment(src, cin)], L.conv_taps(wt, pad=0), cout, hh, ww, 1, ones(cout), npf(sd[f"{pre}.bias"]),
                   pair=True, macs_per_pair=2 * hh * ww * cin * cout, **kw)

    def layernorm(name: str, pre: str, src: str, dst: str, c: int, eps: float, dst_s2d=None) -> None:
        p.ops.append(L.LayerNormSpec(name, src, dst, c, npf(sd[f"{pre}.weight"]), npf(sd[f"{pre}.bias"]), eps, dst_s2d, split=p.split))

    p.tensor("in", 2, h, w, 8)
    p.ops.append(L.InputPackSpec("pack", "in", in_ch, split=p.split))
    feats = []
    x_s2d = None
    hh, ww = h, w
    for s in range(4):
        c, heads, sr = _DIMS[s], _HEADS[s], _SRS[s]
        pe = f"{enc}.patch_embed{s + 1}"
        wt = sd[f"{pe}.proj.weight"]
        if s == 0:
            hh, ww = hh // 4, ww // 4
            t = p.tensor(f"{pe}.conv", 2, hh, ww, c)
            L.add_conv(p, f"{pe}.proj", [L.Segment("in", in_ch, sy=4, sx=4)], L.conv_taps(wt, pad=3), c, hh, ww, 1, ones(c),
                       npf(sd[f"{pe}.proj.bias"]), pair=True, out0=t, macs_per_pair=2 * hh * ww * 49 * in_ch * c)
        else:
            cprev = _DIMS[s - 1]
            hh, ww = hh // 2, ww // 2
            t = p.tensor(f"{pe}.conv", 2, hh, ww, c)
            kk = wt.shape[2]
            L.add_conv(p, f"{pe}.proj", L.s2d_segments(x_s2d, cprev), [(0, 0, L.s2d_conv_taps(wt, pad=kk // 2))], c, hh, ww, 1, ones(c),
                       npf(sd[f"{pe}.proj.bias"]), pair=True, out0=t, macs_per_pair=2 * hh * ww * kk * kk * cprev * c)
        x = p.tensor(f"{pe}.out", 2, hh, ww, c)
        layernorm(f"{pe}.norm", f"{pe}.norm", t, x, c, 1e-5)
        for i in range(depths[s]):
            blk = f"{enc}.block{s + 1}.{i}"
            a = f"{blk}.attn"
            n1 = p.tensor(f"{blk}.n1", 2, hh, ww, c)
            layernorm(f"{blk}.norm1", f"{blk}.norm1", x, n1, c, 1e-6)
            q = p.tensor(f"{a}.q", 2, hh, ww, c)
            linear(f"{a}.q", f"{a}.q", n1, c, c, hh, ww, out0=q)
            if sr > 1:
                hk, wk = hh // sr, ww // sr
                srt = p.tensor(f"{a}.sr", 2, hk, wk, c)
                L.add_conv(p, f"{a}.sr", [L.Segment(n1, c, sy=sr, sx=sr)], L.conv_taps(sd[f"{a}.sr.weight"], pad=0), c, hk, wk, 1,
                           ones(c), npf(sd[f"{a}.sr.bias"]), pair=True, out0=srt, macs_per_pair=2 * hk * wk * sr * sr * c * c)
                kin = p.tensor(f"{a}.srn", 2, hk, wk, c)
                layernorm(f"{a}.norm", f"{a}.norm", srt, kin, c, 1e-5)
            else:
                hk, wk, kin = hh, ww, n1
            kv = p.tensor(f"{a}.kv", 2, hk, wk, 2 * c)
            linear(f"{a}.kv", f"{a}.kv", kin, c, 2 * c, hk, wk, out0=kv)
            ao = p.tensor(f"{a}.o", 2, hh, ww, c)
            d = c // heads
            p.ops.append(L.AttentionSpec(f"{a}.softmax", q, kv, ao, c, heads, float(d ** -0.5),
                                         macs_per_pair=2 * 2 * hh * ww * hk * wk * c, split=p.split))
            x1 = p.tensor(f"{blk}.x1", 2, hh, ww, c)
            linear(f"{a}.proj", f"{a}.proj", ao, c, c, hh, ww, res=x, out0=x1)
            n2 = p.tensor(f"{blk}.n2", 2, hh, ww, c)
            layernorm(f"{blk}.norm2", f"{blk}.norm2", x1, n2, c, 1e-6)
            m = f"{blk}.mlp"
            h1 = p.tensor(f"{m}.h1", 2, hh, ww, 4 * c)
            linear(f"{m}.fc1", f"{m}.fc1", n2, c, 4 * c, hh, ww, out0=h1)
            h2 = p.tensor(f"{m}.h2", 2, hh, ww, 4 * c)
            p.ops.append(L.DWConvSpec(f"{m}.dwconv", h1, h2, 4 * c, npf(sd[f"{m}.dwconv.dwconv.weight"].reshape(4 * c, 9)),
                                      npf(sd[f"{m}.dwconv.dwconv.bias"]), gelu=True, macs_per_pair=2 * hh * ww * 9 * 4 * c,
                                      split=p.split))
            x = p.tensor(f"{blk}.out", 2, hh, ww, c)
            linear(f"{m}.fc2", f"{m}.fc2", h2, 4 * c, c, hh, ww, res=x1, out0=x)
        f = p.tensor(f"{enc}.f{s + 1}", 2, hh, ww, c)
        x_s2d = p.tensor(f"{enc}.f{s + 1}_s2d", 2, hh // 2, ww // 2, 4 * c) if s < 3 else None
        layernorm(f"{enc}.norm{s + 1}", f"{enc}.norm{s + 1}", x, f, c, 1e-6, dst_s2d=x_s2d)
        feats.append((f, c, hh, ww))
    return feats


# ==========================================================================================
# ChangeFormerV1 / V2 (models/ChangeFormer.py:644-674, 918-948): Tenc = EncoderTransformer (patch 7/s4 then 3/s2, depths 3-4-6-3) on
# both dates, |fx1 - fx2| per scale, convprojection_base (V1) or TDec (V2).  Both return ONE tensor.
_DEPTHS_TENC = (3, 4, 6, 3)


def _init_mit(enc: nn.Module) -> None:
    """EncoderTransformer._init_weights, ChangeFormer.py:99-112."""
    for m in enc.modules():
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=.02)
            nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.Conv2d):
            fan_out = m.kernel_size[0] * m.kernel_size[1] * m.out_channels // m.groups
            m.weight.data.normal_(0, (2.0 / fan_out) ** 0.5)
            m.bias.data.zero_()


class _ConvProjectionBase(nn.Module):
    """models/ChangeFormer.py:591-603."""

    def __init__(self):
        super().__init__()
        self.convd16x = _UpsampleConvLayer(512, 320, 4, 2)
        self.dense_4 = nn.Sequential(_ResidualBlock(320))
        self.convd8x = _UpsampleConvLayer(320, 128, 4, 2)
        self.dense_3 = nn.Sequential(_ResidualBlock(128))
        self.convd4x = _UpsampleConvLayer(128, 64, 4, 2)
        self.dense_2 = nn.Sequential(_ResidualBlock(64))
        self.convd2x = _UpsampleConvLayer(64, 16, 4, 2)
        self.dense_1 = nn.Sequential(_ResidualBlock(16))
        self.convd1x = _UpsampleConvLayer(16, 8, 4, 2)


class _TDec(nn.Module):
    """models/ChangeFormer.py:691-735."""

    def __init__(self, in_channels, e: int, output_nc: int):
        super().__init__()
        c1, c2, c3, c4 = in_channels
        self.linear_c4 = _MLP(c4, e)
        self.linear_c3 = _MLP(c3, e)
        self.linear_c2 = _MLP(c2, e)
        self.linear_c1 = _MLP(c1, e)
        self.linear_fuse = nn.Conv2d(e * 4, e, 1)
        self.convd2x = _UpsampleConvLayer(e, e, 4, 2)
        self.dense_2x = nn.Sequential(_ResidualBlock(e))
        self.convd1x = _UpsampleConvLayer(e, e, 4, 2)
        self.dense_1x = nn.Sequential(_ResidualBlock(e))
        self.change_probability = _ConvLayer(e, output_nc, 3, 1, 1)
        self.active = nn.Softmax(dim=1)


class _ChangeFormerTenc(PlannedModule):
    default_chunk_pairs = 32
    _variant = ""

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False):
        super().__init__()
        if decoder_softmax:
            raise NotImplementedError("stcd_b200 serves decoder_softmax=False (models/networks.py:184-187)")
        if input_nc != 3 or output_nc > 8:
            raise NotImplementedError("Tenc is built for 3 input channels upstream (ChangeFormer.py:525-531); output_nc <= 8")
        self.output_nc = output_nc
        self.Tenc = _EncoderTransformerV3(3, depths=_DEPTHS_TENC, patch_k=3, intra_patch=True)
        _init_mit(self.Tenc)

    def lower(self, h: int, w: int) -> L.Program:
        return lower_changeformer_tenc(self.state_dict(), self._variant, self.output_nc, h, w)

    @torch.no_grad()
    def forward(self, x1: torch.Tensor, x2: torch.Tensor) -> torch.Tensor:
        return self.plan_for(x1).forward(x1, x2)[0]


class ChangeFormerV1(_ChangeFormerTenc):
    """models/ChangeFormer.py:644-674."""
    _variant = "v1"

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False):
        super().__init__(input_nc, output_nc, decoder_softmax)
        self.convproj = _ConvProjectionBase()
        self.change_probability = _ConvLayer(8, output_nc, 3, 1, 1)
        self.active = nn.Softmax(dim=1)


class ChangeFormerV2(_ChangeFormerTenc):
    """models/ChangeFormer.py:918-948."""
    _variant = "v2"

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False):
        super().__init__(input_nc, output_nc, decoder_softmax)
        self.TDec = _TDec(_DIMS, 32, output_nc)
        self.output_activation = nn.Softmax(dim=1)


class _TDecV2(nn.Module):
    """models/ChangeFormer.py:793-830."""

    def __init__(self, in_channels, e: int, output_nc: int):
        super().__init__()
        c1, c2, c3, c4 = in_channels
        self.linear_c4 = _MLP(c4, e)
        self.linear_c3 = _MLP(c3, e)
        self.linear_c2 = _MLP(c2, e)
        self.linear_c1 = _MLP(c1, e)
        self.linear_fuse = nn.Conv2d(e * 4, e, 1)
        self.pix_shuffle_conv = nn.Conv2d(e, 16 * output_nc, 3, stride=1, padding=1)
        self.pix_shuffle = nn.PixelShuffle(4)
        self.active = nn.Softmax(dim=1)


class ChangeFormerV3(_ChangeFormerTenc):
    """models/ChangeFormer.py:951-973."""
    _variant = "v3"

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False):
        super().__init__(input_nc, output_nc, decoder_softmax)
        self.TDec = _TDecV2(_DIMS, 64, output_nc)


def lower_changeformer_tenc(sd: Dict[str, torch.Tensor], variant: str, n_class: int, h: int, w: int) -> L.Program:
    """state_dict of the reference ChangeFormerV1 / V2 -> fused-op Program (eval mode)."""
    if h % 256 or w % 256 or (h // 32) * (w // 32) > 64:
        raise ValueError(f"ChangeFormer{variant.upper()} lowering serves 256x256 inputs (the reference's img_size; 64 reduced tokens per image), got {h}x{w}")
    sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
    p = L.Program(model=f"ChangeFormer{variant.upper()}", in_channels=3, h=h, w=w)
    ones = lambda c: np.ones(c, np.float32)  # noqa: E731
    npf = lambda t: np.ascontiguousarray(t.numpy().astype(np.float32))  # noqa: E731
    feats = lower_mit_encoder(p, sd, "Tenc", 3, _DEPTHS_TENC, h, w)
    if variant == "v3":                                         # TDecV2.forward, :867-915
        d, e = "TDec", 64
        _, _, fh, fw = feats[0]
        diffs = []
        for k in (4, 3, 2, 1):
            ft, c, hh, ww = feats[k - 1]
            y = p.tensor(f"{d}.linear_c{k}.o", 2, hh, ww, e)
            L.add_conv(p, f"{d}.linear_c{k}", [L.Segment(ft, c)], L.conv_taps(sd[f"{d}.linear_c{k}.proj.weight"][:, :, None, None], pad=0), e, hh,
                       ww, 1, ones(e), npf(sd[f"{d}.linear_c{k}.proj.bias"]), pair=True, out0=y, macs_per_pair=2 * hh * ww * c * e)
            if k > 1:
                u = p.tensor(f"{d}.linear_c{k}.up", 2, fh, fw, e)
                p.ops.append(L.BilinearUpSpec(f"{d}.linear_c{k}.up", y, u, e, fh // hh))
                y = u
            dk = p.tensor(f"{d}.diff{k}", 1, fh, fw, e)
            p.ops.append(L.AbsDiffSpec(f"{d}.diff{k}", y, dk, e))
            diffs.append(dk)
        fused = p.tensor(f"{d}.fused", 1, fh, fw, e)
        L.add_conv(p, f"{d}.linear_fuse", [L.Segment(t, e) for t in diffs], L.conv_taps(sd[f"{d}.linear_fuse.weight"], pad=0), e, fh, fw, 1,
                   ones(e), npf(sd[f"{d}.linear_fuse.bias"]), out0=fused, macs_per_pair=fh * fw * 4 * e * e)
        # relu(conv3x3 -> 16 * n_class) + PixelShuffle(4): output pixel (4y + i, 4x + j) of class c is conv channel c*16 + i*4 + j at
        # (y, x) -- an up-sampling conv with 16 output phases.  The phases have different biases while a launch shares one
        # per-channel affine, so every phase is its own (small) launch writing its pixels of the fp32 output.
        wps, bps = sd[f"{d}.pix_shuffle_conv.weight"], sd[f"{d}.pix_shuffle_conv.bias"]
        for i in range(4):
            for j in range(4):
                rows = [cc * 16 + i * 4 + j for cc in range(n_class)]
                L.add_conv(p, f"{d}.pix_shuffle_conv.{i}{j}", [L.Segment(fused, e)], [(i, j, L.conv_taps(wps[rows], pad=1)[0][2])], n_class,
                           fh, fw, 1, ones(n_class), npf(bps[rows]), relu=True, osy=4, osx=4, out_ext=0,
                           macs_per_pair=fh * fw * 9 * e * n_class)
        p.ext.append(L.ExtOutput("cp", n_class, 4 * fh, 4 * fw))
        return p
    di = []                                                     # DI[i] = |fx1[i] - fx2[i]| (:664-666, 938-940)
    for i, (ft, c, hh, ww) in enumerate(feats):
        t = p.tensor(f"DI{i}", 1, hh, ww, c)
        p.ops.append(L.AbsDiffSpec(f"DI{i}", ft, t, c))
        di.append((t, c, hh, ww))

    def up(q: str, x: str, cin: int, cout: int, hh: int, ww: int) -> str:
        cp = (cout + 7) // 8 * 8
        o = p.tensor(f"{q}.o", 1, 2 * hh, 2 * ww, cp)
        L.add_conv(p, q, [L.Segment(x, cin)], L.convT_phase_taps(sd[f"{q}.conv2d.weight"], stride=2, pad=1), cout, hh, ww, 1, ones(cout),
                   npf(sd[f"{q}.conv2d.bias"]), osy=2, osx=2, out0=o, macs_per_pair=hh * ww * 16 * cin * cout)
        return o

    def resblock(q: str, u: str, c: int, hh: int, ww: int, extra: str = None) -> str:
        """ResidualBlock (conv, ReLU, conv * 0.1 + u) [+ extra]: the second residual is pre-added to u by one bandwidth op."""
        cp = (c + 7) // 8 * 8
        r1 = p.tensor(f"{q}.t", 1, hh, ww, cp)
        L.add_conv(p, f"{q}.conv1", [L.Segment(u, c)], L.conv_taps(sd[f"{q}.conv1.conv2d.weight"], pad=1), c, hh, ww, 1, ones(c),
                   npf(sd[f"{q}.conv1.conv2d.bias"]), relu=True, out0=r1, macs_per_pair=hh * ww * 9 * c * c)
        res = u
        if extra is not None:
            res = p.tensor(f"{q}.res", 1, hh, ww, cp)
            p.ops.append(L.SumSpec(f"{q}.res", [u, extra], res))
        o = p.tensor(f"{q}.out", 1, hh, ww, cp)
        L.add_conv(p, f"{q}.conv2", [L.Segment(r1, c)], L.conv_taps(sd[f"{q}.conv2.conv2d.weight"], pad=1), c, hh, ww, 1, 0.1 * ones(c),
                   0.1 * npf(sd[f"{q}.conv2.conv2d.bias"]), res=res, out0=o, macs_per_pair=hh * ww * 9 * c * c)
        return o

    if variant == "v1":                                         # convprojection_base.forward, :605-641
        c = "convproj"
        t4, _, hh, ww = di[3]
        x = up(f"{c}.convd16x", t4, 512, 320, hh, ww)
        x = resblock(f"{c}.dense_4.0", x, 320, 2 * hh, 2 * ww, extra=di[2][0])
        x = up(f"{c}.convd8x", x, 320, 128, 2 * hh, 2 * ww)
        x = resblock(f"{c}.dense_3.0", x, 128, 4 * hh, 4 * ww, extra=di[1][0])
        x = up(f"{c}.convd4x", x, 128, 64, 4 * hh, 4 * ww)
        x = resblock(f"{c}.dense_2.0", x, 64, 8 * hh, 8 * ww, extra=di[0][0])
        x = up(f"{c}.convd2x", x, 64, 16, 8 * hh, 8 * ww)
        x = resblock(f"{c}.dense_1.0", x, 16, 16 * hh, 16 * ww)
        x = up(f"{c}.convd1x", x, 16, 8, 16 * hh, 16 * ww)
        hh, ww = 32 * hh, 32 * ww
        L.add_conv(p, "change_probability", [L.Segment(x, 8)], L.conv_taps(sd["change_probability.conv2d.weight"], pad=1), n_class, hh, ww, 1,
                   ones(n_class), npf(sd["change_probability.conv2d.bias"]), out_ext=0, macs_per_pair=hh * ww * 9 * 8 * n_class)
        p.ext.append(L.ExtOutput("cp", n_class, hh, ww))
        return p
    # ---- V2: TDec.forward, :762-790
    d, e = "TDec", 32
    _, _, fh, fw = di[0]
    ups = []
    for k in (4, 3, 2, 1):
        t, c, hh, ww = di[k - 1]
        y = p.tensor(f"{d}.linear_c{k}.o", 1, hh, ww, e)
        L.add_conv(p, f"{d}.linear_c{k}", [L.Segment(t, c)], L.conv_taps(sd[f"{d}.linear_c{k}.proj.weight"][:, :, None, None], pad=0), e, hh, ww, 1,
                   ones(e), npf(sd[f"{d}.linear_c{k}.proj.bias"]), out0=y, macs_per_pair=hh * ww * c * e)
        if k > 1:
            u = p.tensor(f"{d}.linear_c{k}.up", 1, fh, fw, e)
            p.ops.append(L.BilinearUpSpec(f"{d}.linear_c{k}.up", y, u, e, fh // hh))
            y = u
        ups.append(y)
    fused = p.tensor(f"{d}.fused", 1, fh, fw, e)
    L.add_conv(p, f"{d}.linear_fuse", [L.Segment(t, e) for t in ups], L.conv_taps(sd[f"{d}.linear_fuse.weight"], pad=0), e, fh, fw, 1, ones(e),
               npf(sd[f"{d}.linear_fuse.bias"]), out0=fused, macs_per_pair=fh * fw * 4 * e * e)
    lower_decoder_tail(p, sd, fused, fh, fw, e, n_class, d, out_ext=0)
    return p
