"""BIT (bitemporal image transformer) and its ResNet-18 baseline behind the reference's ``net_G(x1, x2)`` contract.

Drop-in for ``models/networks.py::ResNet`` (:223-305, registry key ``base_resnet18``) and ``BASE_Transformer``
(:308-441, keys ``base_transformer_pos_s4``, ``..._dd8``, ``..._dd8_dedim8``, :170-182): same constructor arguments,
same parameter names and registration order (``pos_embedding``, ``resnet.layer1.0.conv1.weight`` ...,
``transformer_decoder.layers.7.0.fn.fn.to_q.weight`` ...: a reference ``state_dict`` loads, including the backbone's
unused ``layer4`` / ``fc``), same return values (``ResNet``: the logits; ``BASE_Transformer``: a one-element list).
Eval mode.  The backbone is never downloaded (``pretrained=True`` upstream): load a ``state_dict``.

Lowering:

* backbone = resnet18 with ``replace_stride_with_dilation=[False, True, True]`` whose BasicBlock resets dilation to 1
  (models/resnet.py:47-49): stride-1 layer3 (/layer4) at 1/8 scale.  Same conv lowering as SegCD's encoder
  (space-to-depth stem, parity-class stride-2 convs, residual + ReLU epilogues);
* ``upsamplex2`` (nearest) + ``conv_pred`` 3x3 is one conv with 4 output phases of merged 2x2 taps, never materialised;
* the token path is K12 (csrc/bit_kernels.cuh): the tokenizer is an online softmax over the image's pixels, the 8-token
  encoder runs in one CTA per pair, and the decoder's cross-attention is collapsed algebraically: with only L = 4 keys
  per image, ``softmax(q k^T) v W_out`` is ``softmax_groups(LN(x) A) B`` with per-image 32x32 matrices
  ``A = scale W_q^T k`` and ``B = v W_out^T`` -- 2 K MACs per pixel and layer instead of 37 K (dim_head 64), computed in
  fp32 by one kernel that keeps the pixel's 32 channels in registers through all decoder layers;
* ``|x1 - x2|``, bilinear x4, and the two classifier convs (BN folded) finish at full resolution.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch
import torch.nn as nn

from . import lowering as L
from .module import PlannedModule
from .segcd import _BasicBlock, stem_s2d_taps


class _ResNet18(nn.Module):
    """models/resnet.py:127-182 with BasicBlock [2, 2, 2, 2] and replace_stride_with_dilation=[False, True, True]
    (parameters only): layer3 / layer4 keep stride 1."""

    def __init__(self, in_channels: int = 3):
        super().__init__()
        self.conv1 = nn.Conv2d(in_channels, 64, 7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        cin = 64
        for li, (cout, stride) in enumerate(((64, 1), (128, 2), (256, 1), (512, 1))):
            setattr(self, f"layer{li + 1}", nn.Sequential(_BasicBlock(cin, cout, stride), _BasicBlock(cout, cout, 1)))
            cin = cout
        self.fc = nn.Linear(512, 1000)
        for m in self.modules():                                  # models/resnet.py:168-173
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")


class _TwoLayerConv2d(nn.Sequential):
    """models/help_funcs.py:7-16."""

    def __init__(self, in_channels: int, out_channels: int, kernel_size: int = 3):
        super().__init__(nn.Conv2d(in_channels, in_channels, kernel_size, padding=kernel_size // 2, bias=False),
                         nn.BatchNorm2d(in_channels), nn.ReLU(),
                         nn.Conv2d(in_channels, out_channels, kernel_size, padding=kernel_size // 2))


class _Wrap(nn.Module):
    """Residual / Residual2 (help_funcs.py:19-33): parameters live under ``.fn``."""

    def __init__(self, fn: nn.Module):
        super().__init__()
        self.fn = fn


class _PreNorm(nn.Module):
    """PreNorm / PreNorm2 (help_funcs.py:36-52)."""

    def __init__(self, dim: int, fn: nn.Module):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.fn = fn


class _FeedForward(nn.Module):
    """help_funcs.py:55-66."""

    def __init__(self, dim: int, hidden: int):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(dim, hidden), nn.GELU(), nn.Dropout(0.0), nn.Linear(hidden, dim), nn.Dropout(0.0))


class _Attention(nn.Module):
    """help_funcs.py:113-125."""

    def __init__(self, dim: int, heads: int, dim_head: int):
        super().__init__()
        self.to_qkv = nn.Linear(dim, dim_head * heads * 3, bias=False)
        self.to_out = nn.Sequential(nn.Linear(dim_head * heads, dim), nn.Dropout(0.0))


class _CrossAttention(nn.Module):
    """help_funcs.py:69-85."""

    def __init__(self, dim: int, heads: int, dim_head: int):
        super().__init__()
        self.to_q = nn.Linear(dim, dim_head * heads, bias=False)
        self.to_k = nn.Linear(dim, dim_head * heads, bias=False)
        self.to_v = nn.Linear(dim, dim_head * heads, bias=False)
        self.to_out = nn.Sequential(nn.Linear(dim_head * heads, dim), nn.Dropout(0.0))


class _Transformer(nn.Module):
    """help_funcs.py:151-163 / 166-182 (decoder=True)."""

    def __init__(self, dim: int, depth: int, heads: int, dim_head: int, mlp_dim: int, decoder: bool):
        super().__init__()
        att = _CrossAttention if decoder else _Attention
        self.layers = nn.ModuleList([nn.ModuleList([_Wrap(_PreNorm(dim, att(dim, heads, dim_head))),
                                                    _Wrap(_PreNorm(dim, _FeedForward(dim, mlp_dim)))]) for _ in range(depth)])


class ResNet(PlannedModule):
    """models/networks.py:223-305."""
    default_chunk_pairs = 32
    supports_precision_path = True

    def __init__(self, input_nc: int, output_nc: int, resnet_stages_num: int = 5, backbone: str = "resnet18",
                 output_sigmoid: bool = False, if_upsample_2x: bool = True):
        super().__init__()
        if backbone != "resnet18":
            raise NotImplementedError("stcd_b200 serves backbone='resnet18' (every BIT key of models/networks.py:170-182)")
        if resnet_stages_num not in (3, 4, 5):
            raise NotImplementedError                                  # like upstream, :256-257
        if output_sigmoid or not if_upsample_2x:
            raise NotImplementedError("stcd_b200 serves output_sigmoid=False, if_upsample_2x=True (the registry's settings)")
        if input_nc > 4 or output_nc > 8:
            raise NotImplementedError("input_nc <= 4, output_nc <= 8")
        self.input_nc, self.output_nc = input_nc, output_nc
        self.resnet = _ResNet18(input_nc)
        self.classifier = _TwoLayerConv2d(32, output_nc)
        self.resnet_stages_num = resnet_stages_num
        self.if_upsample_2x = if_upsample_2x
        self.conv_pred = nn.Conv2d({5: 512, 4: 256, 3: 128}[resnet_stages_num], 32, 3, padding=1)
        self.output_sigmoid = output_sigmoid

    def lower(self, h: int, w: int) -> L.Program:
        return lower_bit(self.state_dict(), self.input_nc, self.output_nc, self.resnet_stages_num, None, h, w, precision=self.plan_precision)

    @torch.no_grad()
    def forward(self, x1: torch.Tensor, x2: torch.Tensor):
        return self.plan_for(x1).forward(x1, x2)[0]


class BASE_Transformer(ResNet):
    """models/networks.py:308-441."""

    def __init__(self, input_nc: int, output_nc: int, with_pos, resnet_stages_num: int = 5, token_len: int = 4,
                 token_trans: bool = True, enc_depth: int = 1, dec_depth: int = 1, dim_head: int = 64,
                 decoder_dim_head: int = 64, tokenizer: bool = True, if_upsample_2x: bool = True, pool_mode: str = "max",
                 pool_size: int = 2, backbone: str = "resnet18", decoder_softmax: bool = True, with_decoder_pos=None,
                 with_decoder: bool = True):
        super().__init__(input_nc, output_nc, backbone=backbone, resnet_stages_num=resnet_stages_num, if_upsample_2x=if_upsample_2x)
        if with_pos != "learned" or not tokenizer or not token_trans or not with_decoder or with_decoder_pos is not None:
            raise NotImplementedError("stcd_b200 serves with_pos='learned', tokenizer=True, token_trans=True, with_decoder=True, "
                                      "with_decoder_pos=None (the registry's BIT keys, models/networks.py:174-182)")
        if token_len != 4:
            raise NotImplementedError("token_len must be 4 (heads x tokens = 32 attention scores per pixel)")
        self.token_len = token_len
        self.conv_a = nn.Conv2d(32, token_len, 1, bias=False)
        self.tokenizer, self.token_trans, self.with_decoder = tokenizer, token_trans, with_decoder
        dim, mlp_dim = 32, 64
        self.with_pos = with_pos
        self.pos_embedding = nn.Parameter(torch.randn(1, token_len * 2, 32))
        self.with_decoder_pos = with_decoder_pos
        self.enc_depth, self.dec_depth, self.dim_head, self.decoder_dim_head = enc_depth, dec_depth, dim_head, decoder_dim_head
        self.decoder_softmax = decoder_softmax
        self.transformer = _Transformer(dim, enc_depth, 8, dim_head, mlp_dim, decoder=False)
        self.transformer_decoder = _Transformer(dim, dec_depth, 8, decoder_dim_head, mlp_dim, decoder=True)

    def lower(self, h: int, w: int) -> L.Program:
        cfg = dict(token_len=self.token_len, heads=8, inner_enc=8 * self.dim_head, inner_dec=8 * self.decoder_dim_head, mlp=64,
                   n_enc=self.enc_depth, n_dec=self.dec_depth, softmax=self.decoder_softmax)
        return lower_bit(self.state_dict(), self.input_nc, self.output_nc, self.resnet_stages_num, cfg, h, w, precision=self.plan_precision)

    @torch.no_grad()
    def forward(self, x1: torch.Tensor, x2: torch.Tensor):
        return [self.plan_for(x1).forward(x1, x2)[0]]              # outputs = [x], :438-440

    def _wrap_outputs(self, outs):
        return list(outs)


# ------------------------------------------------------------------------------------------
def lower_bit(sd: Dict[str, torch.Tensor], in_channels: int, n_class: int, stages: int, cfg: Optional[dict], h: int, w: int,
              precision: str = "bf16") -> L.Program:
    """state_dict of the reference ResNet / BASE_Transformer -> fused-op Program (eval mode).  precision "split": every op carries
    (hi, lo) bf16 planes (lowering.Program.precision)."""
    if h % 16 or w % 16:
        raise ValueError(f"BIT lowering needs H and W divisible by 16 (got {h}x{w})")
    sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
    p = L.Program(model="BIT" if cfg else "BIT-ResNet18", in_channels=in_channels, h=h, w=w, precision=precision)

    def bn(prefix: str, c: int):
        return L.fold_bn(None, L.bn_params(sd, prefix), c)

    def f32(t: torch.Tensor) -> np.ndarray:
        return np.ascontiguousarray(t.numpy().astype(np.float32))

    # ---------------- stem + max-pool (forward_single, :279-282)
    hh, ww = h // 2, w // 2
    p.tensor("in", 2, hh, ww, 16)
    p.ops.append(L.InputPackSpec("pack", "in", in_channels, s2d=True, split=p.split))
    f1s = p.tensor("f1s", 2, hh // 2, ww // 2, 4 * 64)
    sc, sh = bn("resnet.bn1", 64)
    L.add_conv(p, "resnet.conv1", [L.Segment("in", 4 * in_channels)], stem_s2d_taps(sd["resnet.conv1.weight"]), 64, hh, ww, 1, sc, sh,
               pair=True, relu=True, out0=f1s, out0_s2d=True, macs_per_pair=2 * hh * ww * 64 * in_channels * 49)
    hh, ww = hh // 2, ww // 2
    x = p.tensor("p1", 2, hh, ww, 64)
    p.ops.append(L.MaxPoolS2DSpec("resnet.maxpool", f1s, x, 64, split=p.split))
    cin, x_s2d = 64, False

    # ---------------- layer1 .. layer{stages-1} (:284-294): only layer2 strides
    for li in range(stages - 1):
        cout = 64 << li
        for b in range(2):
            pre = f"resnet.layer{li + 1}.{b}"
            stride = 2 if (li == 1 and b == 0) else 1
            to_s2d = li == 0 and b == 1                       # layer1's output is only read by layer2's stride-2 convs
            if stride == 2:
                hh, ww = hh // 2, ww // 2
            t = p.tensor(f"{pre}.t", 2, hh, ww, cout)
            sc, sh = bn(f"{pre}.bn1", cout)
            w1, w2 = sd[f"{pre}.conv1.weight"], sd[f"{pre}.conv2.weight"]
            if stride == 2:
                assert x_s2d
                L.add_conv(p, f"{pre}.conv1", L.s2d_segments(x, cin), [(0, 0, L.s2d_conv_taps(w1, pad=1))], cout, hh, ww, 1, sc, sh,
                           pair=True, relu=True, out0=t, macs_per_pair=2 * hh * ww * 9 * cin * cout)
            else:
                L.add_conv(p, f"{pre}.conv1", [L.Segment(x, cin)], L.conv_taps(w1, pad=1), cout, hh, ww, 1, sc, sh, pair=True,
                           relu=True, out0=t, macs_per_pair=2 * hh * ww * 9 * cin * cout)
            if f"{pre}.downsample.0.weight" in sd:
                ident = p.tensor(f"{pre}.ds", 2, hh, ww, cout)
                sc, sh = bn(f"{pre}.downsample.1", cout)
                wd = sd[f"{pre}.downsample.0.weight"]
                if stride == 2:
                    L.add_conv(p, f"{pre}.downsample", L.s2d_segments(x, cin), [(0, 0, L.s2d_conv_taps(wd, pad=0))], cout, hh, ww, 1,
                               sc, sh, pair=True, out0=ident, macs_per_pair=2 * hh * ww * cin * cout)
                else:
                    L.add_conv(p, f"{pre}.downsample", [L.Segment(x, cin)], L.conv_taps(wd, pad=0), cout, hh, ww, 1, sc, sh, pair=True,
                               out0=ident, macs_per_pair=2 * hh * ww * cin * cout)
            else:
                ident = x
            sc, sh = bn(f"{pre}.bn2", cout)
            o = p.tensor(f"{pre}.o_s2d", 2, hh // 2, ww // 2, 4 * cout) if to_s2d else p.tensor(f"{pre}.o", 2, hh, ww, cout)
            L.add_conv(p, f"{pre}.conv2", [L.Segment(t, cout)], L.conv_taps(w2, pad=1), cout, hh, ww, 1, sc, sh, pair=True, relu=True,
                       res=ident, out0=o, out0_s2d=to_s2d, macs_per_pair=2 * hh * ww * 9 * cout * cout)
            x, x_s2d, cin = o, to_s2d, cout

    # ---------------- upsamplex2 (nearest) + conv_pred (:300-304) as 4 output phases of merged taps
    wp = sd["conv_pred.weight"]
    phases = [(a, b, L.up2_conv_taps(wp, 1, a, b)) for a in range(2) for b in range(2)]
    f = p.tensor("conv_pred.o", 2, 2 * hh, 2 * ww, 32)
    L.add_conv(p, "conv_pred", [L.Segment(x, cin)], phases, 32, hh, ww, 1, np.ones(32, np.float32), f32(sd["conv_pred.bias"]), pair=True,
               osy=2, osx=2, out0=f, macs_per_pair=2 * 4 * hh * ww * 9 * cin * 32)
    hh, ww = 2 * hh, 2 * ww

    # ---------------- tokenizer + transformer encoder / decoder (:414-428)
    if cfg:
        c, ie, idd, mlp = 32, cfg["inner_enc"], cfg["inner_dec"], cfg["mlp"]
        enc_rows, dec_rows = [], []
        for l in range(cfg["n_enc"]):
            a, ff = f"transformer.layers.{l}.0.fn", f"transformer.layers.{l}.1.fn"
            enc_rows.append(L.bit_pack(L.bit_enc_fields(c, ie, mlp), {
                "ln1_g": sd[f"{a}.norm.weight"], "ln1_b": sd[f"{a}.norm.bias"], "wqkv": sd[f"{a}.fn.to_qkv.weight"],
                "wout": sd[f"{a}.fn.to_out.0.weight"], "bout": sd[f"{a}.fn.to_out.0.bias"],
                "ln2_g": sd[f"{ff}.norm.weight"], "ln2_b": sd[f"{ff}.norm.bias"], "w1": sd[f"{ff}.fn.net.0.weight"],
                "b1": sd[f"{ff}.fn.net.0.bias"], "w2": sd[f"{ff}.fn.net.3.weight"], "b2": sd[f"{ff}.fn.net.3.bias"]}))
        for l in range(cfg["n_dec"]):
            a, ff = f"transformer_decoder.layers.{l}.0.fn", f"transformer_decoder.layers.{l}.1.fn"
            dec_rows.append(L.bit_pack(L.bit_dec_fields(c, idd, mlp), {
                "ln1_g": sd[f"{a}.norm.weight"], "ln1_b": sd[f"{a}.norm.bias"], "wq": sd[f"{a}.fn.to_q.weight"],
                "wk": sd[f"{a}.fn.to_k.weight"], "wv": sd[f"{a}.fn.to_v.weight"], "woutt": sd[f"{a}.fn.to_out.0.weight"].t().contiguous(),
                "bout": sd[f"{a}.fn.to_out.0.bias"], "ln2_g": sd[f"{ff}.norm.weight"], "ln2_b": sd[f"{ff}.norm.bias"],
                "w1t": sd[f"{ff}.fn.net.0.weight"].t().contiguous(), "b1": sd[f"{ff}.fn.net.0.bias"],
                "w2t": sd[f"{ff}.fn.net.3.weight"].t().contiguous(), "b2": sd[f"{ff}.fn.net.3.bias"]}))
        g = p.tensor("bit.o", 2, hh, ww, 32)
        # MACs actually executed per pixel and decoder layer by the collapsed form: 2 x 32x32 + 2 x 32x64 (the reference's
        # explicit q / dots / attn.v / to_out is 72 * inner + 4096)
        p.ops.append(L.BitTransformerSpec("bit", f, g, c, cfg["token_len"], cfg["heads"], ie, idd, mlp, f32(sd["conv_a.weight"].reshape(-1, c)),
                                          f32(sd["pos_embedding"].reshape(-1, c)), np.stack(enc_rows), np.stack(dec_rows),
                                          softmax=cfg["softmax"], macs_per_pair=2 * hh * ww * (cfg["n_dec"] * 6144 + cfg["token_len"] * 2 * c),
                                          split=p.split))
        f = g

    # ---------------- |x1 - x2|, bilinear x4, classifier (:430-436)
    d = p.tensor("diff", 1, hh, ww, 32)
    p.ops.append(L.AbsDiffSpec("diff", f, d, 32, split=p.split))
    u = p.tensor("diff.up4", 1, 4 * hh, 4 * ww, 32)
    p.ops.append(L.BilinearUpSpec("upsamplex4", d, u, 32, 4, split=p.split))
    hh, ww = 4 * hh, 4 * ww
    c1 = p.tensor("classifier.t", 1, hh, ww, 32)
    sc, sh = bn("classifier.1", 32)
    L.add_conv(p, "classifier.0", [L.Segment(u, 32)], L.conv_taps(sd["classifier.0.weight"], pad=1), 32, hh, ww, 1, sc, sh, relu=True,
               out0=c1, macs_per_pair=hh * ww * 9 * 32 * 32)
    L.add_conv(p, "classifier.3", [L.Segment(c1, 32)], L.conv_taps(sd["classifier.3.weight"], pad=1), n_class, hh, ww, 1,
               np.ones(n_class, np.float32), f32(sd["classifier.3.bias"]), out_ext=0, macs_per_pair=hh * ww * 9 * 32 * n_class)
    p.ext.append(L.ExtOutput("logits", n_class, hh, ww))
    return p
