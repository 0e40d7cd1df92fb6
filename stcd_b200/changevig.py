"""ChangeGNNV1 (ViG pyramid Siamese encoder + multi-scale difference decoder) behind ``net_G(x1, x2)``.

Drop-in for ``models/ChangeVIG.py::ChangeGNNV1`` (registry key ``ChangeGNNV1``, models/networks.py:196-198): same
constructor arguments, the reference's parameter names (a reference ``state_dict`` loads; the Grapher sub-module names
follow upstream ``gcn_lib``, which the reference imports but does not ship -- SURVEY.md App. D), same return value: a
list of five tensors ``[B,2,8,8] .. [B,2,64,64], [B,2,256,256]`` with the full-resolution logits last.

Lowering (eval mode; both temporal images ride through every encoder launch as Siamese pair tiles):

* Stem (pyramid_vig.py:66-83): 3x3 stride-2 convs read space-to-depth tensors (the image is packed space-to-depth, the
  first conv stores its output space-to-depth); BN + GELU fold into the epilogue; ``+ pos_embed`` is a residual read.
* Grapher (gcn_lib): fc1 (1x1 + BN) -> GRAPH OP (avg-pool by r, dense dilated kNN with the relative-position bias,
  max-relative aggregation: csrc/graph_kernels.cuh) -> the grouped 1x1 conv over the interleaved (x, m) as a dense conv
  over the virtual concat [x, m] with the group structure and the interleave folded into the packed weights, BN + GELU
  in the epilogue -> fc2 (1x1 + BN) + residual.
* FFN (pyramid_vig.py:41-63): two 1x1 convs, GELU and the residual in the epilogues.  The last block of stages 1-3 is
  stored twice: plainly for the decoder and space-to-depth for the stride-2 Downsample conv.
* DecoderV1 (ChangeVIG.py:192-281): per-pixel Linear heads as 1x1 convs; ``conv_diff`` reads ``cat(_c_1, _c_2)`` as two
  stream segments (never materialised), conv -> PReLU -> BN runs as (bias, PReLU, second affine) in one epilogue, the
  coarser scale's bilinear x2 is a residual read; bilinear resizes are one bandwidth kernel; ConvTranspose2d(k4, s2) runs
  as 4 output phases; ResidualBlock's ``* 0.1 + x`` is an epilogue affine + residual.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn as nn

from . import lowering as L
from .module import PlannedModule

_CHANNELS = (80, 160, 400, 640)
_BLOCKS = (2, 2, 6, 2)
_REDUCE = (4, 2, 1, 1)
_K = 9


def _relative_pos(c: int, n: int, r: int) -> torch.Tensor:
    """gcn_lib Grapher's relative_pos parameter: -bicubic(2 E E^T / C) with E the 2-D sin-cos embedding (App. D)."""
    g = int(n ** 0.5)

    def sincos(d, pos):
        omega = 1.0 / 10000 ** (np.arange(d // 2, dtype=np.float64) / (d / 2.0))
        out = np.einsum("m,d->md", pos.reshape(-1), omega)
        return np.concatenate([np.sin(out), np.cos(out)], axis=1)

    grid = np.stack(np.meshgrid(np.arange(g, dtype=np.float32), np.arange(g, dtype=np.float32)), axis=0).reshape(2, 1, g, g)
    emb = np.concatenate([sincos(c // 2, grid[0]), sincos(c // 2, grid[1])], axis=1)
    rel = torch.from_numpy(np.float32(2 * emb @ emb.T / emb.shape[1]))[None, None]
    rel = torch.nn.functional.interpolate(rel, size=(n, n // (r * r)), mode="bicubic", align_corners=False)
    return -rel.squeeze(1)


class _MRConv(nn.Module):
    def __init__(self, c: int):
        super().__init__()
        self.nn = nn.Sequential(nn.Conv2d(2 * c, 2 * c, 1, bias=True, groups=4), nn.BatchNorm2d(2 * c), nn.GELU())


class _DyGraphConv(nn.Module):
    def __init__(self, c: int):
        super().__init__()
        self.gconv = _MRConv(c)


class _Grapher(nn.Module):
    def __init__(self, c: int, k: int, dilation: int, r: int, n: int):
        super().__init__()
        self.k, self.dilation, self.r, self.n = k, dilation, r, n
        self.fc1 = nn.Sequential(nn.Conv2d(c, c, 1), nn.BatchNorm2d(c))
        self.graph_conv = _DyGraphConv(c)
        self.fc2 = nn.Sequential(nn.Conv2d(2 * c, c, 1), nn.BatchNorm2d(c))
        self.relative_pos = nn.Parameter(_relative_pos(c, n, r), requires_grad=False)


class _FFN(nn.Module):
    def __init__(self, c: int):
        super().__init__()
        self.fc1 = nn.Sequential(nn.Conv2d(c, 4 * c, 1), nn.BatchNorm2d(4 * c))
        self.act = nn.GELU()
        self.fc2 = nn.Sequential(nn.Conv2d(4 * c, c, 1), nn.BatchNorm2d(c))


class _Stem(nn.Module):
    def __init__(self, c: int):
        super().__init__()
        self.convs = nn.Sequential(nn.Conv2d(3, c // 2, 3, stride=2, padding=1), nn.BatchNorm2d(c // 2), nn.GELU(),
                                   nn.Conv2d(c // 2, c, 3, stride=2, padding=1), nn.BatchNorm2d(c), nn.GELU(),
                                   nn.Conv2d(c, c, 3, stride=1, padding=1), nn.BatchNorm2d(c))


class _Downsample(nn.Module):
    def __init__(self, cin: int, cout: int):
        super().__init__()
        self.conv = nn.Sequential(nn.Conv2d(cin, cout, 3, stride=2, padding=1), nn.BatchNorm2d(cout))


class _EncoderV1(nn.Module):
    """models/ChangeVIG.py:26-97 (parameters only)."""

    def __init__(self, img_size: int):
        super().__init__()
        self.stem = _Stem(_CHANNELS[0])
        self.pos_embed = nn.Parameter(torch.zeros(1, _CHANNELS[0], img_size // 4, img_size // 4))
        hw = (img_size // 4) ** 2
        max_dilation = 49 // _K
        mods: List[nn.Module] = []
        idx = 0
        for i, n_blocks in enumerate(_BLOCKS):
            if i > 0:
                mods.append(_Downsample(_CHANNELS[i - 1], _CHANNELS[i]))
                hw //= 4
            for _ in range(n_blocks):
                mods.append(nn.Sequential(_Grapher(_CHANNELS[i], _K, min(idx // 4 + 1, max_dilation), _REDUCE[i], hw),
                                          _FFN(_CHANNELS[i])))
                idx += 1
        self.backbone = nn.Sequential(*mods)


class _MLP(nn.Module):
    def __init__(self, cin: int, cout: int):
        super().__init__()
        self.proj = nn.Linear(cin, cout)


def _conv_diff(cin: int, cout: int) -> nn.Sequential:
    return nn.Sequential(nn.Conv2d(cin, cout, 3, padding=1), nn.PReLU(), nn.BatchNorm2d(cout), nn.Dropout(p=0.6),
                         nn.Conv2d(cout, cout, 3, padding=1), nn.PReLU(), nn.BatchNorm2d(cout), nn.Dropout(p=0.6))


def _make_prediction(cin: int, cout: int) -> nn.Sequential:
    return nn.Sequential(nn.Conv2d(cin, cout, 3, padding=1), nn.ReLU(), nn.BatchNorm2d(cout), nn.Conv2d(cout, cout, 3, padding=1))


class _ConvLayer(nn.Module):
    def __init__(self, cin, cout, k, stride, padding):
        super().__init__()
        self.conv2d = nn.Conv2d(cin, cout, k, stride, padding)


class _UpsampleConvLayer(nn.Module):
    def __init__(self, cin, cout, k, stride):
        super().__init__()
        self.conv2d = nn.ConvTranspose2d(cin, cout, k, stride=stride, padding=1)


class _ResidualBlock(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv1 = _ConvLayer(c, c, 3, 1, 1)
        self.conv2 = _ConvLayer(c, c, 3, 1, 1)
        self.relu = nn.ReLU()


class _DecoderV1(nn.Module):
    """models/ChangeVIG.py:100-165 with decoder_heads="MLP"."""

    def __init__(self, in_channels, e: int, output_nc: int, head: str = "decoder_heads_c"):
        super().__init__()
        c1, c2, c3, c4 = in_channels
        for k, c in ((4, c4), (3, c3), (2, c2), (1, c1)):      # DecoderTransformer_v3 calls them linear_c{k}
            setattr(self, f"{head}{k}", _MLP(c, e))
        for k in (4, 3, 2, 1):
            setattr(self, f"diff_c{k}", _conv_diff(2 * e, e))
        for k in (4, 3, 2, 1):
            setattr(self, f"make_pred_c{k}", _make_prediction(e, output_nc))
        self.linear_fuse = nn.Sequential(nn.Conv2d(e * 4, e, 1), nn.BatchNorm2d(e))
        self.convd2x = _UpsampleConvLayer(e, e, 4, 2)
        self.dense_2x = nn.Sequential(_ResidualBlock(e))
        self.convd1x = _UpsampleConvLayer(e, e, 4, 2)
        self.dense_1x = nn.Sequential(_ResidualBlock(e))
        self.change_probability = _ConvLayer(e, output_nc, 3, 1, 1)
        self.active = nn.Sigmoid()


class ChangeGNNV1(PlannedModule):
    """models/ChangeVIG.py:284-312."""
    default_chunk_pairs = 32

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False, embed_dim: int = 256,
                 decoder_heads: str = "MLP", img_size: int = 256):
        super().__init__()
        if input_nc != 3:
            raise NotImplementedError("ChangeGNNV1's Stem is hard-wired to 3 input channels (pyramid_vig.py:70)")
        if decoder_softmax or decoder_heads != "MLP":
            raise NotImplementedError("stcd_b200.ChangeGNNV1 serves decoder_heads='MLP', decoder_softmax=False (networks.py:197)")
        if output_nc > 8 or embed_dim % 16:
            raise NotImplementedError("output_nc <= 8, embed_dim a multiple of 16")
        self.embed_dims = list(_CHANNELS)
        self.embedding_dim = embed_dim
        self.output_nc = output_nc
        self.img_size = img_size
        self.encoder = _EncoderV1(img_size)
        self.decoder = _DecoderV1(_CHANNELS, embed_dim, output_nc)
        for m in self.encoder.modules():            # EncoderV1.model_init, ChangeVIG.py:76-83
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight)
                if m.bias is not None:
                    m.bias.data.zero_()

    def lower(self, h: int, w: int) -> L.Program:
        return lower_changegnn(self.state_dict(), self.embedding_dim, self.output_nc, self.img_size, h, w)

    @torch.no_grad()
    def forward(self, x1: torch.Tensor, x2: torch.Tensor):
        return self.plan_for(x1).forward(x1, x2)        # list of 5, full-resolution logits last (evaluator.py:176 takes [-1])

    def _wrap_outputs(self, outs):
        return list(outs)


# ------------------------------------------------------------------------------------------
def _s2d_input_taps(weight: torch.Tensor, pad: int) -> List:
    """A stride-2 conv over the image == a stride-1 conv over its space-to-depth packing (channel (py*2+px)*cin + c):
    kernel row ky reads input row 2i + ky - pad = 2(i + dy) + py."""
    cout, cin, k, _ = weight.shape
    taps = {}
    for ky in range(k):
        dy, py = divmod(ky - pad, 2)
        for kx in range(k):
            dx, px = divmod(kx - pad, 2)
            wt = taps.setdefault((dy, dx), torch.zeros(cout, 4 * cin, dtype=torch.float32))
            wt[:, (py * 2 + px) * cin: (py * 2 + px + 1) * cin] = weight[:, :, ky, kx].to(torch.float32)
    return [(0, 0, [(dy, dx, wt) for (dy, dx), wt in sorted(taps.items())])]


def lower_changegnn(sd: Dict[str, torch.Tensor], e: int, n_class: int, img_size: int, h: int, w: int) -> L.Program:
    """state_dict of the reference ChangeGNNV1 -> fused-op Program (eval mode)."""
    if h != img_size or w != img_size:
        # pos_embed is [1, C, img/4, img/4] and is added without resizing (ChangeVIG.py:87): the net only runs at img_size
        raise ValueError(f"ChangeGNNV1 was built for {img_size}x{img_size} inputs (its pos_embed is not resized), got {h}x{w}")
    if h % 32:
        raise ValueError("img_size must be a multiple of 32")
    sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
    p = L.Program(model="ChangeGNNV1", in_channels=3, h=h, w=w)
    feats = lower_vig_encoder(p, sd, h, w)
    lower_diff_decoder(p, sd, feats, e, n_class, "decoder", "decoder.decoder_heads_c{k}")
    return p


def lower_vig_encoder(p: L.Program, sd: Dict[str, torch.Tensor], h: int, w: int):
    """EncoderV1 == EncoderV2 (ChangeVIG.py:26-97, 463-534): Stem + pos_embed, 12 Grapher + FFN blocks, 3 Downsamples.
    Returns [(tensor, channels, h, w)] per stage, both streams."""
    ones = lambda c: np.ones(c, np.float32)  # noqa: E731,F841
    npf = lambda t: t.numpy().astype(np.float32)  # noqa: E731

    def conv_bn(pre: str, cout: int):
        return L.fold_bn(sd.get(f"{pre}.0.bias"), L.bn_params(sd, f"{pre}.1"), cout)

    # ---------------- Stem
    c0 = _CHANNELS[0]
    hh, ww = h // 2, w // 2
    p.tensor("in", 2, hh, ww, 16)
    p.ops.append(L.InputPackSpec("pack", "in", 3, s2d=True))
    s = "encoder.stem.convs"
    t0 = p.tensor("stem.t0_s2d", 2, hh // 2, ww // 2, 4 * (c0 // 2))
    sc, sh = L.fold_bn(sd[f"{s}.0.bias"], L.bn_params(sd, f"{s}.1"), c0 // 2)
    L.add_conv(p, f"{s}.0", [L.Segment("in", 12)], _s2d_input_taps(sd[f"{s}.0.weight"], 1), c0 // 2, hh, ww, 1, sc, sh, pair=True,
               act="gelu", out0=t0, out0_s2d=True, macs_per_pair=2 * hh * ww * 27 * (c0 // 2))
    hh, ww = hh // 2, ww // 2
    t1 = p.tensor("stem.t1", 2, hh, ww, c0)
    sc, sh = L.fold_bn(sd[f"{s}.3.bias"], L.bn_params(sd, f"{s}.4"), c0)
    L.add_conv(p, f"{s}.3", L.s2d_segments(t0, c0 // 2), [(0, 0, L.s2d_conv_taps(sd[f"{s}.3.weight"], pad=1))], c0, hh, ww, 1, sc, sh,
               pair=True, act="gelu", out0=t1, macs_per_pair=2 * hh * ww * 9 * (c0 // 2) * c0)
    pos = p.tensor("pos_embed", 2, hh, ww, c0)
    p.consts[pos] = sd["encoder.pos_embed"][0].permute(1, 2, 0).contiguous()
    x = p.tensor("stem.out", 2, hh, ww, c0)
    sc, sh = L.fold_bn(sd[f"{s}.6.bias"], L.bn_params(sd, f"{s}.7"), c0)
    L.add_conv(p, f"{s}.6", [L.Segment(t1, c0)], L.conv_taps(sd[f"{s}.6.weight"], pad=1), c0, hh, ww, 1, sc, sh, pair=True, res=pos,
               out0=x, macs_per_pair=2 * hh * ww * 9 * c0 * c0)

    # ---------------- ViG pyramid
    feats = []                    # (tensor, channels, h, w) per stage, plain layout
    max_dilation = 49 // _K
    bi = idx = 0
    x_s2d = None
    for i, n_blocks in enumerate(_BLOCKS):
        c = _CHANNELS[i]
        if i > 0:
            pre = f"encoder.backbone.{bi}.conv"
            cprev = _CHANNELS[i - 1]
            hh, ww = hh // 2, ww // 2
            x = p.tensor(f"down{i}", 2, hh, ww, c)
            sc, sh = conv_bn(pre, c)
            L.add_conv(p, pre, L.s2d_segments(x_s2d, cprev), [(0, 0, L.s2d_conv_taps(sd[f"{pre}.0.weight"], pad=1))], c, hh, ww, 1,
                       sc, sh, pair=True, out0=x, macs_per_pair=2 * hh * ww * 9 * cprev * c)
            bi += 1
        for b in range(n_blocks):
            g, f = f"encoder.backbone.{bi}.0", f"encoder.backbone.{bi}.1"
            dil = min(idx // 4 + 1, max_dilation)
            r = _REDUCE[i]
            # ---- Grapher
            x1 = p.tensor(f"{g}.x1", 2, hh, ww, c)
            sc, sh = conv_bn(f"{g}.fc1", c)
            L.add_conv(p, f"{g}.fc1", [L.Segment(x, c)], L.conv_taps(sd[f"{g}.fc1.0.weight"], pad=0), c, hh, ww, 1, sc, sh, pair=True,
                       out0=x1, macs_per_pair=2 * hh * ww * c * c)
            m = p.tensor(f"{g}.m", 2, hh, ww, c)
            rp = sd.get(f"{g}.relative_pos")
            n, mk = hh * ww, hh * ww // (r * r)
            if rp is not None and tuple(rp.shape[1:]) != (n, mk):
                rp = torch.nn.functional.interpolate(rp.unsqueeze(0), size=(n, mk), mode="bicubic").squeeze(0)
            p.ops.append(L.GraphConvSpec(f"{g}.graph", x1, m, c, _K, dil, r, None if rp is None else npf(rp[0]),
                                         macs_per_pair=2 * n * mk * c))
            # grouped 1x1 conv (groups=4) over the interleaved z = (x0, m0, x1, m1, ...): dense weights over [x, m]
            wg = sd[f"{g}.graph_conv.gconv.nn.0.weight"][:, :, 0, 0]            # [2c, 2c/4]
            dense = torch.zeros(2 * c, 2 * c)
            per = 2 * c // 4
            for grp in range(4):
                dense[grp * per:(grp + 1) * per, grp * per:(grp + 1) * per] = wg[grp * per:(grp + 1) * per]
            wx, wm = dense[:, 0::2], dense[:, 1::2]                                 # z[2j] = x[j], z[2j+1] = m[j]
            gz = p.tensor(f"{g}.gz", 2, hh, ww, 2 * c)
            sc, sh = L.fold_bn(sd.get(f"{g}.graph_conv.gconv.nn.0.bias"), L.bn_params(sd, f"{g}.graph_conv.gconv.nn.1"), 2 * c)
            L.add_conv(p, f"{g}.graph_conv.nn", [L.Segment(x1, c), L.Segment(m, c)],
                       [(0, 0, [(0, 0, torch.cat([wx, wm], 1))])], 2 * c, hh, ww, 1, sc, sh, pair=True, act="gelu", out0=gz,
                       macs_per_pair=2 * hh * ww * 2 * c * (2 * c // 4))
            xg = p.tensor(f"{g}.out", 2, hh, ww, c)
            sc, sh = conv_bn(f"{g}.fc2", c)
            L.add_conv(p, f"{g}.fc2", [L.Segment(gz, 2 * c)], L.conv_taps(sd[f"{g}.fc2.0.weight"], pad=0), c, hh, ww, 1, sc, sh,
                       pair=True, res=x, out0=xg, macs_per_pair=2 * hh * ww * 2 * c * c)
            # ---- FFN
            hdn = p.tensor(f"{f}.h", 2, hh, ww, 4 * c)
            sc, sh = conv_bn(f"{f}.fc1", 4 * c)
            L.add_conv(p, f"{f}.fc1", [L.Segment(xg, c)], L.conv_taps(sd[f"{f}.fc1.0.weight"], pad=0), 4 * c, hh, ww, 1, sc, sh,
                       pair=True, act="gelu", out0=hdn, macs_per_pair=2 * hh * ww * c * 4 * c)
            x = p.tensor(f"{f}.out", 2, hh, ww, c)
            sc, sh = conv_bn(f"{f}.fc2", c)
            L.add_conv(p, f"{f}.fc2", [L.Segment(hdn, 4 * c)], L.conv_taps(sd[f"{f}.fc2.0.weight"], pad=0), c, hh, ww, 1, sc, sh,
                       pair=True, res=xg, out0=x, macs_per_pair=2 * hh * ww * 4 * c * c)
            if b == n_blocks - 1 and i < 3:
                # the stage output also feeds the stride-2 Downsample: second, space-to-depth copy of the same conv
                x_s2d = p.tensor(f"{f}.out_s2d", 2, hh // 2, ww // 2, 4 * c)
                L.add_conv(p, f"{f}.fc2.s2d", [L.Segment(hdn, 4 * c)], L.conv_taps(sd[f"{f}.fc2.0.weight"], pad=0), c, hh, ww, 1,
                           sc, sh, pair=True, res=xg, out0=x_s2d, out0_s2d=True, macs_per_pair=0)
            bi += 1
            idx += 1
        feats.append((x, c, hh, ww))
    return feats


def lower_diff_decoder(p: L.Program, sd: Dict[str, torch.Tensor], feats, e: int, n_class: int, d: str, head_fmt: str) -> None:
    """DecoderV1 (ChangeVIG.py:192-281) == DecoderTransformer_v3 (ChangeFormer.py:1558-1631): per-scale Linear heads on both
    streams, conv_diff over cat(_c_1, _c_2) (+ the coarser scale's bilinear x2), intermediate predictions, bilinear
    resize to the finest scale, 1x1 fuse + BN, two (ConvTranspose2d(k4, s2) + ResidualBlock), 3x3 head.
    feats: [(tensor, channels, h, w)] fine -> coarse, both streams (mult 2); head_fmt: parameter prefix of the heads."""
    ones = lambda c: np.ones(c, np.float32)  # noqa: E731
    npf = lambda t: t.numpy().astype(np.float32)  # noqa: E731

    def conv_bn(pre: str, cout: int):
        return L.fold_bn(sd.get(f"{pre}.0.bias"), L.bn_params(sd, f"{pre}.1"), cout)

    full_h, full_w = feats[0][2], feats[0][3]
    c_prev = None
    ups = []
    for k in (4, 3, 2, 1):
        ft, fc, fh, fw = feats[k - 1]
        hd = p.tensor(f"{d}.c{k}", 2, fh, fw, e)
        wl = sd[head_fmt.format(k=k) + ".proj.weight"][:, :, None, None]
        L.add_conv(p, head_fmt.format(k=k), [L.Segment(ft, fc)], L.conv_taps(wl, pad=0), e, fh, fw, 1, ones(e),
                   npf(sd[head_fmt.format(k=k) + ".proj.bias"]), pair=True, out0=hd, macs_per_pair=2 * fh * fw * fc * e)
        dk = f"{d}.diff_c{k}"
        ta = p.tensor(f"{dk}.a", 1, fh, fw, e)
        s2, b2 = L.fold_bn(None, L.bn_params(sd, f"{dk}.2"), e)
        L.add_conv(p, f"{dk}.0", [L.Segment(hd, e, stream=0), L.Segment(hd, e, stream=1)], L.conv_taps(sd[f"{dk}.0.weight"], pad=1), e,
                   fh, fw, 1, ones(e), npf(sd[f"{dk}.0.bias"]), act="prelu", act_alpha=float(sd[f"{dk}.1.weight"][0]), act_pre=True,
                   scale2=s2, shift2=b2, out0=ta, macs_per_pair=fh * fw * 9 * 2 * e * e)
        res = None
        if c_prev is not None:
            res = p.tensor(f"{dk}.up_prev", 1, fh, fw, e)
            p.ops.append(L.BilinearUpSpec(f"{dk}.up_prev", c_prev, res, e, 2, split=p.split))
        ck = p.tensor(f"{dk}.out", 1, fh, fw, e)
        s2, b2 = L.fold_bn(None, L.bn_params(sd, f"{dk}.6"), e)
        L.add_conv(p, f"{dk}.4", [L.Segment(ta, e)], L.conv_taps(sd[f"{dk}.4.weight"], pad=1), e, fh, fw, 1, ones(e),
                   npf(sd[f"{dk}.4.bias"]), act="prelu", act_alpha=float(sd[f"{dk}.5.weight"][0]), act_pre=True, scale2=s2, shift2=b2,
                   res=res, out0=ck, macs_per_pair=fh * fw * 9 * e * e)
        # intermediate prediction (outputs[0..3]): conv, ReLU, BN, conv -> fp32
        mp = f"{d}.make_pred_c{k}"
        tp = p.tensor(f"{mp}.t", 1, fh, fw, 8)
        w0 = torch.zeros(8, e, 3, 3)
        w0[:n_class] = sd[f"{mp}.0.weight"]
        b0 = np.zeros(8, np.float32)
        b0[:n_class] = npf(sd[f"{mp}.0.bias"])
        s2, b2 = L.fold_bn(None, L.bn_params(sd, f"{mp}.2"), n_class)
        s2p, b2p = np.zeros(8, np.float32), np.zeros(8, np.float32)
        s2p[:n_class], b2p[:n_class] = s2, b2
        L.add_conv(p, f"{mp}.0", [L.Segment(ck, e)], L.conv_taps(w0, pad=1), 8, fh, fw, 1, ones(8), b0, act="relu", act_pre=True,
                   scale2=s2p, shift2=b2p, out0=tp, macs_per_pair=fh * fw * 9 * e * n_class)
        L.add_conv(p, f"{mp}.3", [L.Segment(tp, n_class)], L.conv_taps(sd[f"{mp}.3.weight"], pad=1), n_class, fh, fw, 1, ones(n_class),
                   npf(sd[f"{mp}.3.bias"]), out_ext=4 - k, macs_per_pair=fh * fw * 9 * n_class * n_class)
        p.ext.append(L.ExtOutput(f"p_c{k}", n_class, fh, fw))
        if k == 1:
            ups.append(ck)
        else:
            up = p.tensor(f"{dk}.up_full", 1, full_h, full_w, e)
            p.ops.append(L.BilinearUpSpec(f"{dk}.up_full", ck, up, e, full_h // fh, split=p.split))
            ups.append(up)
        c_prev = ck
    fused = p.tensor(f"{d}.fused", 1, full_h, full_w, e)
    sc, sh = conv_bn(f"{d}.linear_fuse", e)
    L.add_conv(p, f"{d}.linear_fuse", [L.Segment(t, e) for t in ups], L.conv_taps(sd[f"{d}.linear_fuse.0.weight"], pad=0), e,
               full_h, full_w, 1, sc, sh, out0=fused, macs_per_pair=full_h * full_w * 4 * e * e)
    lower_decoder_tail(p, sd, fused, full_h, full_w, e, n_class, d, out_ext=4)


def lower_decoder_tail(p: L.Program, sd: Dict[str, torch.Tensor], x: str, hh: int, ww: int, e: int, n_class: int, d: str, out_ext: int) -> None:
    """convd2x -> dense_2x -> convd1x -> dense_1x -> change_probability (ChangeVIG.py:264-274, 612-624): two
    (ConvTranspose2d(k4, s2, p1) as 4 phases + ResidualBlock with the 0.1 scale in the epilogue), 3x3 head -> fp32."""
    ones = lambda c: np.ones(c, np.float32)  # noqa: E731
    npf = lambda t: t.numpy().astype(np.float32)  # noqa: E731
    for up_name, res_name in (("convd2x", "dense_2x.0"), ("convd1x", "dense_1x.0")):
        wt = sd[f"{d}.{up_name}.conv2d.weight"]              # ConvTranspose2d [cin, cout, 4, 4], stride 2, padding 1
        u = p.tensor(f"{d}.{up_name}.out", 1, 2 * hh, 2 * ww, e)
        L.add_conv(p, f"{d}.{up_name}", [L.Segment(x, e)], L.convT_phase_taps(wt, stride=2, pad=1), e, hh, ww, 1, ones(e),
                   npf(sd[f"{d}.{up_name}.conv2d.bias"]), osy=2, osx=2, out0=u, macs_per_pair=hh * ww * 16 * e * e)
        hh, ww = 2 * hh, 2 * ww
        r1 = p.tensor(f"{d}.{res_name}.t", 1, hh, ww, e)
        L.add_conv(p, f"{d}.{res_name}.conv1", [L.Segment(u, e)], L.conv_taps(sd[f"{d}.{res_name}.conv1.conv2d.weight"], pad=1), e, hh,
                   ww, 1, ones(e), npf(sd[f"{d}.{res_name}.conv1.conv2d.bias"]), relu=True, out0=r1, macs_per_pair=hh * ww * 9 * e * e)
        x = p.tensor(f"{d}.{res_name}.out", 1, hh, ww, e)
        L.add_conv(p, f"{d}.{res_name}.conv2", [L.Segment(r1, e)], L.conv_taps(sd[f"{d}.{res_name}.conv2.conv2d.weight"], pad=1), e, hh,
                   ww, 1, 0.1 * ones(e), 0.1 * npf(sd[f"{d}.{res_name}.conv2.conv2d.bias"]), res=u, out0=x,
                   macs_per_pair=hh * ww * 9 * e * e)
    L.add_conv(p, f"{d}.change_probability", [L.Segment(x, e)], L.conv_taps(sd[f"{d}.change_probability.conv2d.weight"], pad=1),
               n_class, hh, ww, 1, ones(n_class), npf(sd[f"{d}.change_probability.conv2d.bias"]), out_ext=out_ext,
               macs_per_pair=hh * ww * 9 * e * n_class)
    p.ext.append(L.ExtOutput("cp", n_class, hh, ww))


# ==========================================================================================
# ChangeGNNV2 / ChangeGNNV2_Compare (models/ChangeVIG.py:315-460, 537-918): the same ViG encoder, HFFM + VFFM decoder
def _res_bottleneck_modules(holder: nn.Module, cin: int, cout: int) -> None:
    """conv_res / conv of Cross_ConCat, Sub, Abs, Conc (ChangeVIG.py:323-337)."""
    holder.conv_res = nn.Sequential(nn.Conv2d(cin, cout, 3, padding=1), nn.BatchNorm2d(cout))
    holder.conv = nn.Sequential(nn.Conv2d(cin, cout // 2, 1), nn.BatchNorm2d(cout // 2), nn.ReLU(),
                                nn.Conv2d(cout // 2, cout // 2, 3, padding=1), nn.BatchNorm2d(cout // 2), nn.ReLU(),
                                nn.Conv2d(cout // 2, cout, 1), nn.BatchNorm2d(cout))


class _CrossConCat(nn.Module):
    """models/ChangeVIG.py:315-337."""

    def __init__(self, cin: int, cout: int):
        super().__init__()
        self.diff = nn.Sequential(nn.Conv2d(cin * 2, cin, 3, padding=1, groups=cin), nn.BatchNorm2d(cin), nn.ReLU())
        _res_bottleneck_modules(self, cin, cout)


class _DiffOnly(nn.Module):
    """Sub / Abs (models/ChangeVIG.py:667-718): no parameters besides the residual bottleneck."""

    def __init__(self, cin: int, cout: int):
        super().__init__()
        _res_bottleneck_modules(self, cin, cout)


class _Conc(nn.Module):
    """models/ChangeVIG.py:721-750."""

    def __init__(self, cin: int, cout: int):
        super().__init__()
        self.diff = nn.Sequential(nn.Conv2d(cin * 2, cin, 3, padding=1), nn.BatchNorm2d(cin), nn.ReLU())
        _res_bottleneck_modules(self, cin, cout)


class _GlobalLocal(nn.Module):
    """models/ChangeVIG.py:350-375 (``bt`` is never used in forward; it is a parameter all the same)."""

    def __init__(self, c: int):
        super().__init__()
        self.channel_conv = nn.Conv2d(c, c, kernel_size=(2, 1), groups=c)
        self.channel_bn = nn.BatchNorm2d(c)
        self.spatial_conv = nn.Conv2d(2, 1, 5, padding=2)
        self.local_conv1 = nn.Conv2d(c, c, 1, groups=c)
        self.local_conv2 = nn.Conv2d(c, c, 3, padding=1, groups=c)
        self.local_conv3 = nn.Conv2d(c, c, 7, padding=3, groups=c)
        self.local_conv4 = nn.Conv2d(c * 3, c, 1)
        self.local_conv5 = nn.Conv2d(c, c, 3, padding=1)
        self.local_bn = nn.BatchNorm2d(c)
        self.bt = nn.BatchNorm2d(c)


class _HFFM(nn.Module):
    """HFFM (ChangeVIG.py:408-415) / HFFM_Compare (:753-765)."""

    def __init__(self, cin: int, cout: int, diff_mode: str):
        super().__init__()
        if diff_mode == "cross":
            self.cross_conc = _CrossConCat(cin, cout)
        else:
            self.diff = _Conc(cin, cout) if diff_mode == "conc" else _DiffOnly(cin, cout)
        self.global_local = _GlobalLocal(cout)


class _Upsampling(nn.Module):
    def __init__(self, c: int):
        super().__init__()
        self.up = nn.ConvTranspose2d(c, c, kernel_size=2, stride=2)


class _VFFM(nn.Module):
    """models/ChangeVIG.py:418-450."""

    def __init__(self, c: int, r: int = 4):
        super().__init__()
        i = c // r
        self.up = _Upsampling(c)
        self.global_avg = nn.Sequential(nn.AdaptiveAvgPool2d(1), nn.Conv2d(c, i, 1), nn.BatchNorm2d(i), nn.ReLU(inplace=True),
                                        nn.Conv2d(i, c, 1), nn.BatchNorm2d(c))
        self.global_max = nn.Sequential(nn.AdaptiveMaxPool2d(1), nn.Conv2d(c, i, 1), nn.BatchNorm2d(i), nn.ReLU(inplace=True),
                                        nn.Conv2d(i, c, 1), nn.BatchNorm2d(c))
        self.local_att = nn.Sequential(nn.Conv2d(c, i, 1), nn.BatchNorm2d(i), nn.ReLU(inplace=True), nn.Conv2d(i, c, 1), nn.BatchNorm2d(c))


class _DecoderV2(nn.Module):
    """DecoderV2 (ChangeVIG.py:537-595) / DecoderV2_Compare (:768-826)."""

    def __init__(self, in_channels, e: int, output_nc: int, diff_mode: str):
        super().__init__()
        c1, c2, c3, c4 = in_channels
        self.hffm4 = _HFFM(c4, e, diff_mode)
        self.hffm3 = _HFFM(c3, e, diff_mode)
        self.hffm2 = _HFFM(c2, e, diff_mode)
        self.hffm1 = _HFFM(c1, e, diff_mode)
        self.vffm3 = _VFFM(e)
        self.vffm2 = _VFFM(e)
        self.vffm1 = _VFFM(e)
        self.convd2x = _UpsampleConvLayer(e, e, 4, 2)
        self.dense_2x = nn.Sequential(_ResidualBlock(e))
        self.convd1x = _UpsampleConvLayer(e, e, 4, 2)
        self.dense_1x = nn.Sequential(_ResidualBlock(e))
        self.change_probability = _ConvLayer(e, output_nc, 3, 1, 1)
        self.active = nn.Sigmoid()


class ChangeGNNV2(PlannedModule):
    """models/ChangeVIG.py:634-664 (registry key ``ChangeGNNV2``, models/networks.py:201-202).  ``img_size`` is accepted and,
    like upstream, NOT forwarded to the encoder: EncoderV2 is always built for 256x256 (:647-650)."""
    default_chunk_pairs = 32
    _diff_mode = "cross"

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False, embed_dim: int = 256,
                 decoder_heads: str = "MLP", img_size: int = 256, diff_mode: Optional[str] = None):
        super().__init__()
        mode = self._diff_mode if diff_mode is None else diff_mode
        if input_nc != 3:
            raise NotImplementedError("the ViG Stem is hard-wired to 3 input channels (pyramid_vig.py:70)")
        if decoder_softmax:
            raise NotImplementedError("stcd_b200 serves decoder_softmax=False (models/networks.py:201-208)")
        if mode not in ("cross", "sub", "abs", "conc"):
            raise NotImplementedError(f"diff_mode {mode!r}")
        if output_nc > 8 or embed_dim % 64 or embed_dim > 512:
            raise NotImplementedError("output_nc <= 8, embed_dim a multiple of 64 up to 512")
        self.embed_dims = list(_CHANNELS)
        self.embedding_dim = embed_dim
        self.output_nc = output_nc
        self.diff_mode = mode
        self.encoder = _EncoderV1(256)
        self.decoder = _DecoderV2(_CHANNELS, embed_dim, output_nc, mode)
        for m in self.encoder.modules():            # EncoderV2.model_init, ChangeVIG.py:513-520
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight)
                if m.bias is not None:
                    m.bias.data.zero_()

    def lower(self, h: int, w: int) -> L.Program:
        return lower_changegnn_v2(self.state_dict(), self.embedding_dim, self.output_nc, self.diff_mode, h, w)

    @torch.no_grad()
    def forward(self, x1: torch.Tensor, x2: torch.Tensor):
        return self.plan_for(x1).forward(x1, x2)        # [cp]: a one-element list (ChangeVIG.py:626-631)

    def _wrap_outputs(self, outs):
        return list(outs)


class ChangeGNNV2_Compare(ChangeGNNV2):
    """models/ChangeVIG.py:865-918 (keys ``ChangeGNNV2_sub`` / ``_abs`` / ``_conc``, models/networks.py:203-208)."""
    _diff_mode = "sub"

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False, embed_dim: int = 256,
                 decoder_heads: str = "MLP", img_size: int = 256, diff_mode: str = "sub"):
        super().__init__(input_nc, output_nc, decoder_softmax, embed_dim, decoder_heads, img_size, diff_mode=diff_mode)


def lower_changegnn_v2(sd: Dict[str, torch.Tensor], e: int, n_class: int, diff_mode: str, h: int, w: int) -> L.Program:
    """state_dict of the reference ChangeGNNV2 / ChangeGNNV2_Compare -> fused-op Program (eval mode)."""
    if h != 256 or w != 256:
        raise ValueError(f"ChangeGNNV2's encoder is built for 256x256 inputs (its pos_embed is not resized), got {h}x{w}")
    sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
    p = L.Program(model=f"ChangeGNNV2-{diff_mode}", in_channels=3, h=h, w=w)
    feats = lower_vig_encoder(p, sd, h, w)
    ones = lambda c: np.ones(c, np.float32)  # noqa: E731
    npf = lambda t: np.ascontiguousarray(t.numpy().astype(np.float32))  # noqa: E731

    def cbn(pre: str, i: int, cout: int):
        return L.fold_bn(sd.get(f"{pre}.{i}.bias"), L.bn_params(sd, f"{pre}.{i + 1}"), cout)

    def hffm(k: int) -> str:
        ft, cin, hh, ww = feats[k - 1]
        q = f"decoder.hffm{k}." + ("cross_conc" if diff_mode == "cross" else "diff")
        if diff_mode == "cross":
            return global_local(k, _lower_cross_concat(p, sd, q, ft, cin, hh, ww, e), hh, ww)
        # ---- the difference feature `out` [cin]
        if diff_mode in ("sub", "abs"):
            out = p.tensor(f"{q}.out", 1, hh, ww, cin)
            p.ops.append(L.AbsDiffSpec(f"{q}.sub", ft, out, cin, signed=(diff_mode == "sub")))
        else:                                                              # conc: dense 3x3 over cat(a, b), split along K by stream
            wd = sd[f"{q}.diff.0.weight"]                                  # [cin, 2 cin, 3, 3]
            sc, sh = cbn(f"{q}.diff", 0, cin)
            part = p.tensor(f"{q}.part", 1, hh, ww, cin)
            L.add_conv(p, f"{q}.diff.a", [L.Segment(ft, cin, stream=0)], L.conv_taps(wd[:, :cin], pad=1), cin, hh, ww, 1, sc, 0 * sh, out0=part,
                       macs_per_pair=hh * ww * 9 * cin * cin)
            out = p.tensor(f"{q}.out", 1, hh, ww, cin)
            L.add_conv(p, f"{q}.diff.b", [L.Segment(ft, cin, stream=1)], L.conv_taps(wd[:, cin:], pad=1), cin, hh, ww, 1, sc, sh, relu=True,
                       res=part, out0=out, macs_per_pair=hh * ww * 9 * cin * cin)
        # ---- act(conv_res(out) + conv(out))
        r = p.tensor(f"{q}.res", 1, hh, ww, e)
        sc, sh = cbn(f"{q}.conv_res", 0, e)
        L.add_conv(p, f"{q}.conv_res", [L.Segment(out, cin)], L.conv_taps(sd[f"{q}.conv_res.0.weight"], pad=1), e, hh, ww, 1, sc, sh, out0=r,
                   macs_per_pair=hh * ww * 9 * cin * e)
        c1 = p.tensor(f"{q}.c1", 1, hh, ww, e // 2)
        sc, sh = cbn(f"{q}.conv", 0, e // 2)
        L.add_conv(p, f"{q}.conv.0", [L.Segment(out, cin)], L.conv_taps(sd[f"{q}.conv.0.weight"], pad=0), e // 2, hh, ww, 1, sc, sh, relu=True,
                   out0=c1, macs_per_pair=hh * ww * cin * e // 2)
        c2 = p.tensor(f"{q}.c2", 1, hh, ww, e // 2)
        sc, sh = cbn(f"{q}.conv", 3, e // 2)
        L.add_conv(p, f"{q}.conv.3", [L.Segment(c1, e // 2)], L.conv_taps(sd[f"{q}.conv.3.weight"], pad=1), e // 2, hh, ww, 1, sc, sh, relu=True,
                   out0=c2, macs_per_pair=hh * ww * 9 * (e // 2) * (e // 2))
        d = p.tensor(f"{q}.d", 1, hh, ww, e)
        sc, sh = cbn(f"{q}.conv", 6, e)
        L.add_conv(p, f"{q}.conv.6", [L.Segment(c2, e // 2)], L.conv_taps(sd[f"{q}.conv.6.weight"], pad=0), e, hh, ww, 1, sc, sh, relu=True, res=r,
                   out0=d, macs_per_pair=hh * ww * (e // 2) * e)
        return global_local(k, d, hh, ww)

    def global_local(k: int, d: str, hh: int, ww: int) -> str:
        g = f"decoder.hffm{k}.global_local"
        cs, ct = L.fold_bn(sd[f"{g}.channel_conv.bias"], L.bn_params(sd, f"{g}.channel_bn"), e)
        gated = p.tensor(f"{g}.gated", 1, hh, ww, e)
        wc = sd[f"{g}.channel_conv.weight"]                                # [e, 1, 2, 1]: (avg, max)
        p.ops.append(L.GlobalLocalGateSpec(f"{g}.gate", d, gated, e, npf(wc[:, 0, 0, 0]), npf(wc[:, 0, 1, 0]), cs, ct,
                                           npf(sd[f"{g}.spatial_conv.weight"][0]), float(sd[f"{g}.spatial_conv.bias"][0])))
        # local_conv4(cat(dw1x1, dw3x3, dw7x7)) is linear in x: ONE dense 7x7 conv whose weights are the composition
        w4 = sd[f"{g}.local_conv4.weight"][:, :, 0, 0]                     # [e, 3e]
        wl = w4[:, 2 * e:, None, None] * sd[f"{g}.local_conv3.weight"][:, 0][None]                   # [e, e, 7, 7]
        wl[:, :, 2:5, 2:5] += w4[:, e: 2 * e, None, None] * sd[f"{g}.local_conv2.weight"][:, 0][None]
        wl[:, :, 3, 3] += w4[:, :e] * sd[f"{g}.local_conv1.weight"][:, 0, 0, 0][None]
        bl = (sd[f"{g}.local_conv4.bias"] + w4[:, :e] @ sd[f"{g}.local_conv1.bias"] + w4[:, e: 2 * e] @ sd[f"{g}.local_conv2.bias"]
              + w4[:, 2 * e:] @ sd[f"{g}.local_conv3.bias"])
        sc, sh = L.fold_bn(bl, L.bn_params(sd, f"{g}.local_bn"), e)
        l1 = p.tensor(f"{g}.l1", 1, hh, ww, e)
        L.add_conv(p, f"{g}.local_conv1-4", [L.Segment(d, e)], L.conv_taps(wl, pad=3), e, hh, ww, 1, sc, sh, relu=True, out0=l1,
                   macs_per_pair=hh * ww * (59 * e + 3 * e * e))
        o = p.tensor(f"{g}.out", 1, hh, ww, e)
        L.add_conv(p, f"{g}.local_conv5", [L.Segment(l1, e)], L.conv_taps(sd[f"{g}.local_conv5.weight"], pad=1), e, hh, ww, 1, ones(e),
                   npf(sd[f"{g}.local_conv5.bias"]), res=gated, out0=o, macs_per_pair=hh * ww * 9 * e * e)
        return o

    def vffm(k: int, low: str, high_lr: str) -> str:
        _, _, hh, ww = feats[k - 1]
        v = f"decoder.vffm{k}"
        high = p.tensor(f"{v}.high", 1, hh, ww, e)
        L.add_conv(p, f"{v}.up", [L.Segment(high_lr, e)], L.convT_phase_taps(sd[f"{v}.up.up.weight"], 2, 0), e, hh // 2, ww // 2, 1, ones(e),
                   npf(sd[f"{v}.up.up.bias"]), osy=2, osx=2, out0=high, macs_per_pair=(hh // 2) * (ww // 2) * 4 * e * e)
        mixed = p.tensor(f"{v}.mixed", 1, hh, ww, e)
        p.ops.append(L.SumSpec(f"{v}.mixed", [low, high], mixed))
        i = e // 4
        la1 = p.tensor(f"{v}.la1", 1, hh, ww, i)
        sc, sh = cbn(f"{v}.local_att", 0, i)
        L.add_conv(p, f"{v}.local_att.0", [L.Segment(mixed, e)], L.conv_taps(sd[f"{v}.local_att.0.weight"], pad=0), i, hh, ww, 1, sc, sh,
                   relu=True, out0=la1, macs_per_pair=hh * ww * e * i)
        la2 = p.tensor(f"{v}.la2", 1, hh, ww, e)
        sc, sh = cbn(f"{v}.local_att", 3, e)
        L.add_conv(p, f"{v}.local_att.3", [L.Segment(la1, i)], L.conv_taps(sd[f"{v}.local_att.3.weight"], pad=0), e, hh, ww, 1, sc, sh, out0=la2,
                   macs_per_pair=hh * ww * i * e)
        branches = []
        for nm in ("global_avg", "global_max"):
            s1, t1 = cbn(f"{v}.{nm}", 1, i)
            s2, t2 = cbn(f"{v}.{nm}", 4, e)
            branches.append(dict(w1=npf(sd[f"{v}.{nm}.1.weight"][:, :, 0, 0]), s1=s1, t1=t1, w2=npf(sd[f"{v}.{nm}.4.weight"][:, :, 0, 0]), s2=s2, t2=t2))
        xo = p.tensor(f"{v}.out", 1, hh, ww, e)
        p.ops.append(L.VffmSpec(v, low, high, mixed, la2, xo, e, i, (branches[0], branches[1])))
        return xo

    c = hffm(4)
    for k in (3, 2, 1):
        c = vffm(k, hffm(k), c)
    _, _, hh, ww = feats[0]
    lower_decoder_tail(p, sd, c, hh, ww, e, n_class, "decoder", out_ext=0)
    return p


# ==========================================================================================
# VIG_V20_2 (registry key "GNN", models/ChangeVIG.py:921-1289): the ViG encoder under the prefix VIG_x2, conv_diff_V20 + csam_V20 + AFF
class _ConvDiffV20(_CrossConCat):
    """models/ChangeVIG.py:921-944: Cross_ConCat with in_channels given as 2 * C."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__(in_channels // 2, out_channels)


class _CsamV20(nn.Module):
    """models/ChangeVIG.py:956-980."""

    def __init__(self, c: int, ratio: int = 8):
        super().__init__()
        self.conv1_1 = nn.Conv2d(c, c, kernel_size=(2, 1), groups=c)
        self.batch_normal1 = nn.BatchNorm2d(c)
        self.liner1 = nn.Linear(c, c // ratio, bias=False)
        self.liner2 = nn.Linear(c // ratio, c)
        self.conv2_1 = nn.Conv2d(2, 1, 3, padding=1, bias=False)
        self.conv2_2 = nn.Conv2d(1, 1, 3, padding=1, bias=False)
        self.bt = nn.BatchNorm2d(c)


class _AFF(nn.Module):
    """models/ChangeVIG.py:996-1017."""

    def __init__(self, c: int, r: int = 4):
        super().__init__()
        i = c // r
        self.local_att = nn.Sequential(nn.Conv2d(c, i, 1), nn.BatchNorm2d(i), nn.ReLU(inplace=True), nn.Conv2d(i, c, 1), nn.BatchNorm2d(c))
        self.global_att = nn.Sequential(nn.AdaptiveAvgPool2d(1), nn.Conv2d(c, i, 1), nn.BatchNorm2d(i), nn.ReLU(inplace=True),
                                        nn.Conv2d(i, c, 1), nn.BatchNorm2d(c))


class _DecoderVIGV20(nn.Module):
    """models/ChangeVIG.py:1105-1184."""

    def __init__(self, in_channels, e: int, output_nc: int):
        super().__init__()
        c1, c2, c3, c4 = in_channels
        self.diff_c4 = _ConvDiffV20(2 * c4, e)
        self.diff_c3 = _ConvDiffV20(2 * c3, e)
        self.diff_c2 = _ConvDiffV20(2 * c2, e)
        self.diff_c1 = _ConvDiffV20(2 * c1, e)
        self.trans_conv4 = nn.ConvTranspose2d(e, e, kernel_size=2, stride=2)
        self.trans_conv3 = nn.ConvTranspose2d(e, e, kernel_size=2, stride=2)
        self.trans_conv2 = nn.ConvTranspose2d(e, e, kernel_size=2, stride=2)
        for k in (4, 3, 2, 1):
            setattr(self, f"csam{k}", _CsamV20(e))
        for k in (3, 2, 1):
            setattr(self, f"aff{k}", _AFF(e))
        self.convd2x = _UpsampleConvLayer(e, e, 4, 2)
        self.dense_2x = nn.Sequential(_ResidualBlock(e))
        self.convd1x = _UpsampleConvLayer(e, e, 4, 2)
        self.dense_1x = nn.Sequential(_ResidualBlock(e))
        self.change_probability = _ConvLayer(e, output_nc, 3, 1, 1)
        self.active = nn.Sigmoid()


class VIG_V20_2(PlannedModule):
    """models/ChangeVIG.py:1242-1289 (registry key ``GNN``, models/networks.py:210-211)."""
    default_chunk_pairs = 32

    def __init__(self, input_nc: int = 3, output_nc: int = 2, decoder_softmax: bool = False, embed_dim: int = 256,
                 decoder_heads: str = "MLP"):
        super().__init__()
        if input_nc != 3:
            raise NotImplementedError("the ViG Stem is hard-wired to 3 input channels (pyramid_vig.py:70)")
        if decoder_softmax:
            raise NotImplementedError("stcd_b200 serves decoder_softmax=False (models/networks.py:211)")
        if output_nc > 8 or embed_dim % 64 or embed_dim > 512:
            raise NotImplementedError("output_nc <= 8, embed_dim a multiple of 64 up to 512")
        self.embed_dims = list(_CHANNELS)
        self.embedding_dim = embed_dim
        self.output_nc = output_nc
        self.VIG_x2 = _EncoderV1(256)
        self.TDec_x2 = _DecoderVIGV20(_CHANNELS, embed_dim, output_nc)
        for m in self.VIG_x2.modules():             # EncoderVIG_V20_2.model_init, ChangeVIG.py:1078-1085
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight)
                if m.bias is not None:
                    m.bias.data.zero_()

    def lower(self, h: int, w: int) -> L.Program:
        return lower_vig_v20(self.state_dict(), self.embedding_dim, self.output_nc, h, w)

    @torch.no_grad()
    def forward(self, x1: torch.Tensor, x2: torch.Tensor):
        return self.plan_for(x1).forward(x1, x2)        # [cp]

    def _wrap_outputs(self, outs):
        return list(outs)


def _lower_cross_concat(p: L.Program, sd, q: str, ft: str, cin: int, hh: int, ww: int, e: int) -> str:
    """Cross_ConCat / conv_diff_V20 (ChangeVIG.py:315-347, 921-953) on the pair tensor ft -> [chunk, hh, ww, e]."""
    def cbn(pre: str, i: int, cout: int):
        return L.fold_bn(sd.get(f"{pre}.{i}.bias"), L.bn_params(sd, f"{pre}.{i + 1}"), cout)

    wg = sd[f"{q}.diff.0.weight"]                                  # [cin, 2, 3, 3]
    sc, sh = cbn(f"{q}.diff", 0, cin)
    out = p.tensor(f"{q}.out", 1, hh, ww, cin)
    nb = -(-cin // 320)
    blk = -(-cin // nb // 8) * 8
    for c0 in range(0, cin, blk):
        cb = min(blk, cin - c0)
        taps = []
        for ky in range(3):
            for kx in range(3):
                wt = torch.zeros(cb, 2 * cb)
                idx = torch.arange(cb)
                wt[idx, idx] = wg[c0: c0 + cb, 0, ky, kx]
                wt[idx, cb + idx] = wg[c0: c0 + cb, 1, ky, kx]
                taps.append((ky - 1, kx - 1, wt))
        L.add_conv(p, f"{q}.diff.{c0}", [L.Segment(ft, cb, stream=0, c_off=c0, c_store=cb), L.Segment(ft, cb, stream=1, c_off=c0, c_store=cb)],
                   [(0, 0, taps)], cb, hh, ww, 1, sc[c0: c0 + cb], sh[c0: c0 + cb], relu=True, out0=out, out0_coff=c0,
                   macs_per_pair=hh * ww * 9 * 2 * cb)
    r = p.tensor(f"{q}.res", 1, hh, ww, e)
    sc, sh = cbn(f"{q}.conv_res", 0, e)
    L.add_conv(p, f"{q}.conv_res", [L.Segment(out, cin)], L.conv_taps(sd[f"{q}.conv_res.0.weight"], pad=1), e, hh, ww, 1, sc, sh, out0=r,
               macs_per_pair=hh * ww * 9 * cin * e)
    c1 = p.tensor(f"{q}.c1", 1, hh, ww, e // 2)
    sc, sh = cbn(f"{q}.conv", 0, e // 2)
    L.add_conv(p, f"{q}.conv.0", [L.Segment(out, cin)], L.conv_taps(sd[f"{q}.conv.0.weight"], pad=0), e // 2, hh, ww, 1, sc, sh, relu=True,
               out0=c1, macs_per_pair=hh * ww * cin * e // 2)
    c2 = p.tensor(f"{q}.c2", 1, hh, ww, e // 2)
    sc, sh = cbn(f"{q}.conv", 3, e // 2)
    L.add_conv(p, f"{q}.conv.3", [L.Segment(c1, e // 2)], L.conv_taps(sd[f"{q}.conv.3.weight"], pad=1), e // 2, hh, ww, 1, sc, sh, relu=True,
               out0=c2, macs_per_pair=hh * ww * 9 * (e // 2) * (e // 2))
    d = p.tensor(f"{q}.d", 1, hh, ww, e)
    sc, sh = cbn(f"{q}.conv", 6, e)
    L.add_conv(p, f"{q}.conv.6", [L.Segment(c2, e // 2)], L.conv_taps(sd[f"{q}.conv.6.weight"], pad=0), e, hh, ww, 1, sc, sh, relu=True, res=r,
               out0=d, macs_per_pair=hh * ww * (e // 2) * e)
    return d


def lower_vig_v20(sd: Dict[str, torch.Tensor], e: int, n_class: int, h: int, w: int) -> L.Program:
    """state_dict of the reference VIG_V20_2 -> fused-op Program (eval mode)."""
    if h != 256 or w != 256:
        raise ValueError(f"VIG_V20_2's encoder is built for 256x256 inputs (its pos_embed is not resized), got {h}x{w}")
    sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
    p = L.Program(model="VIG_V20_2", in_channels=3, h=h, w=w)
    # the shared encoder lowering reads the prefix "encoder."
    enc_sd = {("encoder." + k[len("VIG_x2."):]): v for k, v in sd.items() if k.startswith("VIG_x2.")}
    feats = lower_vig_encoder(p, enc_sd, h, w)
    ones = lambda c: np.ones(c, np.float32)  # noqa: E731
    npf = lambda t: np.ascontiguousarray(t.numpy().astype(np.float32))  # noqa: E731
    d = "TDec_x2"

    def cbn(pre: str, i: int, cout: int):
        return L.fold_bn(sd.get(f"{pre}.{i}.bias"), L.bn_params(sd, f"{pre}.{i + 1}"), cout)

    def scale(k: int) -> str:
        ft, cin, hh, ww = feats[k - 1]
        x = _lower_cross_concat(p, sd, f"{d}.diff_c{k}", ft, cin, hh, ww, e)
        g = f"{d}.csam{k}"
        cs, ct = L.fold_bn(sd[f"{g}.conv1_1.bias"], L.bn_params(sd, f"{g}.batch_normal1"), e)
        bs, bt = L.fold_bn(None, L.bn_params(sd, f"{g}.bt"), e)
        wc = sd[f"{g}.conv1_1.weight"]
        o = p.tensor(f"{g}.o", 1, hh, ww, e)
        p.ops.append(L.CsamGateSpec(g, x, o, e, npf(wc[:, 0, 0, 0]), npf(wc[:, 0, 1, 0]), cs, ct, npf(sd[f"{g}.liner1.weight"]),
                                    npf(sd[f"{g}.liner2.weight"]), npf(sd[f"{g}.liner2.bias"]), bs, bt, npf(sd[f"{g}.conv2_1.weight"][0]),
                                    npf(sd[f"{g}.conv2_2.weight"][0, 0])))
        return o

    def up(k: int, x: str) -> str:
        _, _, hh, ww = feats[k - 1]
        o = p.tensor(f"{d}.trans_conv{k}.o", 1, 2 * hh, 2 * ww, e)
        L.add_conv(p, f"{d}.trans_conv{k}", [L.Segment(x, e)], L.convT_phase_taps(sd[f"{d}.trans_conv{k}.weight"], 2, 0), e, hh, ww, 1, ones(e),
                   npf(sd[f"{d}.trans_conv{k}.bias"]), osy=2, osx=2, out0=o, macs_per_pair=hh * ww * 4 * e * e)
        return o

    def aff(k: int, x: str, residual: str) -> str:
        _, _, hh, ww = feats[k - 1]
        a = f"{d}.aff{k}"
        i = e // 4
        xa = p.tensor(f"{a}.xa", 1, hh, ww, e)
        p.ops.append(L.SumSpec(f"{a}.xa", [x, residual], xa))
        l1 = p.tensor(f"{a}.l1", 1, hh, ww, i)
        sc, sh = cbn(f"{a}.local_att", 0, i)
        L.add_conv(p, f"{a}.local_att.0", [L.Segment(xa, e)], L.conv_taps(sd[f"{a}.local_att.0.weight"], pad=0), i, hh, ww, 1, sc, sh, relu=True,
                   out0=l1, macs_per_pair=hh * ww * e * i)
        l2 = p.tensor(f"{a}.l2", 1, hh, ww, e)
        sc, sh = cbn(f"{a}.local_att", 3, e)
        L.add_conv(p, f"{a}.local_att.3", [L.Segment(l1, i)], L.conv_taps(sd[f"{a}.local_att.3.weight"], pad=0), e, hh, ww, 1, sc, sh, out0=l2,
                   macs_per_pair=hh * ww * i * e)
        s1, t1 = cbn(f"{a}.global_att", 1, i)
        s2, t2 = cbn(f"{a}.global_att", 4, e)
        avg = dict(w1=npf(sd[f"{a}.global_att.1.weight"][:, :, 0, 0]), s1=s1, t1=t1, w2=npf(sd[f"{a}.global_att.4.weight"][:, :, 0, 0]), s2=s2, t2=t2)
        zero = dict(w1=np.zeros((i, e), np.float32), s1=np.zeros(i, np.float32), t1=np.zeros(i, np.float32), w2=np.zeros((e, i), np.float32),
                    s2=np.zeros(e, np.float32), t2=np.zeros(e, np.float32))     # AFF has no max branch
        o = p.tensor(f"{a}.o", 1, hh, ww, e)
        p.ops.append(L.VffmSpec(a, x, residual, xa, l2, o, e, i, (avg, zero)))
        return o

    c = up(4, scale(4))
    c = up(3, aff(3, scale(3), c))
    c = up(2, aff(2, scale(2), c))
    c = aff(1, scale(1), c)
    _, _, hh, ww = feats[0]
    lower_decoder_tail(p, sd, c, hh, ww, e, n_class, d, out_ext=0)
    return p
