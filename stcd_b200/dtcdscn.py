"""DTCDSCN (``CDNet34``: Siamese SE-ResNet-34, dilated centre block, SCSE decoder on feature differences) behind the
reference's ``net_G(x1, x2)`` contract.

Drop-in for ``models.DTCDSCN.CDNet34`` (models/DTCDSCN.py:316-320; registry key ``"DTCDSCN"``,
models/networks.py:159-160): same constructor, same parameter names and registration order (a reference
``state_dict`` loads, including the single-image branch ``decoder1..4`` / ``dblock`` / ``finaldeconv1`` /
``finalconv2`` / ``finalconv3`` whose forward is commented out upstream, :256-292: they are held as parameters
and never lowered), same return value: the change logits ``[B, num_classes, H, W]``.  Eval mode only.

Lowering (both temporal images ride through every encoder launch as Siamese pair tiles sharing the weights):

* stem: the 7x7 stride-2 conv reads a space-to-depth packing of the input (a 4x4 stride-1 conv with halo reuse), its
  output is stored space-to-depth so the 3x3 stride-2 max-pool and, later, every stride-2 conv read parity classes;
* ``SEBasicBlock`` (:78-109): conv1+BN+ReLU and conv2+BN are tcgen05 convs; the SE tail ``relu(out * g + residual)``
  needs the per-image channel mean of ``out`` before any pixel can be finished, so it is the two-pass bandwidth
  kernel K11 (channel sums, then gate + residual + ReLU), which also writes the space-to-depth copy the next
  layer's stride-2 convs read;
* ``e_x - e_y`` (:294-300) is one signed-difference kernel per level, fused with the ``decoder(...) +`` addend;
* ``Dblock`` (:52-71): dilation-d 3x3 convs are 9-tap convs with a 2d halo (thinner K chunks keep the stage in
  shared memory); taps that can only ever read padding (d >= feature size) are dropped at lowering time;
* ``DecoderBlock`` (:112-141): 1x1 conv+BN+ReLU, ``x + scse(x) = x * (1 + g_c + g_s(pixel))`` as K11 mode 1, the
  stride-2 ConvTranspose2d as 4 output phases (no zero-stuffing), 1x1 conv+BN+ReLU;
* head: ConvTranspose2d(64, 32, 4, 2, 1) as 4 phases of 2x2 taps, two 3x3 convs, fp32 logits.
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import lowering as L
from .module import PlannedModule
from .segcd import stem_s2d_taps

_FILTERS = (64, 128, 256, 512)


class _SELayer(nn.Module):
    """models/DTCDSCN.py:11-26 (parameters only)."""

    def __init__(self, channel: int, reduction: int = 16):
        super().__init__()
        self.fc = nn.Sequential(nn.Linear(channel, channel // reduction, bias=False), nn.ReLU(inplace=True),
                                nn.Linear(channel // reduction, channel, bias=False), nn.Sigmoid())


class _SEBasicBlock(nn.Module):
    """models/DTCDSCN.py:78-91."""

    def __init__(self, inplanes: int, planes: int, stride: int = 1, downsample=None, reduction: int = 16):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 3, stride=stride, padding=1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.se = _SELayer(planes, reduction)
        self.downsample = downsample


class _SCSEBlock(nn.Module):
    """models/DTCDSCN.py:144-162."""

    def __init__(self, channel: int, reduction: int = 16):
        super().__init__()
        self.channel_excitation = nn.Sequential(nn.Conv2d(channel, channel // reduction, 1, bias=False), nn.ReLU(inplace=True),
                                                nn.Conv2d(channel // reduction, channel, 1, bias=False), nn.Sigmoid())
        self.spatial_se = nn.Sequential(nn.Conv2d(channel, 1, 1, bias=False), nn.Sigmoid())


class _DecoderBlock(nn.Module):
    """models/DTCDSCN.py:112-127."""

    def __init__(self, in_channels: int, n_filters: int):
        super().__init__()
        mid = in_channels // 4
        self.conv1 = nn.Conv2d(in_channels, mid, 1)
        self.norm1 = nn.BatchNorm2d(mid)
        self.scse = _SCSEBlock(mid)
        self.deconv2 = nn.ConvTranspose2d(mid, mid, 3, stride=2, padding=1, output_padding=1)
        self.norm2 = nn.BatchNorm2d(mid)
        self.conv3 = nn.Conv2d(mid, n_filters, 1)
        self.norm3 = nn.BatchNorm2d(n_filters)


class _Dblock(nn.Module):
    """models/DTCDSCN.py:52-63 (biases start at zero)."""

    def __init__(self, channel: int):
        super().__init__()
        self.dilate1 = nn.Conv2d(channel, channel, 3, dilation=1, padding=1)
        self.dilate2 = nn.Conv2d(channel, channel, 3, dilation=2, padding=2)
        self.dilate3 = nn.Conv2d(channel, channel, 3, dilation=4, padding=4)
        self.dilate4 = nn.Conv2d(channel, channel, 3, dilation=8, padding=8)
        for m in self.modules():
            if isinstance(m, nn.Conv2d) and m.bias is not None:
                m.bias.data.zero_()


class CDNet_model(PlannedModule):
    """models/DTCDSCN.py:176-313."""
    default_chunk_pairs = 16
    supports_precision_path = True

    def __init__(self, in_channels: int = 3, block=None, layers: Sequence[int] = (3, 4, 6, 3), num_classes: int = 2):
        super().__init__()
        if block not in (None, _SEBasicBlock) and getattr(block, "__name__", "") != "SEBasicBlock":
            raise NotImplementedError("stcd_b200 serves the SEBasicBlock variant (CDNet34)")
        if in_channels > 4:
            raise NotImplementedError("in_channels <= 4")
        self.inchannels, self.layers, self.num_classes = in_channels, tuple(layers), num_classes
        f = _FILTERS
        self.inplanes = 64
        self.firstconv = nn.Conv2d(in_channels, 64, 7, stride=2, padding=3, bias=False)
        self.firstbn = nn.BatchNorm2d(64)
        self.encoder1 = self._make_layer(64, layers[0])
        self.encoder2 = self._make_layer(128, layers[1], stride=2)
        self.encoder3 = self._make_layer(256, layers[2], stride=2)
        self.encoder4 = self._make_layer(512, layers[3], stride=2)
        # the single-image branch: parameters only (its forward is commented out upstream, :256-292)
        self.decoder4 = _DecoderBlock(f[3], f[2])
        self.decoder3 = _DecoderBlock(f[2], f[1])
        self.decoder2 = _DecoderBlock(f[1], f[0])
        self.decoder1 = _DecoderBlock(f[0], f[0])
        self.dblock_master = _Dblock(512)
        self.dblock = _Dblock(512)
        self.decoder4_master = _DecoderBlock(f[3], f[2])
        self.decoder3_master = _DecoderBlock(f[2], f[1])
        self.decoder2_master = _DecoderBlock(f[1], f[0])
        self.decoder1_master = _DecoderBlock(f[0], f[0])
        self.finaldeconv1_master = nn.ConvTranspose2d(f[0], 32, 4, 2, 1)
        self.finalconv2_master = nn.Conv2d(32, 32, 3, padding=1)
        self.finalconv3_master = nn.Conv2d(32, num_classes, 3, padding=1)
        self.finaldeconv1 = nn.ConvTranspose2d(f[0], 32, 4, 2, 1)
        self.finalconv2 = nn.Conv2d(32, 32, 3, padding=1)
        self.finalconv3 = nn.Conv2d(32, num_classes, 3, padding=1)
        for m in self.modules():                                   # :218-224
            if isinstance(m, nn.Conv2d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2.0 / n))
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.data.fill_(1)
                m.bias.data.zero_()

    def _make_layer(self, planes: int, blocks: int, stride: int = 1) -> nn.Sequential:
        """models/DTCDSCN.py:226-242."""
        downsample = None
        if stride != 1 or self.inplanes != planes:
            downsample = nn.Sequential(nn.Conv2d(self.inplanes, planes, 1, stride=stride, bias=False), nn.BatchNorm2d(planes))
        layers = [_SEBasicBlock(self.inplanes, planes, stride, downsample)]
        self.inplanes = planes
        layers += [_SEBasicBlock(planes, planes) for _ in range(1, blocks)]
        return nn.Sequential(*layers)

    def lower(self, h: int, w: int) -> L.Program:
        return lower_dtcdscn(self.state_dict(), self.inchannels, self.layers, self.num_classes, h, w, precision=self.plan_precision)

    @torch.no_grad()
    def forward(self, x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
        return self.plan_for(x).forward(x, y)[0]


def CDNet34(in_channels: int, num_classes: int, **kwargs) -> CDNet_model:
    """models/DTCDSCN.py:316-320."""
    return CDNet_model(in_channels, _SEBasicBlock, [3, 4, 6, 3], num_classes, **kwargs)


# ------------------------------------------------------------------------------------------
def dilated_taps(weight: torch.Tensor, d: int, h: int, w: int) -> List:
    """3x3 conv, dilation = padding = d: taps at (+-d, +-d).  A tap whose offset is >= the feature size only ever reads the
    zero padding, for every output pixel: it is dropped (an 8x8 map under dilation 8 keeps the centre tap alone)."""
    taps = [((ky - 1) * d, (kx - 1) * d, weight[:, :, ky, kx].to(torch.float32)) for ky in range(3) for kx in range(3)
            if abs(ky - 1) * d < h and abs(kx - 1) * d < w]
    return [(0, 0, taps)]


def lower_dtcdscn(sd: Dict[str, torch.Tensor], in_channels: int, layers: Sequence[int], num_classes: int, h: int, w: int,
                  precision: str = "bf16") -> L.Program:
    """state_dict of the reference CDNet_model -> fused-op Program (eval mode).  precision "split": every op carries (hi, lo) bf16
    planes (lowering.Program.precision)."""
    if h % 32 or w % 32:
        raise ValueError(f"DTCDSCN lowering needs H and W divisible by 32 (got {h}x{w}): the reference's skip additions "
                         "do not line up otherwise")
    sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
    p = L.Program(model="CDNet34", in_channels=in_channels, h=h, w=w, precision=precision)

    def bn(prefix: str, c: int, bias=None):
        return L.fold_bn(bias, L.bn_params(sd, prefix), c)

    def f32(t: torch.Tensor) -> np.ndarray:
        return np.ascontiguousarray(t.numpy().astype(np.float32))

    # ---------------- stem (:246-249): space-to-depth pack, 4x4 conv, BN, ReLU (stored space-to-depth), max-pool
    hh, ww = h // 2, w // 2
    p.tensor("in", 2, hh, ww, 16)
    p.ops.append(L.InputPackSpec("pack", "in", in_channels, s2d=True, split=p.split))
    f1s = p.tensor("f1s", 2, hh // 2, ww // 2, 4 * 64)
    sc, sh = bn("firstbn", 64)
    L.add_conv(p, "firstconv", [L.Segment("in", 4 * in_channels)], stem_s2d_taps(sd["firstconv.weight"]), 64, hh, ww, 1, sc, sh,
               pair=True, relu=True, out0=f1s, out0_s2d=True, macs_per_pair=2 * hh * ww * 64 * in_channels * 49)
    hh, ww = hh // 2, ww // 2
    x = p.tensor("p1", 2, hh, ww, 64)
    p.ops.append(L.MaxPoolS2DSpec("firstmaxpool", f1s, x, 64, split=p.split))
    x_s2d = None                      # space-to-depth copy of x (what a stride-2 conv reads)
    cin = 64

    # ---------------- SE-ResNet encoder (:251-254, 269-272)
    feats = []                        # (tensor, channels, h, w) of e1..e4, both streams
    for li, (n_blocks, cout) in enumerate(zip(layers, _FILTERS)):
        for b in range(n_blocks):
            pre = f"encoder{li + 1}.{b}"
            stride = 2 if (b == 0 and li > 0) else 1
            last_of_layer = b == n_blocks - 1
            if stride == 2:
                hh, ww = hh // 2, ww // 2
            w1, w2 = sd[f"{pre}.conv1.weight"], sd[f"{pre}.conv2.weight"]
            t = p.tensor(f"{pre}.t", 2, hh, ww, cout)
            sc, sh = bn(f"{pre}.bn1", cout)
            if stride == 2:
                L.add_conv(p, f"{pre}.conv1", L.s2d_segments(x_s2d, cin), [(0, 0, L.s2d_conv_taps(w1, pad=1))], cout, hh, ww, 1, sc, sh,
                           pair=True, relu=True, out0=t, macs_per_pair=2 * hh * ww * 9 * cin * cout)
            else:
                L.add_conv(p, f"{pre}.conv1", [L.Segment(x, cin)], L.conv_taps(w1, pad=1), cout, hh, ww, 1, sc, sh, pair=True,
                           relu=True, out0=t, macs_per_pair=2 * hh * ww * 9 * cin * cout)
            u = p.tensor(f"{pre}.u", 2, hh, ww, cout)
            sc, sh = bn(f"{pre}.bn2", cout)
            L.add_conv(p, f"{pre}.conv2", [L.Segment(t, cout)], L.conv_taps(w2, pad=1), cout, hh, ww, 1, sc, sh, pair=True,
                       out0=u, macs_per_pair=2 * hh * ww * 9 * cout * cout)
            if f"{pre}.downsample.0.weight" in sd:
                ident = p.tensor(f"{pre}.ds", 2, hh, ww, cout)
                sc, sh = bn(f"{pre}.downsample.1", cout)
                wd = sd[f"{pre}.downsample.0.weight"]
                if stride == 2:
                    L.add_conv(p, f"{pre}.downsample", L.s2d_segments(x_s2d, cin), [(0, 0, L.s2d_conv_taps(wd, pad=0))], cout, hh, ww, 1,
                               sc, sh, pair=True, out0=ident, macs_per_pair=2 * hh * ww * cin * cout)
                else:
                    L.add_conv(p, f"{pre}.downsample", [L.Segment(x, cin)], L.conv_taps(wd, pad=0), cout, hh, ww, 1, sc, sh, pair=True,
                               out0=ident, macs_per_pair=2 * hh * ww * cin * cout)
            else:
                ident = x
            o = p.tensor(f"{pre}.o", 2, hh, ww, cout)
            o_s2d = p.tensor(f"{pre}.o_s2d", 2, hh // 2, ww // 2, 4 * cout) if (last_of_layer and li < 3) else None
            p.ops.append(L.ChannelGateSpec(f"{pre}.se", u, o, cout, f32(sd[f"{pre}.se.fc.0.weight"]), f32(sd[f"{pre}.se.fc.2.weight"]),
                                           mode=0, res=ident, dst_s2d=o_s2d, split=p.split))
            x, x_s2d, cin = o, o_s2d, cout
        feats.append((x, cout, hh, ww))

    # ---------------- centre: Dblock on e4_x - e4_y (:294; Dblock.forward :65-71)
    e4, c4, hh, ww = feats[3]
    dsum = [p.tensor("e4.diff", 1, hh, ww, c4)]
    p.ops.append(L.AbsDiffSpec("e4.diff", e4, dsum[0], c4, signed=True, split=p.split))
    cur = dsum[0]
    for i, dil in enumerate((1, 2, 4, 8)):
        nm = f"dblock_master.dilate{i + 1}"
        o = p.tensor(f"{nm}.o", 1, hh, ww, c4)
        taps = dilated_taps(sd[f"{nm}.weight"], dil, hh, ww)
        halo = max(t_[0] for t_ in taps[0][2]) - min(t_[0] for t_ in taps[0][2])
        L.add_conv(p, nm, [L.Segment(cur, c4)], taps, c4, hh, ww, 1, np.ones(c4, np.float32), f32(sd[f"{nm}.bias"]), relu=True, out0=o,
                   macs_per_pair=hh * ww * len(taps[0][2]) * c4 * c4, max_kc=64 if halo <= 4 else (32 if halo <= 8 else 16))
        dsum.append(o)
        cur = o
    x = p.tensor("dblock_master.o", 1, hh, ww, c4)
    p.ops.append(L.SumSpec("dblock_master.sum", dsum, x, split=p.split))
    cin = c4

    # ---------------- decoder on the differences (:296-299)
    for di, (nm, cout) in enumerate((("decoder4_master", 256), ("decoder3_master", 128), ("decoder2_master", 64), ("decoder1_master", 64))):
        mid = cin // 4
        midp = (mid + 7) // 8 * 8
        t1 = p.tensor(f"{nm}.t1", 1, hh, ww, midp)
        sc, sh = bn(f"{nm}.norm1", mid, sd[f"{nm}.conv1.bias"])
        L.add_conv(p, f"{nm}.conv1", [L.Segment(x, cin)], L.conv_taps(sd[f"{nm}.conv1.weight"], pad=0), mid, hh, ww, 1, sc, sh, relu=True,
                   out0=t1, macs_per_pair=hh * ww * cin * mid)
        hid = sd[f"{nm}.scse.channel_excitation.0.weight"].shape[0]
        w1g = np.zeros((hid, midp), np.float32)
        w2g = np.zeros((midp, hid), np.float32)
        wsg = np.zeros(midp, np.float32)
        w1g[:, :mid] = f32(sd[f"{nm}.scse.channel_excitation.0.weight"].reshape(hid, mid))
        w2g[:mid] = f32(sd[f"{nm}.scse.channel_excitation.2.weight"].reshape(mid, hid))
        wsg[:mid] = f32(sd[f"{nm}.scse.spatial_se.0.weight"].reshape(mid))
        t2 = p.tensor(f"{nm}.t2", 1, hh, ww, midp)
        p.ops.append(L.ChannelGateSpec(f"{nm}.scse", t1, t2, midp, w1g, w2g, mode=1, ws=wsg, split=p.split))
        t3 = p.tensor(f"{nm}.t3", 1, 2 * hh, 2 * ww, midp)
        sc, sh = bn(f"{nm}.norm2", mid, sd[f"{nm}.deconv2.bias"])
        L.add_conv(p, f"{nm}.deconv2", [L.Segment(t2, mid)], L.convT_phase_taps(sd[f"{nm}.deconv2.weight"], 2, 1), mid, hh, ww, 1, sc, sh,
                   relu=True, osy=2, osx=2, out0=t3, macs_per_pair=hh * ww * 9 * mid * mid)
        hh, ww = 2 * hh, 2 * ww
        o = p.tensor(f"{nm}.o", 1, hh, ww, cout)
        sc, sh = bn(f"{nm}.norm3", cout, sd[f"{nm}.conv3.bias"])
        L.add_conv(p, f"{nm}.conv3", [L.Segment(t3, mid)], L.conv_taps(sd[f"{nm}.conv3.weight"], pad=0), cout, hh, ww, 1, sc, sh, relu=True,
                   out0=o, macs_per_pair=hh * ww * mid * cout)
        if di < 3:
            e, ce, _, _ = feats[2 - di]
            d = p.tensor(f"{nm}.d", 1, hh, ww, cout)
            p.ops.append(L.AbsDiffSpec(f"{nm}.skip", e, d, ce, signed=True, add=o, split=p.split))
            o = d
        x, cin = o, cout

    # ---------------- head (:301-305)
    t = p.tensor("final.t1", 1, 2 * hh, 2 * ww, 32)
    L.add_conv(p, "finaldeconv1_master", [L.Segment(x, cin)], L.convT_phase_taps(sd["finaldeconv1_master.weight"], 2, 1), 32, hh, ww, 1,
               np.ones(32, np.float32), f32(sd["finaldeconv1_master.bias"]), relu=True, osy=2, osx=2, out0=t,
               macs_per_pair=hh * ww * 16 * cin * 32)
    hh, ww = 2 * hh, 2 * ww
    t2 = p.tensor("final.t2", 1, hh, ww, 32)
    L.add_conv(p, "finalconv2_master", [L.Segment(t, 32)], L.conv_taps(sd["finalconv2_master.weight"], pad=1), 32, hh, ww, 1,
               np.ones(32, np.float32), f32(sd["finalconv2_master.bias"]), relu=True, out0=t2, macs_per_pair=hh * ww * 9 * 32 * 32)
    L.add_conv(p, "finalconv3_master", [L.Segment(t2, 32)], L.conv_taps(sd["finalconv3_master.weight"], pad=1), num_classes, hh, ww, 1,
               np.ones(num_classes, np.float32), f32(sd["finalconv3_master.bias"]), out_ext=0,
               macs_per_pair=hh * ww * 9 * 32 * num_classes)
    p.ext.append(L.ExtOutput("change", num_classes, hh, ww))
    return p
