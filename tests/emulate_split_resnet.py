"""Split-precision emulation of the ResNet-family ops (BIT, DTCDSCN).  TEST INFRASTRUCTURE.

``emulate_split`` executes the MiT / decoder bandwidth ops in split precision (lowering.Program.precision "split": every
activation is hi + lo bf16 planes) and hands every other op to ``oracle.emulate``.  This module adds the split forms of the
ops BIT and DTCDSCN need, with the rounding points of their ``SPLIT = true`` kernels (csrc/aux_kernels.cuh,
csrc/transformer_kernels.cuh, csrc/bit_kernels.cuh) and of the conv epilogue's split store (csrc/conv_ws.cuh):

* the space-to-depth input pack (hi plane in channels [0, 16), lo plane in [16, 32));
* the space-to-depth conv store (hi of parity class k at k*cout, lo at 4*cout + k*cout);
* the space-to-depth max-pool: the max over hi + lo in the kernel's window order (first maximum wins), the winner's (hi, lo)
  pair copied;
* the feature differences, sums, SE / SCSE gates and BIT's token path: read hi + lo, compute in fp32, write hi = bf16(v) and
  lo = bf16(v - hi).

``run_program`` is ``emulate_split.run_program`` with these ops dispatched here as well.
"""
from __future__ import annotations

import dataclasses
from typing import Dict, List

import torch

import emulate_split as S
from oracle import emulate as E
from stcd_b200 import lowering as L

_EVERY = (slice(None), slice(None), slice(None))


def _planes(T: Dict[str, torch.Tensor], name: str) -> torch.Tensor:
    """Every stored channel of a split tensor as fp32 hi + lo values."""
    t = T[name]
    half = t.shape[-1] // 2
    return t[..., :half] + t[..., half:]


def run_input_pack_s2d(op: L.InputPackSpec, T: Dict[str, torch.Tensor], x: torch.Tensor, imgs: slice) -> None:
    """x: fp32 NHWC [n, 2h, 2w, cin] -> class (py, px) at channel (py*2 + px)*cin (split: its lo plane 16 channels further)."""
    for py in range(2):
        for px in range(2):
            E._store(T, op.dst, (imgs, slice(None), slice(None)), (py * 2 + px) * op.cin, x[:, py::2, px::2], op.split)


def run_maxpool_s2d(op: L.MaxPoolS2DSpec, T: Dict[str, torch.Tensor]) -> None:
    src, c = T[op.src], op.c
    hi = [src[..., k * c: (k + 1) * c] for k in range(4)]
    lo = [src[..., 4 * c + k * c: 4 * c + (k + 1) * c] for k in range(4)]

    def at(k: int, dy: int, dx: int):
        """class k at half-res pixel (y + dy, x + dx), dy, dx in {0, -1}; value -inf outside the map."""
        h_, l_ = hi[k], lo[k]
        v = h_ + l_
        if dy or dx:
            pad = (0, 0, -dx, 0, -dy, 0)
            h_ = torch.nn.functional.pad(h_, pad)[:, : h_.shape[1], : h_.shape[2]]
            l_ = torch.nn.functional.pad(l_, pad)[:, : l_.shape[1], : l_.shape[2]]
            v = torch.nn.functional.pad(v, pad, value=float("-inf"))[:, : v.shape[1], : v.shape[2]]
        return v, h_, l_

    # the kernel's window order: (2y, 2x), (2y, 2x+1), (2y+1, 2x), (2y+1, 2x+1), (2y, 2x-1), (2y+1, 2x-1), (2y-1, 2x), ...
    order = [(0, 0, 0), (1, 0, 0), (2, 0, 0), (3, 0, 0), (1, 0, -1), (3, 0, -1), (2, -1, 0), (3, -1, 0), (3, -1, -1)]
    bv, bh, bl = at(*order[0])
    for k, dy, dx in order[1:]:
        v, h_, l_ = at(k, dy, dx)
        m = v > bv
        bv, bh, bl = torch.where(m, v, bv), torch.where(m, h_, bh), torch.where(m, l_, bl)
    half = T[op.dst].shape[-1] // 2
    T[op.dst][..., :c] = bh
    T[op.dst][..., half: half + c] = bl


def run_absdiff(op: L.AbsDiffSpec, T: Dict[str, torch.Tensor], chunk: int) -> None:
    x = _planes(T, op.src)
    a, b = x[:chunk], x[chunk: 2 * chunk]
    if op.add is not None:
        a = _planes(T, op.add) + a                  # reference order: (d + e_x) - e_y
    d = a - b
    E._store(T, op.dst, _EVERY, 0, d if op.signed else d.abs(), True)


def run_sum(op: L.SumSpec, T: Dict[str, torch.Tensor]) -> None:
    acc = torch.zeros_like(_planes(T, op.dst))
    for s_ in op.srcs:                              # fp32, in source order
        acc = acc + _planes(T, s_)
    E._store(T, op.dst, _EVERY, 0, acc, True)


def run_channel_gate(op: L.ChannelGateSpec, T: Dict[str, torch.Tensor]) -> None:
    x = E._load(T, op.src, _EVERY, op.c, True)
    g = torch.sigmoid(torch.relu(x.mean(dim=(1, 2)) @ torch.from_numpy(op.w1).T) @ torch.from_numpy(op.w2).T)[:, None, None, :]
    if op.mode == 0:
        y = torch.relu(x * g + (E._load(T, op.res, _EVERY, op.c, True) if op.res is not None else 0.0))
    else:
        gs = torch.sigmoid((x * torch.from_numpy(op.ws)).sum(-1, keepdim=True))
        y = x * (1.0 + g + gs)
    E._store(T, op.dst, _EVERY, 0, y, True)
    if op.dst_s2d is not None:          # hi of class k at k*c, lo at 4c + k*c
        for py in range(2):
            for px in range(2):
                E._store(T, op.dst_s2d, _EVERY, (py * 2 + px) * op.c, y[:, py::2, px::2], True)


def run_bit_transformer(op: L.BitTransformerSpec, T: Dict[str, torch.Tensor], chunk: int) -> None:
    """``oracle.emulate.run_bit_transformer`` on the hi + lo map, the result written as both planes."""
    import torch.nn.functional as F
    x = E._load(T, op.src, _EVERY, op.c, True)      # [2*chunk, h, w, c]
    n2, h, w, c = x.shape
    xf = x.reshape(n2, h * w, c)
    a = torch.softmax(xf @ torch.from_numpy(op.conv_a).T, dim=1)
    tok = torch.einsum("bnl,bnc->blc", a, xf)
    t = torch.cat([tok[:chunk], tok[chunk:]], dim=1) + torch.from_numpy(op.pos)[None]
    scale = c ** -0.5

    def attend(q, k, v, softmax=True):
        b, n, inner = q.shape
        d = inner // op.heads
        qh, kh, vh = (z.reshape(b, -1, op.heads, d).transpose(1, 2) for z in (q, k, v))
        dots = torch.einsum("bhid,bhjd->bhij", qh, kh) * scale
        at = dots.softmax(-1) if softmax else dots
        return torch.einsum("bhij,bhjd->bhid", at, vh).transpose(1, 2).reshape(b, n, inner)

    for row in op.enc:
        P = L.bit_unpack(L.bit_enc_fields(c, op.inner_enc, op.mlp), row)
        y = F.layer_norm(t, (c,), P["ln1_g"], P["ln1_b"])
        q, k, v = (y @ P["wqkv"].T).chunk(3, dim=-1)
        t = attend(q, k, v) @ P["wout"].T + P["bout"] + t
        y = F.layer_norm(t, (c,), P["ln2_g"], P["ln2_b"])
        t = F.gelu(y @ P["w1"].T + P["b1"]) @ P["w2"].T + P["b2"] + t
    m = torch.cat([t[:, : op.token_len], t[:, op.token_len:]], dim=0)
    z = xf
    for row in op.dec:
        P = L.bit_unpack(L.bit_dec_fields(c, op.inner_dec, op.mlp), row)
        zn, mn = F.layer_norm(z, (c,), P["ln1_g"], P["ln1_b"]), F.layer_norm(m, (c,), P["ln1_g"], P["ln1_b"])
        o = attend(zn @ P["wq"].T, mn @ P["wk"].T, mn @ P["wv"].T, op.softmax)
        z = o @ P["woutt"] + P["bout"] + z
        y = F.layer_norm(z, (c,), P["ln2_g"], P["ln2_b"])
        z = F.gelu(y @ P["w1t"] + P["b1"]) @ P["w2t"] + P["b2"] + z
    E._store(T, op.dst, _EVERY, 0, z.reshape(n2, h, w, c), True)


def run_conv(op: L.ConvSpec, T: Dict[str, torch.Tensor], chunk: int, ext: List[torch.Tensor], nv: int) -> None:
    """``oracle.emulate.run_conv``; a split op with a space-to-depth out0 is run into a full-resolution split tensor first and
    then stored per parity class, both planes."""
    if not (op.split and op.out0_s2d):
        return E.run_conv(op, T, chunk, ext, nv)
    t = T[op.out0]
    tmp = f"{op.out0}.full"
    T[tmp] = torch.zeros(t.shape[0], 2 * t.shape[1], 2 * t.shape[2], 2 * op.cout)
    E.run_conv(dataclasses.replace(op, out0=tmp, out0_s2d=False), T, chunk, ext, nv)
    v = E._load(T, tmp, _EVERY, op.cout, True)
    del T[tmp]
    for py in range(2):
        for px in range(2):
            E._store(T, op.out0, _EVERY, (py * 2 + px) * op.cout, v[:, py::2, px::2], True)


_SPLIT_OPS = {L.MaxPoolS2DSpec: run_maxpool_s2d, L.SumSpec: run_sum, L.ChannelGateSpec: run_channel_gate}
_SPLIT_OPS_CHUNK = {L.AbsDiffSpec: run_absdiff, L.BitTransformerSpec: run_bit_transformer}     # ops that need the chunk size


def run_program(prog: L.Program, x1: torch.Tensor, x2: torch.Tensor, chunk: int | None = None,
                keep: Dict[str, torch.Tensor] | None = None) -> List[torch.Tensor]:
    """x1, x2: fp32 NCHW [B, cin, H, W] -> list of fp32 NCHW external outputs (``oracle.emulate.run_program``'s contract)."""
    if any(isinstance(op, L.InputPackSpec) and op.u8_norm is not None for op in prog.ops):
        raise ValueError("split programs take fp32 inputs")
    n = x1.shape[0]
    chunk = chunk or n
    outs = [torch.zeros(n, e.channels, e.h, e.w) for e in prog.ext]
    for start in range(0, n, chunk):
        nv = min(chunk, n - start)
        T = {name: torch.zeros(t.mult * chunk, t.h, t.w, t.c) for name, t in prog.tensors.items()}
        for name, val in prog.consts.items():
            T[name][..., : val.shape[2]] = E._bf16(val)[None]
        ext = [torch.zeros(chunk, e.channels, e.h, e.w) for e in prog.ext]
        for op in prog.ops:
            split = getattr(op, "split", False)
            if isinstance(op, L.InputPackSpec) and op.s2d:
                run_input_pack_s2d(op, T, x1[start: start + nv].permute(0, 2, 3, 1), slice(0, nv))
                run_input_pack_s2d(op, T, x2[start: start + nv].permute(0, 2, 3, 1), slice(chunk, chunk + nv))
            elif isinstance(op, L.InputPackSpec):
                every = (slice(None), slice(None))
                E._store(T, op.dst, (slice(0, nv),) + every, 0, x1[start: start + nv].permute(0, 2, 3, 1), op.split)
                E._store(T, op.dst, (slice(chunk, chunk + nv),) + every, 0, x2[start: start + nv].permute(0, 2, 3, 1), op.split)
            elif isinstance(op, L.ConvSpec):
                run_conv(op, T, chunk, ext, nv)
            elif split and type(op) in _SPLIT_OPS:
                _SPLIT_OPS[type(op)](op, T)
            elif split and type(op) in _SPLIT_OPS_CHUNK:
                _SPLIT_OPS_CHUNK[type(op)](op, T, chunk)
            elif split and type(op) in S._SPLIT_OPS:
                S._SPLIT_OPS[type(op)](op, T)
            else:
                E.run_aux(op, T, chunk, ext, nv)
        for k in range(len(outs)):
            outs[k][start: start + nv] = ext[k][:nv]
        if keep is not None:
            keep.update(T)
    return outs
