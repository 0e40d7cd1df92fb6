"""Split-precision emulation of the MiT / decoder bandwidth ops.  TEST INFRASTRUCTURE.

``oracle.emulate`` executes convs, input packs and the ECAM head in split precision (lowering.Program.precision "split": every
activation is hi + lo bf16 planes).  This module adds the split forms of LayerNorm, spatial-reduction attention, the depth-wise
3x3 conv and bilinear up-sampling with the rounding points of their ``SPLIT = true`` kernels (csrc/transformer_kernels.cuh,
csrc/graph_kernels.cuh):

* read hi + lo, compute in fp32, write hi = bf16(v) and lo = bf16(v - hi);
* attention: the fp32 scores over hi + lo operands, P = exp(s - max) stored as hi + lo for P V, the fp32 row sum.

``run_program`` is ``oracle.emulate.run_program`` with these ops dispatched here; every other op runs in ``oracle.emulate``.
"""
from __future__ import annotations

from typing import Dict, List

import torch

from oracle import emulate as E
from stcd_b200 import lowering as L

_EVERY = (slice(None), slice(None), slice(None))


def run_layernorm(op: L.LayerNormSpec, T: Dict[str, torch.Tensor]) -> None:
    x = E._load(T, op.src, _EVERY, op.c, True)
    y = torch.nn.functional.layer_norm(x, (op.c,), torch.from_numpy(op.gamma), torch.from_numpy(op.beta), op.eps)
    E._store(T, op.dst, _EVERY, 0, y, True)
    if op.dst_s2d is not None:          # hi of class k at k*c, lo at 4c + k*c (the half of the 8c stored channels)
        for py in range(2):
            for px in range(2):
                E._store(T, op.dst_s2d, _EVERY, (py * 2 + px) * op.c, y[:, py::2, px::2], True)


def run_attention(op: L.AttentionSpec, T: Dict[str, torch.Tensor]) -> None:
    q = E._load(T, op.q, _EVERY, op.c, True)
    b, h, w, c = q.shape
    kv, half = T[op.kv], T[op.kv].shape[-1] // 2
    k = kv[..., :c] + kv[..., half: half + c]
    v = kv[..., c: 2 * c] + kv[..., half + c: half + 2 * c]
    d = c // op.heads
    qh = q.reshape(b, h * w, op.heads, d).permute(0, 2, 1, 3)
    k = k.reshape(b, -1, op.heads, d).permute(0, 2, 1, 3)
    v = v.reshape(b, -1, op.heads, d).permute(0, 2, 1, 3)
    if k.shape[2] != 64:
        raise ValueError(f"{op.name}: the split attention kernel takes exactly 64 keys")
    s_ = (qh @ k.transpose(-2, -1)) * op.scale
    p_ = torch.exp(s_ - s_.amax(dim=-1, keepdim=True))
    ph = E._bf16(p_)
    o = ((ph + E._bf16(p_ - ph)) @ v) / p_.sum(dim=-1, keepdim=True)
    E._store(T, op.dst, _EVERY, 0, o.transpose(1, 2).reshape(b, h, w, c), True)


def run_dwconv(op: L.DWConvSpec, T: Dict[str, torch.Tensor]) -> None:
    x = E._load(T, op.src, _EVERY, op.c, True).permute(0, 3, 1, 2)
    wt = torch.from_numpy(op.weight).reshape(op.c, 1, 3, 3)
    y = torch.nn.functional.conv2d(x, wt, torch.from_numpy(op.bias), padding=1, groups=op.c)
    if op.gelu:
        y = torch.nn.functional.gelu(y)
    E._store(T, op.dst, _EVERY, 0, y.permute(0, 2, 3, 1), True)


def run_bilinear_up(op: L.BilinearUpSpec, T: Dict[str, torch.Tensor]) -> None:
    x = E._load(T, op.src, _EVERY, op.c, True).permute(0, 3, 1, 2)
    y = torch.nn.functional.interpolate(x, scale_factor=op.scale, mode="bilinear", align_corners=False)
    E._store(T, op.dst, _EVERY, 0, y.permute(0, 2, 3, 1), True)


_SPLIT_OPS = {L.LayerNormSpec: run_layernorm, L.AttentionSpec: run_attention, L.DWConvSpec: run_dwconv,
              L.BilinearUpSpec: run_bilinear_up}


def run_program(prog: L.Program, x1: torch.Tensor, x2: torch.Tensor, chunk: int | None = None,
                keep: Dict[str, torch.Tensor] | None = None) -> List[torch.Tensor]:
    """x1, x2: fp32 NCHW [B, cin, H, W] -> list of fp32 NCHW external outputs (``oracle.emulate.run_program``'s contract)."""
    if any(isinstance(op, L.InputPackSpec) and (op.u8_norm is not None or op.s2d) for op in prog.ops):
        raise ValueError("split programs take fp32 inputs through the plain input pack")
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
            if isinstance(op, L.InputPackSpec):
                every = (slice(None), slice(None))
                E._store(T, op.dst, (slice(0, nv),) + every, 0, x1[start: start + nv].permute(0, 2, 3, 1), op.split)
                E._store(T, op.dst, (slice(chunk, chunk + nv),) + every, 0, x2[start: start + nv].permute(0, 2, 3, 1), op.split)
            elif isinstance(op, L.ConvSpec):
                E.run_conv(op, T, chunk, ext, nv)
            elif getattr(op, "split", False) and type(op) in _SPLIT_OPS:
                _SPLIT_OPS[type(op)](op, T)
            else:
                E.run_aux(op, T, chunk, ext, nv)
        for k in range(len(outs)):
            outs[k][start: start + nv] = ext[k][:nv]
        if keep is not None:
            keep.update(T)
    return outs
