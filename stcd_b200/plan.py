"""Program -> libstcd_b200 plan (the device-side object behind ``net_G(x1, x2)``).

``Plan`` hands a lowered ``Program`` (stcd_b200/lowering.py) to the C-ABI: it declares the
activation tensors, adds each fused op, finalizes (workspace, weight upload, TMA descriptors)
and then runs ``stcd_forward`` on device pointers or ``stcd_forward_host`` on host buffers.
PyTorch appears only as the owner of the caller's device memory and stream.  There is no CPU
path: constructing a Plan without an sm_100 device raises ``StcdError``.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .lowering import (AbsDiffSpec, AttentionSpec, BitTransformerSpec, ChannelAttentionSpec, ChannelGateSpec, CsamGateSpec, GlobalLocalGateSpec, SpatialGateSpec, SumSpec, VffmSpec, BilinearUpSpec, ConvSpec, DWConvSpec, EcamHeadSpec, GraphConvSpec, InputPackSpec,
                       LayerNormSpec, MaxPoolS2DSpec, Program, SegHeadSpec)


def _fptr(a: Optional[np.ndarray]):
    if a is None:
        return C.cast(None, C.POINTER(C.c_float))
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_float))


class Plan:
    def __init__(self, prog: Program, chunk_pairs: int, device: int = 0):
        """device = -1: a validation plan -- every op descriptor goes through the library's checks (as on a GPU box), nothing
        is finalized and nothing can run (the host-side tests use it without a GPU)."""
        self.lib = _lib.lib()
        self.prog = prog
        self.chunk = int(chunk_pairs)
        self.device = int(device)
        self.u8 = False                      # set by _build when the input op takes uint8 HWC images
        self._h = C.c_void_p()
        precision = _lib.PRECISION_SPLIT if prog.split else _lib.PRECISION_BF16
        _lib.check(self.lib.stcd_plan_create(self.device, self.chunk, precision, C.byref(self._h)), "stcd_plan_create")
        try:
            self._build()
        except Exception:
            self.close()
            raise

    # ------------------------------------------------------------------ construction
    def _build(self) -> None:
        lib, h, prog = self.lib, self._h, self.prog
        ids = {}
        for name, t in prog.tensors.items():
            ids[name] = _lib.check_id(lib.stcd_plan_add_tensor(h, t.mult, t.h, t.w, t.c, 0), f"tensor {name}")
        self.tensor_ids = ids
        for op in prog.ops:
            if isinstance(op, InputPackSpec) and op.u8_norm is not None and prog.split:
                raise NotImplementedError("split precision takes fp32 inputs (forward_uint8 is the bf16 path's loader fusion)")
            if isinstance(op, InputPackSpec) and op.u8_norm is not None:
                mean = (C.c_float * op.cin)(*op.u8_norm[0][: op.cin])
                std = (C.c_float * op.cin)(*op.u8_norm[1][: op.cin])
                _lib.check_id(lib.stcd_plan_add_input_pack_u8(h, ids[op.dst], op.cin, 1 if op.s2d else 0, mean, std),
                              f"uint8 input pack {op.name}")
                self.u8 = True
            elif isinstance(op, InputPackSpec):
                add = lib.stcd_plan_add_input_pack_s2d if op.s2d else lib.stcd_plan_add_input_pack
                _lib.check_id(add(h, ids[op.dst], op.cin), f"input pack {op.name}")
            elif isinstance(op, GraphConvSpec):
                rp = None if op.relpos is None else np.ascontiguousarray(op.relpos, np.float32)
                _lib.check_id(lib.stcd_plan_add_graph_conv(h, ids[op.src], ids[op.dst], op.c, op.k, op.dilation, op.r, _fptr(rp)),
                              f"graph conv {op.name}")
            elif isinstance(op, AbsDiffSpec):
                if op.signed:
                    r = lib.stcd_plan_add_subdiff(h, ids[op.src], -1 if op.add is None else ids[op.add], ids[op.dst])
                else:
                    r = lib.stcd_plan_add_absdiff(h, ids[op.src], ids[op.dst])
                _lib.check_id(r, f"diff {op.name}")
            elif isinstance(op, ChannelGateSpec):
                w1, w2 = np.ascontiguousarray(op.w1, np.float32), np.ascontiguousarray(op.w2, np.float32)
                ws = None if op.ws is None else np.ascontiguousarray(op.ws, np.float32)
                _lib.check_id(lib.stcd_plan_add_channel_gate(h, ids[op.src], -1 if op.res is None else ids[op.res], ids[op.dst],
                                                             -1 if op.dst_s2d is None else ids[op.dst_s2d], op.c, w1.shape[0], _fptr(w1),
                                                             _fptr(w2), _fptr(ws), op.mode), f"channel gate {op.name}")
            elif isinstance(op, BitTransformerSpec):
                d = _lib.BitDesc()
                d.c, d.token_len, d.heads, d.mlp = op.c, op.token_len, op.heads, op.mlp
                d.n_enc, d.n_dec, d.inner_enc, d.inner_dec, d.softmax = len(op.enc), len(op.dec), op.inner_enc, op.inner_dec, int(op.softmax)
                keep = [np.ascontiguousarray(a, np.float32) for a in (op.conv_a, op.pos, op.enc, op.dec)]
                if len(op.enc) == 0:
                    keep[2] = np.zeros(1, np.float32)
                d.conv_a, d.pos, d.enc, d.dec = (_fptr(a) for a in keep)
                _lib.check_id(lib.stcd_plan_add_bit_transformer(h, ids[op.src], ids[op.dst], C.byref(d)), f"BIT transformer {op.name}")
            elif isinstance(op, ChannelAttentionSpec):
                n = len(op.srcs)
                ts = (C.c_int * n)(*[ids[s_[0]] for s_ in op.srcs])
                ss = (C.c_int * n)(*[s_[1] for s_ in op.srcs])
                cs = (C.c_int * n)(*[s_[2] for s_ in op.srcs])
                fc1, fc2 = np.ascontiguousarray(op.fc1, np.float32), np.ascontiguousarray(op.fc2, np.float32)
                _lib.check_id(lib.stcd_plan_add_channel_attention(h, ts, ss, cs, n, ids[op.dst], fc1.shape[0], _fptr(fc1), _fptr(fc2)),
                              f"channel attention {op.name}")
            elif isinstance(op, SpatialGateSpec):
                w_, sc_, sh_ = (np.ascontiguousarray(a, np.float32) for a in (op.w, op.scale, op.shift))
                _lib.check_id(lib.stcd_plan_add_spatial_gate(h, ids[op.src], ids[op.dst], op.c, _fptr(w_), _fptr(sc_), _fptr(sh_)),
                              f"spatial gate {op.name}")
            elif isinstance(op, GlobalLocalGateSpec):
                prm = op.packed()
                _lib.check_id(lib.stcd_plan_add_global_local_gate(h, ids[op.src], ids[op.dst], op.c, _fptr(prm)), f"global-local gate {op.name}")
            elif isinstance(op, CsamGateSpec):
                prm = op.packed()
                _lib.check_id(lib.stcd_plan_add_csam_gate(h, ids[op.src], ids[op.dst], op.c, op.l1.shape[0], _fptr(prm)), f"csam gate {op.name}")
            elif isinstance(op, VffmSpec):
                prm = op.packed()
                _lib.check_id(lib.stcd_plan_add_vffm(h, ids[op.low], ids[op.high], ids[op.mixed], ids[op.local], ids[op.dst], op.c, op.inter,
                                                     _fptr(prm)), f"VFFM {op.name}")
            elif isinstance(op, SumSpec):
                arr = (C.c_int * len(op.srcs))(*[ids[s_] for s_ in op.srcs])
                _lib.check_id(lib.stcd_plan_add_sum(h, arr, len(op.srcs), ids[op.dst]), f"sum {op.name}")
            elif isinstance(op, LayerNormSpec):
                g, b = np.ascontiguousarray(op.gamma, np.float32), np.ascontiguousarray(op.beta, np.float32)
                _lib.check_id(lib.stcd_plan_add_layernorm(h, ids[op.src], ids[op.dst], -1 if op.dst_s2d is None else ids[op.dst_s2d], op.c,
                                                          _fptr(g), _fptr(b), float(op.eps)), f"layer norm {op.name}")
            elif isinstance(op, AttentionSpec):
                _lib.check_id(lib.stcd_plan_add_sr_attention(h, ids[op.q], ids[op.kv], ids[op.dst], op.c, op.heads, float(op.scale)),
                              f"attention {op.name}")
            elif isinstance(op, DWConvSpec):
                wt, b = np.ascontiguousarray(op.weight, np.float32), np.ascontiguousarray(op.bias, np.float32)
                _lib.check_id(lib.stcd_plan_add_dwconv3x3(h, ids[op.src], ids[op.dst], op.c, _fptr(wt), _fptr(b), 1 if op.gelu else 0),
                              f"dw conv {op.name}")
            elif isinstance(op, BilinearUpSpec):
                _lib.check_id(lib.stcd_plan_add_bilinear_up(h, ids[op.src], ids[op.dst], op.c, op.scale), f"bilinear {op.name}")
            elif isinstance(op, MaxPoolS2DSpec):
                _lib.check_id(lib.stcd_plan_add_maxpool_s2d(h, ids[op.src], ids[op.dst], op.c), f"maxpool {op.name}")
            elif isinstance(op, SegHeadSpec):
                d = _lib.SegHeadDesc()
                d.src, d.c, d.bias, d.out_ext = ids[op.src], op.c, float(op.bias), op.out_ext
                d.diff_src = -1 if op.diff_src is None else ids[op.diff_src]
                wkeep = np.ascontiguousarray(op.weight, np.float32)
                d.weight = _fptr(wkeep)
                _lib.check_id(lib.stcd_plan_add_seg_head(h, C.byref(d)), f"seg head {op.name}")
            elif isinstance(op, ConvSpec):
                self._add_conv(op)
            elif isinstance(op, EcamHeadSpec):
                self._add_ecam(op)
            else:
                raise TypeError(f"unknown op {op!r}")
        if self.device < 0:
            return
        _lib.check(lib.stcd_plan_finalize(h), "stcd_plan_finalize")
        for name, val in prog.consts.items():          # constant tensors: the same [h, w, c] block for every image
            t = prog.tensors[name]
            full = torch.zeros(t.mult * self.chunk, t.h, t.w, t.c)
            full[..., : val.shape[2]] = val.to(torch.float32)[None]
            self.write_tensor(name, full)

    def _add_conv(self, op: ConvSpec) -> None:
        ids = self.tensor_ids
        d = _lib.ConvDesc()
        d.n_src = len(op.srcs)
        for i, s in enumerate(op.srcs):
            d.src[i] = ids[s]
            d.src_sy[i] = op.src_sy[i]
            d.src_sx[i] = op.src_sx[i]
            d.src_ey[i] = op.src_ey[i]
            d.src_ex[i] = op.src_ex[i]
        d.hg, d.wg = op.hg, op.wg
        d.img_mult = op.img_mult
        d.pair = 1 if op.pair else 0
        w = np.ascontiguousarray(op.weights, dtype=np.uint16)
        d.weights = w.ctypes.data_as(C.POINTER(C.c_uint16))
        d.w_elems = w.size
        d.kc, d.n_tile, d.cout, d.cout_pad = op.kc, op.n_tile, op.cout, op.cout_pad
        d.n_phase = len(op.phases)
        for i, ph in enumerate(op.phases):
            d.phase[i] = _lib.Phase(ph.chunk_begin, ph.chunk_count, ph.oy, ph.ox, ph.w_block, ph.n_blocks)
        ck = (_lib.Chunk * len(op.chunks))()
        for i, e in enumerate(op.chunks):
            ck[i] = _lib.Chunk(e.src, e.c0, e.by, e.bx, e.stream * self.chunk, e.tap_begin, e.n_taps)
        d.chunks = C.cast(ck, C.POINTER(_lib.Chunk))
        d.n_chunks = len(op.chunks)
        tp = (_lib.Tap * len(op.taps))()
        for i, (ty, tx) in enumerate(op.taps):
            tp[i] = _lib.Tap(ty, tx)
        d.taps = C.cast(tp, C.POINTER(_lib.Tap))
        d.n_taps = len(op.taps)
        d.osy, d.osx = op.osy, op.osx
        keep = [np.ascontiguousarray(op.scale, np.float32), np.ascontiguousarray(op.shift, np.float32),
                None if op.scale2 is None else np.ascontiguousarray(op.scale2, np.float32),
                None if op.shift2 is None else np.ascontiguousarray(op.shift2, np.float32)]
        d.scale, d.shift, d.scale2, d.shift2 = (_fptr(a) for a in keep)
        d.relu = op.act_kind if op.act_kind else (1 if op.relu else 0)
        d.act_pre, d.act_alpha = (1 if op.act_pre else 0), float(op.act_alpha)
        tid = lambda n: -1 if n is None else ids[n]  # noqa: E731
        d.res = tid(op.res)
        d.out0, d.out0_coff = tid(op.out0), op.out0_coff
        d.out_raw, d.out_pool, d.out_diff = tid(op.out_raw), tid(op.out_pool), tid(op.out_diff)
        d.out_ext = op.out_ext
        d.out0_s2d = 1 if op.out0_s2d else 0
        d.fold_cs, d.fold_cout = op.fold_cs, op.fold_cout
        d.xf_cs = op.xf_cs
        _lib.check_id(self.lib.stcd_plan_add_conv(self._h, C.byref(d)), f"conv {op.name}")

    def _add_ecam(self, op: EcamHeadSpec) -> None:
        d = _lib.EcamDesc()
        for i, s in enumerate(op.srcs):
            d.src[i] = self.tensor_ids[s]
        d.c, d.n_class = op.c, op.n_class
        d.r, d.r1 = op.ca_fc1.shape[0], op.ca1_fc1.shape[0]
        keep = [np.ascontiguousarray(a, np.float32) for a in
                (op.ca_fc1, op.ca_fc2, op.ca1_fc1, op.ca1_fc2, op.w_final, op.b_final)]
        d.ca_fc1, d.ca_fc2, d.ca1_fc1, d.ca1_fc2, d.w_final, d.b_final = (_fptr(a) for a in keep)
        d.out_ext = op.out_ext
        _lib.check_id(self.lib.stcd_plan_add_ecam_head(self._h, C.byref(d)), f"ecam head {op.name}")

    # ------------------------------------------------------------------ queries
    @property
    def workspace_bytes(self) -> int:
        return int(self.lib.stcd_plan_workspace_bytes(self._h))

    def launches(self, n_pairs: int) -> int:
        return int(self.lib.stcd_plan_launches(self._h, int(n_pairs)))

    def out_shapes(self, n_pairs: int) -> List[tuple]:
        return [(n_pairs, e.channels, e.h, e.w) for e in self.prog.ext]

    # ------------------------------------------------------------------ execution
    def _check_inputs(self, x1: torch.Tensor, x2: torch.Tensor) -> int:
        p = self.prog
        if x1.shape != x2.shape:
            raise ValueError(f"x1 {tuple(x1.shape)} and x2 {tuple(x2.shape)} differ")
        if self.u8:
            if x1.dim() != 4 or tuple(x1.shape[1:]) != (p.h, p.w, p.in_channels):
                raise ValueError(f"plan was built for uint8 [B,{p.h},{p.w},{p.in_channels}] (HWC) inputs, got {tuple(x1.shape)}")
            if x1.dtype != torch.uint8 or x2.dtype != torch.uint8:
                raise TypeError("this plan takes uint8 HWC images (the decoded RGB the reference's loader starts from)")
            return int(x1.shape[0])
        if x1.dim() != 4 or tuple(x1.shape[1:]) != (p.in_channels, p.h, p.w):
            raise ValueError(f"plan was built for [B,{p.in_channels},{p.h},{p.w}] inputs, got {tuple(x1.shape)}")
        if x1.dtype != torch.float32 or x2.dtype != torch.float32:
            raise TypeError("inputs must be float32 (the reference's input dtype: data/dataset.py:196-203)")
        return int(x1.shape[0])

    def forward(self, x1: torch.Tensor, x2: torch.Tensor, outs: Optional[Sequence[torch.Tensor]] = None
                ) -> List[torch.Tensor]:
        """Device tensors in, device fp32 NCHW tensors out; asynchronous on torch's current stream."""
        n = self._check_inputs(x1, x2)
        if not x1.is_cuda or not x2.is_cuda or x1.device.index != self.device or x2.device.index != self.device:
            raise ValueError(f"inputs must live on cuda:{self.device}")
        x1 = x1.contiguous()
        x2 = x2.contiguous()
        if outs is None:
            outs = [torch.empty(s, dtype=torch.float32, device=x1.device) for s in self.out_shapes(n)]
        ptrs = (C.c_void_p * len(outs))(*[o.data_ptr() for o in outs])
        stream = torch.cuda.current_stream(x1.device).cuda_stream
        fwd = self.lib.stcd_forward_u8 if self.u8 else self.lib.stcd_forward
        _lib.check(fwd(self._h, x1.data_ptr(), x2.data_ptr(), n, ptrs, len(outs), C.c_void_p(stream)), "stcd_forward")
        return list(outs)

    def forward_host(self, x1: torch.Tensor, x2: torch.Tensor, outs: Optional[Sequence[torch.Tensor]] = None
                     ) -> List[torch.Tensor]:
        """Host (ideally pinned) tensors in, host tensors out; blocks until the results have landed."""
        n = self._check_inputs(x1, x2)
        if x1.is_cuda or x2.is_cuda:
            raise ValueError("forward_host takes host tensors")
        x1 = x1.contiguous()
        x2 = x2.contiguous()
        if outs is None:
            outs = [torch.empty(s, dtype=torch.float32).pin_memory() for s in self.out_shapes(n)]
        ptrs = (C.c_void_p * len(outs))(*[o.data_ptr() for o in outs])
        fwd = self.lib.stcd_forward_host_u8 if self.u8 else self.lib.stcd_forward_host
        _lib.check(fwd(self._h, x1.data_ptr(), x2.data_ptr(), n, ptrs, len(outs)), "stcd_forward_host")
        return list(outs)

    def profile(self, x1: torch.Tensor, x2: torch.Tensor) -> List[tuple]:
        """Measurement pass: [(op name, ms, reference-equivalent MACs for this batch)] per op, device
        time from CUDA events around every launch (summed over chunks)."""
        n = self._check_inputs(x1, x2)
        outs = [torch.empty(s, dtype=torch.float32, device=x1.device) for s in self.out_shapes(n)]
        ptrs = (C.c_void_p * max(1, len(outs)))(*[o.data_ptr() for o in outs])
        n_ops = len(self.prog.ops)
        ms = (C.c_float * n_ops)()
        stream = torch.cuda.current_stream(x1.device).cuda_stream
        _lib.check(self.lib.stcd_forward_profile(self._h, x1.data_ptr(), x2.data_ptr(), n, ptrs, len(outs),
                                                 C.c_void_p(stream), ms, n_ops), "stcd_forward_profile")
        return [(op.name, float(ms[i]), int(getattr(op, "macs_per_pair", 0)) * n) for i, op in enumerate(self.prog.ops)]

    # ------------------------------------------------------------------ diagnostics
    def read_tensor(self, name: str) -> torch.Tensor:
        """Activation tensor `name` as fp32 logical NHWC [mult*chunk, h, w, c] on the host (synchronous)."""
        t = self.prog.tensors[name]
        buf = torch.empty(t.mult * self.chunk, t.c // 8, t.h, t.w, 8, dtype=torch.bfloat16)   # device layout
        _lib.check(self.lib.stcd_plan_tensor_copy(self._h, self.tensor_ids[name], C.c_void_p(buf.data_ptr()),
                                                  buf.numel() * 2, 0), f"read tensor {name}")
        return buf.permute(0, 2, 3, 1, 4).reshape(t.mult * self.chunk, t.h, t.w, t.c).to(torch.float32)

    def write_tensor(self, name: str, value: torch.Tensor) -> None:
        t = self.prog.tensors[name]
        if tuple(value.shape) != (t.mult * self.chunk, t.h, t.w, t.c):
            raise ValueError(f"tensor {name} is {(t.mult * self.chunk, t.h, t.w, t.c)}, got {tuple(value.shape)}")
        buf = value.to(torch.bfloat16).reshape(t.mult * self.chunk, t.h, t.w, t.c // 8, 8).permute(0, 3, 1, 2, 4).contiguous()
        _lib.check(self.lib.stcd_plan_tensor_copy(self._h, self.tensor_ids[name], C.c_void_p(buf.data_ptr()),
                                                  buf.numel() * 2, 1), f"write tensor {name}")

    def run_raw(self, n_valid: Optional[int] = None) -> List[torch.Tensor]:
        """Run the op list on whatever the activation tensors hold (programs without an input
        pack op: layer-wise tests).  Returns the external outputs (device tensors)."""
        n = self.chunk if n_valid is None else n_valid
        dev = torch.device("cuda", self.device)
        outs = [torch.empty(s, dtype=torch.float32, device=dev) for s in self.out_shapes(n)]
        ptrs = (C.c_void_p * max(1, len(outs)))(*[o.data_ptr() for o in outs])
        dummy = torch.zeros(16, dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(self.lib.stcd_forward(self._h, dummy.data_ptr(), dummy.data_ptr(), n, ptrs, len(outs),
                                         C.c_void_p(stream)), "stcd_forward")
        torch.cuda.synchronize(dev)
        return outs

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.stcd_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass
