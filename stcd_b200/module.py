"""Shared plumbing of the drop-in ``nn.Module`` wrappers: plan caching and the eval-only contract.

A wrapper keeps the reference module's parameter names (so a reference ``state_dict`` loads) and
lowers itself to a libstcd_b200 plan per (device, H, W, chunk) on first use; anything that touches
the weights drops the packed copies: ``load_state_dict`` / ``.to`` / ``.cuda`` / re-initialisation
through ``networks.init_weights`` explicitly, and everything else (a child's ``load_state_dict``,
``p.data.copy_``, an EMA update, fine-tuning the same parameters elsewhere) through a fingerprint of
every parameter's and buffer's ``(data_ptr, _version)`` that is compared before each forward.

Plans hold ctypes handles of device objects: they are never copied or pickled.  ``copy.deepcopy(net)``
(train_stcd.py:81-87,326), ``torch.save(net)`` and ``pickle`` see a module without plans; the copy
lowers itself again on its first forward.
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn as nn

from . import lowering as L


class PlannedModule(nn.Module):
    #: image pairs per pass through the layer stack (one plan workspace holds this many)
    default_chunk_pairs = 32
    #: families whose lowering implements the split-precision path (``precision = "tf32"``)
    supports_precision_path = False
    #: "bf16" (default; north star: logits within 2e-2 of the fp32 reference) or "tf32" (north star: within 1e-3).  The
    #: reference computes in fp32 and its only numeric switch is cudnn.benchmark (train_stcd.py:59); "tf32" names the tolerance
    #: class the north star asks for, served by split-bf16 operands (lowering.Program.precision: 16 mantissa bits per operand,
    #: three bf16 MMAs per product) because plain tf32 MMAs miss 1e-3 on these nets.  Set it before the first forward or any
    #: time after: plans are cached per precision.
    precision = "bf16"

    @property
    def plan_precision(self) -> str:
        """The lowering's name for the selected precision ("bf16" or "split")."""
        if self.precision not in ("bf16", "tf32"):
            raise ValueError(f"precision must be 'bf16' or 'tf32', got {self.precision!r}")
        if self.precision == "tf32" and not self.supports_precision_path:
            raise NotImplementedError(f"{type(self).__name__} has no 'tf32' precision path (implemented: the FC-Siam family, SNUNet-CD, ChangeFormerV6, BIT and DTCDSCN)")
        return "split" if self.precision == "tf32" else "bf16"

    def __init__(self):
        super().__init__()
        self._plans: Dict[tuple, object] = {}
        self._fp_tensors = None      # parameters + buffers the cached plans were lowered from
        self._fp = None              # their fingerprint at lowering time
        self.chunk_pairs = self.default_chunk_pairs

    # weights changed (load_state_dict / .to / re-init): packed copies are stale
    def _apply(self, fn, *a, **k):
        self.invalidate_plans()
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self.invalidate_plans()
        return super().load_state_dict(*a, **k)

    def invalidate_plans(self) -> None:
        self._plans = {}
        self._fp_tensors = None
        self._fp = None

    # plans own device objects through ctypes handles: a copy / pickle of the module starts without them
    def __getstate__(self):
        state = self.__dict__.copy()
        state["_plans"] = {}
        state["_fp_tensors"] = None
        state["_fp"] = None
        return state

    def _weights_fingerprint(self):
        """(data_ptr, _version) over every parameter and buffer: changes on any in-place write (``copy_``, optimiser
        steps, a child's ``load_state_dict``) and on ``p.data = ...``.  The tensor list is cached with the plans."""
        ts = self._fp_tensors
        if ts is None:
            ts = self._fp_tensors = [t for t in list(self.parameters()) + list(self.buffers()) if t is not None]
        h = len(ts)
        for t in ts:
            h = (h * 1000003 + t._version * 31 + t.data_ptr()) & 0xFFFFFFFFFFFFFFFF
        return h

    def lower(self, h: int, w: int) -> L.Program:  # pragma: no cover - abstract
        raise NotImplementedError

    #: the reference loader's normalisation (CD_Dataset.MEAN / STD, data/dataset.py:171-172)
    IMAGENET_MEAN = (0.485, 0.456, 0.406)
    IMAGENET_STD = (0.229, 0.224, 0.225)

    @torch.no_grad()
    def forward_uint8(self, a: torch.Tensor, b: torch.Tensor, mean=None, std=None):
        """The same forward fed with the decoded uint8 HWC images ``[B, H, W, 3]`` the reference's loader starts
        from (data/dataset.py:196-203): ToTensor + Normalize run inside the input-pack kernel, bit-identical to
        ``self(normalize(a), normalize(b))`` at a quarter of the host-to-device bytes.  Returns what ``forward``
        returns."""
        norm = (tuple(mean or self.IMAGENET_MEAN), tuple(std or self.IMAGENET_STD))
        outs = self.plan_for(a, u8_norm=norm).forward(a, b)
        return self._wrap_outputs(outs)

    def _wrap_outputs(self, outs):
        return outs[0] if len(outs) == 1 else tuple(outs)

    def plan_for(self, x: torch.Tensor, u8_norm=None):
        from .plan import Plan
        if self.training:
            raise RuntimeError("stcd_b200 implements the eval-mode inference path; call .eval() first "
                               "(training stays with the reference, models/trainer.py)")
        if not x.is_cuda:
            raise RuntimeError("stcd_b200 has no CPU path: move the module and its inputs to a B200 (cuda) device")
        chunk = max(1, min(int(self.chunk_pairs), int(x.shape[0])))
        h, w = (int(x.shape[1]), int(x.shape[2])) if u8_norm is not None else (int(x.shape[2]), int(x.shape[3]))
        key = (x.device.index, h, w, chunk, u8_norm, self.plan_precision)
        if self._plans:
            if self._weights_fingerprint() != self._fp:     # weights were written since the plans were lowered
                self.invalidate_plans()
        plan = self._plans.get(key)
        if plan is None:
            prog = self.lower(h, w)
            if u8_norm is not None:
                for op in prog.ops:
                    if isinstance(op, L.InputPackSpec):
                        op.u8_norm = u8_norm
            plan = Plan(prog, chunk, device=key[0])
            if not self._plans:
                self._fp = self._weights_fingerprint()
            self._plans[key] = plan
        return plan
