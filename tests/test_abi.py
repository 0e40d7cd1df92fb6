"""The C-ABI library loads and exports every symbol include/stcd_b200.h declares; without a GPU
every compute entry point fails loudly (no CPU fallback)."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

from stcd_b200 import _lib


def _declared_symbols():
    text = _lib.HEADER.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(stcd_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_header_symbols():
    lib = _lib.lib()
    declared = _declared_symbols()
    assert len(declared) >= 14
    bound = {n for n, _, _ in _lib.SYMBOLS}
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/stcd_b200.h but not exported"
        assert name in bound, f"{name} has no ctypes signature in stcd_b200/_lib.py"
    assert lib.stcd_abi_version() == _lib.ABI_VERSION


def test_struct_layouts_match_header():
    # sizes the C side static_asserts / validates; a drifted ctypes mirror corrupts plans silently
    assert C.sizeof(_lib.Chunk) == 16 and C.sizeof(_lib.Tap) == 4
    assert C.sizeof(_lib.Phase) == 24


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_gpu_fails_loudly_at_either_precision():
    lib = _lib.lib()
    assert lib.stcd_device_count() == 0
    h = C.c_void_p()
    for precision in (_lib.PRECISION_BF16, _lib.PRECISION_SPLIT):
        rc = lib.stcd_plan_create(0, 4, precision, C.byref(h))
        assert rc == 3 and not h.value          # STCD_ERR_NO_DEVICE
        assert b"no CPU fallback" in lib.stcd_last_error()
    cm = (C.c_int64 * 4)()
    buf = (C.c_uint8 * 16)()
    rc = lib.stcd_confusion_add_batch(buf, 3, 0.0, buf, 1, 1, 16, 2, cm, None, None)
    assert rc == 3
    from stcd_b200.metric import SegmentationMetric
    with pytest.raises(_lib.StcdError):
        SegmentationMetric(2)


def test_argument_validation_without_gpu():
    lib = _lib.lib()
    cm = (C.c_int64 * 4)()
    buf = (C.c_uint8 * 16)()
    assert lib.stcd_confusion_add_batch(None, 3, 0.0, buf, 1, 1, 16, 2, cm, None, None) == 1
    assert lib.stcd_confusion_add_batch(buf, 9, 0.0, buf, 1, 1, 16, 2, cm, None, None) == 1
    assert lib.stcd_confusion_add_batch(buf, 0, 0.0, buf, 1, 1, 16, 3, cm, None, None) == 1
    assert lib.stcd_forward(None, None, None, 1, None, 0, None) == 4      # STCD_ERR_STATE


def test_plan_precision():
    """The precision is declared once, for the whole plan: a split plan declares only two-plane tensors (channels a multiple
    of 16) and refuses the ops that have no split form, all of which a bf16 plan accepts."""
    lib = _lib.lib()
    h = C.c_void_p()
    for bad in (-1, 2):
        assert lib.stcd_plan_create(-1, 1, bad, C.byref(h)) == 1 and not h.value     # STCD_ERR_INVALID
        assert b"precision" in lib.stcd_last_error()
    z, ones = np.zeros(1 << 16, np.float32), np.ones(16, np.float32)
    f = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    for precision in (_lib.PRECISION_BF16, _lib.PRECISION_SPLIT):
        split = precision == _lib.PRECISION_SPLIT
        _lib.check(lib.stcd_plan_create(-1, 1, precision, C.byref(h)), "create")
        try:
            t = lambda mult, c: lib.stcd_plan_add_tensor(h, mult, 16, 16, c, 0)  # noqa: E731
            assert (t(1, 24) < 0) == split
            a, b, c = t(1, 32), t(1, 32), t(1, 32)
            pair16 = t(2, 16)
            seg = _lib.SegHeadDesc(pair16, 16, f(z), 0.0, 0, -1)
            calls = [
                ("graph conv", lambda: lib.stcd_plan_add_graph_conv(h, a, b, 32, 9, 1, 1, None)),
                ("channel attention", lambda: lib.stcd_plan_add_channel_attention(h, (C.c_int * 1)(a), (C.c_int * 1)(0), (C.c_int * 1)(32),
                                                                                  1, b, 8, f(z), f(z))),
                ("spatial gate", lambda: lib.stcd_plan_add_spatial_gate(h, a, b, 32, f(z), f(ones), f(z))),
                ("global-local gate", lambda: lib.stcd_plan_add_global_local_gate(h, a, b, 32, f(z))),
                ("csam gate", lambda: lib.stcd_plan_add_csam_gate(h, a, b, 32, 8, f(z))),
                ("VFFM", lambda: lib.stcd_plan_add_vffm(h, a, b, a, b, c, 32, 8, f(z))),
                ("seg head", lambda: lib.stcd_plan_add_seg_head(h, C.byref(seg))),
                ("uint8 input pack", lambda: lib.stcd_plan_add_input_pack_u8(h, pair16, 3, 0, f(z), f(ones))),
            ]
            for name, call in calls:
                rc = call()
                if split:
                    assert rc < 0 and f"{name} has no split form" in lib.stcd_last_error().decode(), name
                else:
                    assert rc >= 0, (name, lib.stcd_last_error())
        finally:
            lib.stcd_plan_destroy(h)


# every registry family at a small legal size: the library's own descriptor checks run on the lowered programs without a
# GPU (a validation plan, device -1), so a lowering change that the C side rejects fails HERE, not on the GPU box
_VALIDATE = [
    ("SiamUnet_diff", (3, 2), 64, 64), ("SiamUnet_conc", (3, 2), 64, 64), ("SiamUnet_sub", (3, 2), 32, 48),
    ("SiamUnet_cross_conc", (3, 2), 48, 32), ("Unet", (3, 2), 32, 32), ("SNUNet_ECAM", (3, 2), 64, 96),
    ("SegCD", ("resnet34",), 64, 96), ("CDNet_model", (3,), 64, 96), ("DSIFN", (), 64, 96),
    ("ChangeFormerV6", (3, 2, False, 256), 256, 256), ("ChangeGNNV1", (3, 2, False, 256), 256, 256),
    ("SiamUnet_diff", (3, 2), 256, 256), ("SNUNet_ECAM", (3, 2), 256, 256),
]
_VALIDATE_SPLIT = [("SiamUnet_diff", (3, 2), 64, 64), ("SiamUnet_conc", (3, 2), 64, 64), ("SNUNet_ECAM", (3, 2), 64, 96),
                   ("SiamUnet_diff", (3, 2), 256, 256), ("SNUNet_ECAM", (3, 2), 256, 256)]


@pytest.mark.parametrize("name,args,h,w,precision", [v + ("bf16",) for v in _VALIDATE] + [v + ("tf32",) for v in _VALIDATE_SPLIT],
                         ids=[f"{n}-{h}x{w}" for n, _, h, w in _VALIDATE] + [f"{n}-{h}x{w}-tf32" for n, _, h, w in _VALIDATE_SPLIT])
def test_lowered_programs_pass_the_library_checks(name, args, h, w, precision):
    from stcd_b200.networks import CLASSES
    from stcd_b200.plan import Plan
    net = CLASSES[name](*args).eval()
    net.precision = precision
    prog = net.lower(h, w)
    for chunk in (1, 4):
        plan = Plan(prog, chunk, device=-1)
        assert plan.launches(chunk) == 0 or plan.launches(chunk) > 0      # recorded, never finalized
        lib = _lib.lib()
        assert lib.stcd_plan_finalize(plan._h) == 3                        # STCD_ERR_NO_DEVICE: nothing can run
        assert b"no CPU fallback" in lib.stcd_last_error()
        plan.close()
