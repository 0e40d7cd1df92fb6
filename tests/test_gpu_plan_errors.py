"""Error behaviour of the plan-building entry points added for the DTCDSCN / BIT / IFNet / ChangeGNNV2 / GNN ops: a bad
argument is a negative return code with a message in stcd_last_error(), never a crash, and it leaves the plan usable."""
import ctypes as C

import numpy as np
import pytest

from stcd_b200 import _lib

pytestmark = pytest.mark.gpu


def _f(a):
    return np.ascontiguousarray(a, np.float32).ctypes.data_as(C.POINTER(C.c_float))


def test_bf16_plan_ops_reject_bad_arguments():
    lib = _lib.lib()
    h = C.c_void_p()
    _lib.check(lib.stcd_plan_create(0, 2, _lib.PRECISION_BF16, C.byref(h)), "stcd_plan_create")
    try:
        pair32 = _lib.check_id(lib.stcd_plan_add_tensor(h, 2, 16, 16, 32, 0), "tensor")       # [2*chunk, 16, 16, 32]
        one32 = _lib.check_id(lib.stcd_plan_add_tensor(h, 1, 16, 16, 32, 0), "tensor")
        one64 = _lib.check_id(lib.stcd_plan_add_tensor(h, 1, 16, 16, 64, 0), "tensor")
        one32b = _lib.check_id(lib.stcd_plan_add_tensor(h, 1, 16, 16, 32, 0), "tensor")
        small = _lib.check_id(lib.stcd_plan_add_tensor(h, 1, 8, 8, 32, 0), "tensor")
        z = np.zeros(1 << 16, np.float32)

        def bad(rc, needle):
            assert rc < 0, "expected an error code"
            msg = lib.stcd_last_error().decode()
            assert needle in msg, msg

        # signed difference: the addend must have the destination's shape
        bad(lib.stcd_plan_add_subdiff(h, pair32, small, one32), "addend")
        bad(lib.stcd_plan_add_subdiff(h, pair32, 99, one32), "tensor id")
        # channel gate: c not a multiple of 8, too many hidden units, NULL weights, space-to-depth copy of the wrong shape
        bad(lib.stcd_plan_add_channel_gate(h, one32, -1, one32b, -1, 12, 2, _f(z), _f(z), None, 0), "channel gate")
        bad(lib.stcd_plan_add_channel_gate(h, one32, -1, one32b, -1, 32, 64, _f(z), _f(z), None, 0), "channel gate")
        bad(lib.stcd_plan_add_channel_gate(h, one32, -1, one32b, -1, 32, 2, None, _f(z), None, 0), "channel gate")
        bad(lib.stcd_plan_add_channel_gate(h, one32, -1, one32b, one64, 32, 2, _f(z), _f(z), None, 0), "space-to-depth")
        bad(lib.stcd_plan_add_channel_gate(h, one32, -1, one32b, -1, 32, 2, _f(z), _f(z), None, 1), "channel gate")     # mode 1 needs ws
        # sum: shapes must agree, 1..5 sources
        srcs = (C.c_int * 2)(one32, one64)
        bad(lib.stcd_plan_add_sum(h, srcs, 2, one32b), "shapes differ")
        bad(lib.stcd_plan_add_sum(h, srcs, 0, one32b), "1..5")
        # BIT token path: only c = 32, token_len = 4, heads = 8, mlp = 64; both tensors must hold both streams
        d = _lib.BitDesc()
        d.c, d.token_len, d.heads, d.mlp, d.n_enc, d.n_dec, d.inner_enc, d.inner_dec, d.softmax = 32, 4, 8, 64, 1, 1, 512, 512, 1
        d.conv_a = d.pos = d.enc = d.dec = _f(z)
        bad(lib.stcd_plan_add_bit_transformer(h, one32, one32b, C.byref(d)), "both streams")
        d.token_len = 8
        bad(lib.stcd_plan_add_bit_transformer(h, pair32, pair32, C.byref(d)), "32 / 4 / 8 / 64")
        d.token_len, d.n_dec = 4, 0
        bad(lib.stcd_plan_add_bit_transformer(h, pair32, pair32, C.byref(d)), "depths")
        # channel attention: the destination must hold exactly the concatenated channels; streams must exist
        ts, ss, cs = (C.c_int * 2)(one32, pair32), (C.c_int * 2)(0, 1), (C.c_int * 2)(32, 32)
        bad(lib.stcd_plan_add_channel_attention(h, ts, ss, cs, 2, one32b, 8, _f(z), _f(z)), "dst must be")
        ss_bad = (C.c_int * 2)(1, 1)                                  # stream 1 of a one-stream tensor
        bad(lib.stcd_plan_add_channel_attention(h, ts, ss_bad, cs, 2, one64, 8, _f(z), _f(z)), "source 0")
        # spatial gate / global-local gate / csam gate / VFFM: shape and size checks
        bad(lib.stcd_plan_add_spatial_gate(h, one32, one64, 48, _f(z), _f(z), _f(z)), "spatial gate")
        bad(lib.stcd_plan_add_global_local_gate(h, one32, small, 32, _f(z)), "global-local gate")
        bad(lib.stcd_plan_add_csam_gate(h, one32, one32b, 32, 0, _f(z)), "hid")
        bad(lib.stcd_plan_add_vffm(h, one32, one32b, one32, one64, one32b, 32, 8, _f(z)), "VFFM")
        bad(lib.stcd_plan_add_vffm(h, one32, one32b, one32, one32, one32b, 32, 500, _f(z)), "VFFM")
        # the plan is still usable: valid ops go in and it finalizes
        assert lib.stcd_plan_add_subdiff(h, pair32, -1, one32) >= 0
        assert lib.stcd_plan_add_spatial_gate(h, one32, one32b, 32, _f(z), _f(np.ones(32)), _f(z)) >= 0
        _lib.check(lib.stcd_plan_finalize(h), "stcd_plan_finalize")
        # ... and refuses further ops once finalized
        bad(lib.stcd_plan_add_subdiff(h, pair32, -1, one32), "finalized")
    finally:
        lib.stcd_plan_destroy(h)
