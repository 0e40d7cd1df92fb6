"""ChangeFormerV6 on the precision path (``net.precision = "tf32"``: split-bf16 operands, lowering.Program.precision) without a
GPU: the split program through the emulator against the fp32 oracle, the K partitioning of the split convs whose K-programs
outgrow the conv kernel's tables, and the library's own descriptor checks on the program (validation plans)."""
import pytest
import torch

import emulate_split as emulate
from oracle import nets
from stcd_b200 import _lib, changeformer, changevig, lowering as L, synth

TF32_TOL = 1e-3
GAIN = 0.6                   # full-resolution logit std 0.38 (the registry gain of 0.5 gives 0.158)
# split ops whose K-program exceeds MAX_CHUNKS / MAX_TAPS: the 7x7 stride-4 patch embedding (one strided box per tap), the
# 8x8 stride-8 spatial reductions of stage 1, the 7x7 stride-2 patch embedding over 4 x 320 space-to-depth channels
PARTITIONED = {"Tenc_x2.patch_embed1.proj", "Tenc_x2.block1.0.attn.sr", "Tenc_x2.block1.1.attn.sr", "Tenc_x2.block1.2.attn.sr",
               "Tenc_x2.patch_embed4.proj"}


def _net(precision: str, gain: float = GAIN):
    net = synth.randomize_(changeformer.ChangeFormerV6().eval(), gain=gain)
    net.precision = precision
    return net


def _split_kinds():
    return (L.ConvSpec, L.InputPackSpec, L.LayerNormSpec, L.AttentionSpec, L.DWConvSpec, L.BilinearUpSpec)


def test_split_program_meets_1e3():
    net = _net("tf32")
    x1, x2 = synth.image_pairs(1, 256, 256)
    with torch.no_grad():
        ref = nets.changeformer_forward(net.state_dict(), x1, x2)
    prog = net.lower(256, 256)
    assert prog.split
    assert all(o.split for o in prog.ops if isinstance(o, _split_kinds()))
    assert {type(o) for o in prog.ops} <= set(_split_kinds())          # nothing without a split form
    ys = emulate.run_program(prog, x1, x2, chunk=1)
    assert len(ys) == 5
    for y, r in zip(ys, ref):
        assert y.shape == r.shape and (y - r).abs().max().item() < TF32_TOL
    y, r = ys[-1], ref[-1]
    assert r.std().item() >= 0.25, r.std().item()
    assert (y - r).abs().max().item() < 2e-4                         # 16-bit operand mantissas
    margin = (r[:, 1] - r[:, 0]).abs()
    agree = ((y[:, 1] > y[:, 0]) == (r[:, 1] > r[:, 0]))[margin > TF32_TOL]
    assert agree.all()
    assert 0.02 < (r[:, 1] > r[:, 0]).float().mean().item() < 0.98, "degenerate change map"


def test_k_partitioning():
    prog = _net("tf32").lower(256, 256)
    convs = [o for o in prog.ops if isinstance(o, L.ConvSpec)]
    for o in convs:
        for ph in o.phases:
            assert ph.chunk_count <= L.MAX_CHUNKS and ph.n_blocks <= L.MAX_TAPS, o.name
    parts = [o for o in convs if ".part" in o.name]
    assert {o.name.rsplit(".part", 1)[0] for o in parts} == PARTITIONED
    assert len(parts) == len(PARTITIONED)                            # two launches each
    by_name = {o.name: o for o in convs}
    for name in PARTITIONED:
        first, last = by_name[f"{name}.part0"], by_name[name]
        # the first launch: acc * scale into the split intermediate; the last: + shift + partial
        assert first.out0 == f"{name}.part0" and first.res is None and not first.relu and not first.shift.any()
        assert last.res == f"{name}.part0" and first.macs_per_pair == 0 and last.macs_per_pair > 0
        assert prog.tensors[first.out0].c == 2 * last.cout
    assert abs(2 * prog.macs_per_pair() / 1e9 - 277.459) < 0.01      # the same reference MACs as the bf16 program

    bf = _net("bf16").lower(256, 256)
    assert not bf.split and not any(".part" in n for n in bf.tensors)
    assert sum(isinstance(o, L.AttentionSpec) for o in bf.ops) == 13 and sum(isinstance(o, L.LayerNormSpec) for o in bf.ops) == 44
    assert not any(getattr(o, "split", False) for o in bf.ops)
    split_convs = [o.name for o in convs if ".part" not in o.name]
    assert split_convs == [o.name for o in bf.ops if isinstance(o, L.ConvSpec)]


def test_partitioning_refuses_other_epilogues():
    prog = L.Program(model="t", in_channels=8, h=64, w=64, precision="split")
    src = prog.tensor("src", 2, 64, 64, 64)
    dst = prog.tensor("dst", 2, 8, 8, 64)
    res = prog.tensor("res", 2, 8, 8, 64)
    wt = torch.randn(64, 64, 8, 8)
    ones = torch.ones(64).numpy()
    with pytest.raises(NotImplementedError, match="bad.sr"):
        L.add_conv(prog, "bad.sr", [L.Segment(src, 64, sy=8, sx=8)], L.conv_taps(wt, pad=0), 64, 8, 8, 1, ones, 0 * ones, pair=True,
                   res=res, out0=dst)
    L.add_conv(prog, "ok.sr", [L.Segment(src, 64, sy=8, sx=8)], L.conv_taps(wt, pad=0), 64, 8, 8, 1, ones, 0 * ones, pair=True, out0=dst)
    assert [o.name for o in prog.ops] == ["ok.sr.part0", "ok.sr"]


@pytest.mark.parametrize("chunk", [1, 4])
def test_split_program_passes_the_library_checks(chunk):
    from stcd_b200.plan import Plan
    prog = _net("tf32", synth.GAINS["ChangeFormerV6"]).lower(256, 256)
    plan = Plan(prog, chunk, device=-1)
    lib = _lib.lib()
    assert lib.stcd_plan_finalize(plan._h) == 3                        # STCD_ERR_NO_DEVICE: validated, nothing can run
    plan.close()


def test_split_plan_rejects_bad_tensors():
    """In a split plan the bandwidth ops need tensors that store twice their logical channels; attention needs exactly 64
    keys."""
    import ctypes as C
    import numpy as np
    lib = _lib.lib()
    h = C.c_void_p()
    _lib.check(lib.stcd_plan_create(-1, 1, _lib.PRECISION_SPLIT, C.byref(h)), "create")
    try:
        t = lambda mult, hh, ww, c: lib.stcd_plan_add_tensor(h, mult, hh, ww, c, 0)  # noqa: E731
        one, two = t(2, 16, 16, 64), t(2, 16, 16, 128)
        g = np.ones(64, np.float32)
        gp = g.ctypes.data_as(C.POINTER(C.c_float))
        w9 = np.ones(64 * 9, np.float32).ctypes.data_as(C.POINTER(C.c_float))
        assert lib.stcd_plan_add_layernorm(h, one, two, -1, 64, gp, gp, 1e-6) < 0
        assert lib.stcd_plan_add_layernorm(h, two, two, -1, 64, gp, gp, 1e-6) >= 0
        assert lib.stcd_plan_add_dwconv3x3(h, two, one, 64, w9, gp, 1) < 0
        assert lib.stcd_plan_add_dwconv3x3(h, two, two, 64, w9, gp, 1) >= 0
        up = t(2, 32, 32, 128)
        assert lib.stcd_plan_add_bilinear_up(h, one, up, 64, 2) < 0
        assert lib.stcd_plan_add_bilinear_up(h, two, up, 64, 2) >= 0
        kv64, kv16 = t(2, 8, 8, 256), t(2, 4, 4, 256)
        assert lib.stcd_plan_add_sr_attention(h, two, kv16, two, 64, 1, 0.125) < 0          # 16 keys
        assert lib.stcd_plan_add_sr_attention(h, one, kv64, one, 64, 1, 0.125) < 0          # single-plane q / dst
        assert lib.stcd_plan_add_sr_attention(h, two, kv64, two, 64, 1, 0.125) >= 0
    finally:
        lib.stcd_plan_destroy(h)


@pytest.mark.parametrize("cls", ["ChangeFormerV1", "ChangeFormerV2", "ChangeFormerV3"])
def test_families_sharing_the_lowering_still_refuse_tf32(cls):
    net = getattr(changeformer, cls)().eval()
    net.precision = "tf32"
    with pytest.raises(NotImplementedError):
        net.plan_precision
    gnn = changevig.ChangeGNNV1().eval()
    gnn.precision = "tf32"
    with pytest.raises(NotImplementedError):
        gnn.plan_precision
