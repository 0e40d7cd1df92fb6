"""BIT (BASE_Transformer s4 / dd8 / dd8_dedim8, the ResNet-18 baseline) and DTCDSCN on the precision path
(``net.precision = "tf32"``: split-bf16 operands, lowering.Program.precision) without a GPU: the split programs through the
emulator against the fp32 oracle, the bf16 programs left as they were, and the library's own descriptor checks (validation
plans, the split plan's tensor checks, split convs with a space-to-depth store)."""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

import emulate_split_resnet as emulate
from oracle import nets
from stcd_b200 import _lib, bit, dtcdscn, lowering as L, synth
from stcd_b200.plan import Plan

TF32_TOL = 1e-3
NETS = ["s4", "dd8", "dd8_dedim8", "resnet18", "dtcdscn"]
VARIANTS = {"s4": {}, "dd8": dict(enc_depth=1, dec_depth=8), "dd8_dedim8": dict(enc_depth=1, dec_depth=8, decoder_dim_head=8)}
# (weight gain, head scale, offset added to the class-0 head bias) per net: a full-resolution logit std near 0.3 with the class
# margin centred (a change fraction near one half) at 64 x 96.  The registry gains of synth.GAINS give a std of 0.04-0.09 here,
# too small for an absolute 1e-3 bound to mean anything.  Raising the gain of every layer instead puts the random ResNets in
# their chaotic range (the logit std grows ~10x per 0.1 of gain), where a perturbation of the input grows faster than the
# signal; scaling the head alone leaves the relative error of the network as it is.
WEIGHTS = {"s4": (0.6, 2.0, -0.23), "dd8": (0.6, 1.0, 0.95), "dd8_dedim8": (0.6, 1.15, -0.47), "resnet18": (0.6, 8.5, -0.40),
           "dtcdscn": (0.7, 1.0, 0.68)}


def make(name: str, precision: str = "tf32"):
    """The net `name` with this module's test weights, set to `precision`."""
    if name == "dtcdscn":
        net, head = dtcdscn.CDNet34(3, 2), "finalconv3_master.bias"
    elif name == "resnet18":
        net, head = bit.ResNet(3, 2), "classifier.3.bias"
    else:
        net = bit.BASE_Transformer(3, 2, with_pos="learned", resnet_stages_num=4, token_len=4, **VARIANTS[name])
        head = "classifier.3.bias"
    gain, scale, b0 = WEIGHTS[name]
    net = synth.randomize_(net.eval(), gain=gain)
    params = dict(net.named_parameters())
    with torch.no_grad():
        params[head.replace(".bias", ".weight")].mul_(scale)
        params[head].mul_(scale)[0] += b0
    net.precision = precision
    return net


def oracle(name: str, net, x1: torch.Tensor, x2: torch.Tensor) -> torch.Tensor:
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    with torch.no_grad():
        if name == "dtcdscn":
            return nets.dtcdscn_forward(sd, x1, x2)
        return nets.bit_forward(sd, x1, x2, stages=5 if name == "resnet18" else 4)


@pytest.mark.parametrize("name", NETS)
def test_split_program_meets_1e3(name):
    net = make(name)
    x1, x2 = synth.image_pairs(3, 64, 96)
    ref = oracle(name, net, x1, x2)
    prog = net.lower(64, 96)
    assert prog.split and all(op.split for op in prog.ops)              # every op type of these nets has a split form
    y = emulate.run_program(prog, x1, x2, chunk=2)[0]
    assert y.shape == ref.shape
    assert ref.std().item() >= 0.25, ref.std().item()
    assert 0.02 < (ref[:, 1] > ref[:, 0]).float().mean().item() < 0.98, "degenerate change map"
    err = (y - ref).abs().max().item()
    assert err < TF32_TOL and err < 2e-4, err                           # 16-bit operand mantissas
    margin = (ref[:, 1] - ref[:, 0]).abs()
    assert ((y[:, 1] > y[:, 0]) == (ref[:, 1] > ref[:, 0]))[margin > TF32_TOL].all()


@pytest.mark.parametrize("name", NETS)
def test_bf16_program_is_unchanged(name):
    bf, sp = make(name, "bf16").lower(64, 96), make(name).lower(64, 96)
    assert not bf.split and not any(getattr(op, "split", False) for op in bf.ops)
    assert [op.name for op in bf.ops] == [op.name for op in sp.ops]     # the split programs need no K partitioning
    assert {n: 2 * t.c for n, t in bf.tensors.items()} == {n: t.c for n, t in sp.tensors.items()}
    assert bf.macs_per_pair() == sp.macs_per_pair()


@pytest.mark.parametrize("chunk", [1, 4])
@pytest.mark.parametrize("name", ["dd8", "resnet18", "dtcdscn"])
def test_split_program_passes_the_library_checks(name, chunk):
    prog = make(name).lower(256, 256)
    for op in prog.ops:
        for ph in getattr(op, "phases", ()):
            assert ph.chunk_count <= L.MAX_CHUNKS and ph.n_blocks <= L.MAX_TAPS, op.name
    plan = Plan(prog, chunk, device=-1)
    assert _lib.lib().stcd_plan_finalize(plan._h) == 3                 # STCD_ERR_NO_DEVICE: validated, nothing can run
    plan.close()


def test_split_plan_rejects_single_plane_tensors():
    lib = _lib.lib()
    h = C.c_void_p()
    _lib.check(lib.stcd_plan_create(-1, 1, _lib.PRECISION_SPLIT, C.byref(h)), "create")
    try:
        t = lambda mult, hh, ww, c: lib.stcd_plan_add_tensor(h, mult, hh, ww, c, 0)  # noqa: E731
        f = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
        # input pack: 32 stored channels (hi [0, 16), lo [16, 32))
        assert lib.stcd_plan_add_input_pack_s2d(h, t(2, 16, 16, 16), 3) < 0
        assert lib.stcd_plan_add_input_pack_s2d(h, t(2, 16, 16, 32), 3) >= 0
        # max-pool: src 8c, dst 2c
        s4, s8, d1, d2 = t(2, 8, 8, 256), t(2, 8, 8, 512), t(2, 8, 8, 64), t(2, 8, 8, 128)
        assert lib.stcd_plan_add_maxpool_s2d(h, s4, d2, 64) < 0
        assert lib.stcd_plan_add_maxpool_s2d(h, s8, d1, 64) < 0
        assert lib.stcd_plan_add_maxpool_s2d(h, s8, d2, 64) >= 0
        # differences and sums: a split plan declares no tensor that cannot hold two planes of 8-channel groups
        assert t(2, 8, 8, 24) < 0 and t(1, 8, 8, 24) < 0
        a32, b32 = t(2, 8, 8, 32), t(1, 8, 8, 32)
        assert lib.stcd_plan_add_absdiff(h, a32, b32) >= 0
        assert lib.stcd_plan_add_subdiff(h, a32, t(1, 8, 8, 32), b32) >= 0
        assert lib.stcd_plan_add_sum(h, (C.c_int * 2)(b32, b32), 2, t(1, 8, 8, 32)) >= 0
        # SE gate: src / res / dst 2c, space-to-depth copy 8c
        w1, w2 = np.ones((4, 64), np.float32), np.ones((64, 4), np.float32)
        g1, g2, gs4, gs8 = t(2, 16, 16, 64), t(2, 16, 16, 128), t(2, 8, 8, 256), t(2, 8, 8, 512)
        gate = lambda src, res, dst, s2d: lib.stcd_plan_add_channel_gate(h, src, res, dst, s2d, 64, 4, f(w1), f(w2), None, 0)  # noqa: E731
        assert gate(g1, -1, g2, -1) < 0
        assert gate(g2, g1, g2, -1) < 0
        assert gate(g2, g2, g2, gs4) < 0
        assert gate(g2, g2, t(2, 16, 16, 128), gs8) >= 0
        # BIT token path: 64 stored channels
        d = _lib.BitDesc()
        d.c, d.token_len, d.heads, d.mlp, d.n_enc, d.n_dec, d.inner_enc, d.inner_dec, d.softmax = 32, 4, 8, 64, 1, 1, 64, 64, 1
        keep = [np.zeros(n, np.float32) for n in (4 * 32, 8 * 32, 100000, 100000)]
        d.conv_a, d.pos, d.enc, d.dec = (f(a) for a in keep)
        m32, m64 = t(2, 16, 16, 32), t(2, 16, 16, 64)
        assert lib.stcd_plan_add_bit_transformer(h, m32, m32, C.byref(d)) < 0
        assert lib.stcd_plan_add_bit_transformer(h, m64, t(2, 16, 16, 64), C.byref(d)) >= 0
    finally:
        lib.stcd_plan_destroy(h)


def _s2d_conv_program():
    """A split stride-1 3x3 conv + BN + residual + ReLU whose output is stored space-to-depth (BIT's layer1.1.conv2)."""
    g = torch.Generator().manual_seed(3)
    p = L.Program(model="t", in_channels=3, h=16, w=16, precision="split")
    x, res = p.tensor("x", 2, 16, 16, 32), p.tensor("res", 2, 16, 16, 32)
    o = p.tensor("o_s2d", 2, 8, 8, 4 * 32)
    wt = torch.randn(32, 32, 3, 3, generator=g) * 0.1
    sc, sh = (0.8 + 0.4 * torch.rand(32, generator=g)).numpy(), (0.1 * torch.randn(32, generator=g)).numpy()
    op = L.add_conv(p, "conv", [L.Segment(x, 32)], L.conv_taps(wt, pad=1), 32, 16, 16, 1, sc, sh, pair=True, relu=True, res=res,
                    out0=o, out0_s2d=True)
    return p, op, wt, sc, sh


def test_split_conv_with_space_to_depth_store():
    p, op, wt, sc, sh = _s2d_conv_program()
    assert op.split and op.out0_s2d and not op.fold_cs and not op.xf_cs
    assert p.tensors["o_s2d"].c == 8 * 32                              # 4 parity classes x (hi, lo)
    plan = Plan(p, 1, device=-1)                                        # accepted by the library
    plan.close()
    # the emulator's store against the fp32 conv: hi of class k at k*32, lo at 128 + k*32
    g = torch.Generator().manual_seed(4)
    x, r = torch.randn(2, 16, 16, 32, generator=g), torch.randn(2, 16, 16, 32, generator=g)
    T = {n: torch.zeros(t.mult, t.h, t.w, t.c) for n, t in p.tensors.items()}
    for name, v in (("x", x), ("res", r)):
        emulate.E._store(T, name, (slice(None), slice(None), slice(None)), 0, v, True)
    emulate.run_conv(op, T, 1, [], 1)
    xs = T["x"][..., :32] + T["x"][..., 32:]
    want = torch.nn.functional.conv2d(xs.permute(0, 3, 1, 2), wt, padding=1).permute(0, 2, 3, 1)
    want = torch.relu(want * torch.from_numpy(sc) + torch.from_numpy(sh) + T["res"][..., :32] + T["res"][..., 32:])
    got = T["o_s2d"]
    for py in range(2):
        for px in range(2):
            k = (py * 2 + px) * 32
            v = got[..., k: k + 32] + got[..., 128 + k: 128 + k + 32]
            assert (v - want[:, py::2, px::2]).abs().max().item() < 1e-4


@pytest.mark.parametrize("field", ["fold_cs", "xf_cs"])
def test_split_conv_refuses_folded_stores(field):
    p, op, *_ = _s2d_conv_program()
    p.ops[0] = dataclasses.replace(op, out0_s2d=False, out0=p.tensor("o", 2, 16, 16, 32), **{field: 16})
    with pytest.raises(_lib.StcdError, match="folded"):
        Plan(p, 1, device=-1)
