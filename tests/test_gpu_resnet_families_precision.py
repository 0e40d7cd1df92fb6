"""BIT (s4 / dd8 / dd8_dedim8 and the ResNet-18 baseline) and DTCDSCN on the precision path (``net.precision = "tf32"``:
split-bf16 operands, lowering.Program.precision) on the GPU: logits within 1e-3 ABSOLUTE of the fp32 oracle through the split
space-to-depth stem pack, conv store and max-pool, the feature differences, sums, SE gates and BIT's token kernels."""
import os

import numpy as np
import pytest
import torch

import emulate_split_resnet as emulate
import parity
from stcd_b200 import bit, dtcdscn, lowering as L, synth
from test_resnet_families_precision import NETS, make, oracle

pytestmark = pytest.mark.gpu
TF32_TOL = 1e-3


def _out(y):
    return y[0] if isinstance(y, (list, tuple)) else y


def _check(name, y, ref, min_std=0.25):
    """test_gpu_precision's tf32 bar."""
    r = parity.check(name, y.cpu(), ref, "argmax", abs_tol=TF32_TOL, rms_rel=1e-3, max_rel=4e-3, all_px=0.9995, decided=1.0,
                     min_std=min_std)
    assert r["max_abs_err"] < TF32_TOL
    return r


@pytest.mark.parametrize("name", NETS)
def test_forward_within_1e3_and_matches_emulator(name):
    net = make(name)
    x1, x2 = synth.image_pairs(3, 64, 96)
    ref = oracle(name, net, x1, x2)
    emu = emulate.run_program(net.lower(64, 96), x1, x2, chunk=2)[0]
    net = net.cuda()
    net.chunk_pairs = 2                      # 3 pairs -> one full chunk + a ragged one
    y = _out(net(x1.cuda(), x2.cuda())).cpu()
    assert y.shape == ref.shape and y.dtype == torch.float32
    _check(f"tf32:{name}:3x64x96", y, ref)
    assert (y - emu).abs().max().item() < 2e-4, "kernel vs emulator (same split points, fp32 accumulation order differs)"


@pytest.mark.parametrize("name", ["dd8", "dtcdscn"])
def test_layerwise_against_emulator(name):
    """Every plan tensor (hi + lo) against the emulator's: the stem pack, the space-to-depth conv stores, the max-pool, BIT's
    token path (dd8) and the SE / SCSE gates, signed differences and the Dblock sum (DTCDSCN), each at its own tensor."""
    net = make(name)
    x1, x2 = synth.image_pairs(1, 64, 96, seed=9)
    keep = {}
    emulate.run_program(net.lower(64, 96), x1, x2, chunk=1, keep=keep)
    net = net.cuda()
    net.chunk_pairs = 1
    net(x1.cuda(), x2.cuda())
    torch.cuda.synchronize()
    plan = net.plan_for(x1.cuda())
    # a difference of the two streams' features cancels most of their magnitude: its error is measured against its operands
    scale_of = {op.dst: op.src for op in plan.prog.ops if isinstance(op, L.AbsDiffSpec)}
    both = lambda t: t[..., : t.shape[-1] // 2] + t[..., t.shape[-1] // 2:]  # noqa: E731
    worst = {}
    for tname in plan.prog.tensors:
        got, want = both(plan.read_tensor(tname)), both(keep[tname])
        worst[tname] = ((got - want).abs().mean() / (both(keep[scale_of.get(tname, tname)]).abs().mean() + 1e-6)).item()
    bad = {k: v for k, v in worst.items() if v > 1e-4}
    assert not bad, bad


@pytest.mark.parametrize("case", ["bit_dd8", "bit_resnet18", "dtcdscn"])
def test_golden_within_1e3(case, golden_dir):
    """The reference's own outputs (registry gains: logit std 0.04-0.09, so the spread floor of the other tests does not apply)."""
    g = np.load(os.path.join(golden_dir, f"{case}.npz"))
    if case == "dtcdscn":
        net = synth.prepare_(dtcdscn.CDNet34(3, 2).eval(), "CDNet_model", seed=int(g["weight_seed"]))
    elif case == "bit_resnet18":
        net = synth.prepare_(bit.ResNet(3, 2).eval(), "ResNet")
    else:
        net = synth.prepare_(bit.BASE_Transformer(3, 2, with_pos="learned", resnet_stages_num=4, token_len=4, enc_depth=1,
                                                  dec_depth=8).eval(), "BASE_Transformer")
    net.precision = "tf32"
    net = net.cuda()
    x1, x2 = synth.image_pairs(int(g["batch"]), int(g["h"]), int(g["w"]), seed=int(g["data_seed"]))
    y = _out(net(x1.cuda(), x2.cuda())).cpu()
    ref = torch.from_numpy(g["out0"])
    r = parity.report(f"tf32:{case}:golden", y, ref, "argmax", abs_tol=TF32_TOL)
    assert r["max_abs_err"] < TF32_TOL and r["agree_decided"] == 1.0, r


@pytest.mark.parametrize("name", ["dd8", "dtcdscn"])
def test_bench_shape_within_1e3(name):
    """The bench shapes (bit_dd8_256_b32, dtcdscn_256_b32: 32 pairs of 256 x 256, chunk 32): two sampled pairs against the
    oracle, the same logits at chunk 8, deterministic."""
    net = make(name)
    x1, x2 = synth.image_pairs(32, 256, 256, seed=5)
    pick = torch.tensor([0, 31])
    ref = oracle(name, net, x1[pick], x2[pick])
    net = net.cuda()
    net.chunk_pairs = 32
    a, b = x1.cuda(), x2.cuda()
    y = _out(net(a, b))
    _check(f"tf32:{name}:32x256x256 (pairs 0, 31 vs oracle)", y[pick.cuda()], ref)
    assert torch.equal(y, _out(net(a, b))), "deterministic"
    net.chunk_pairs = 8
    assert torch.equal(y, _out(net(a, b))), "pairs are independent of the chunking"


def test_bf16_and_tf32_side_by_side():
    net = make("dd8", "bf16")
    x1, x2 = synth.image_pairs(2, 64, 96, seed=7)
    ref = oracle("dd8", net, x1, x2)
    net = net.cuda()
    a, b = x1.cuda(), x2.cuda()
    y16 = _out(net(a, b))
    net.precision = "tf32"
    y32 = _out(net(a, b))
    e16 = parity.report("bf16:dd8:2x64x96 (for the comparison)", y16.cpu(), ref, "argmax")["max_abs_err"]
    e32 = (y32.cpu() - ref).abs().max().item()
    assert e32 < TF32_TOL and e16 > 10 * e32, (e16, e32)
    net.precision = "bf16"
    assert torch.equal(y16, _out(net(a, b))), "the bf16 plan is unchanged by the tf32 one"


@pytest.mark.parametrize("key", ["base_transformer_pos_s4_dd8", "base_resnet18", "DTCDSCN"])
def test_define_G_tf32(key):
    from types import SimpleNamespace
    from stcd_b200 import networks
    net = networks.define_G(SimpleNamespace(net_G=key, n_class=2, precision="tf32"), gpu_ids=[0])
    assert isinstance(net, (bit.ResNet, dtcdscn.CDNet_model)) and net.plan_precision == "split"
    x1, x2 = synth.image_pairs(1, 64, 64)
    y = _out(net.eval()(x1.cuda(), x2.cuda()))
    assert y.shape == (1, 2, 64, 64) and torch.isfinite(y).all()
