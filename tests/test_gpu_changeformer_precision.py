"""ChangeFormerV6 (config C5) on the precision path (``net.precision = "tf32"``: split-bf16 operands, lowering.Program.precision)
on the GPU: logits within 1e-3 ABSOLUTE of the fp32 oracle, through the split forms of the LayerNorm, attention, depth-wise conv
and bilinear kernels and the K-partitioned split convs."""
import os

import numpy as np
import pytest
import torch

import parity
import emulate_split as emulate
from oracle import nets
from stcd_b200 import changeformer, synth

pytestmark = pytest.mark.gpu
TF32_TOL = 1e-3
GAIN = 0.6                   # full-resolution logit std 0.38 (>= 0.25); the registry gain of 0.5 gives 0.158


def _net():
    net = synth.randomize_(changeformer.ChangeFormerV6().eval(), gain=GAIN)
    net.precision = "tf32"
    return net


def _check(name, ys, refs, min_std=0.25):
    """test_gpu_precision's tf32 bar on the full-resolution logits, abs < 1e-3 on all five outputs."""
    assert isinstance(ys, list) and len(ys) == 5
    for y, ref in zip(ys, refs):
        assert y.shape == ref.shape and y.dtype == torch.float32
        assert (y.cpu() - ref).abs().max().item() < TF32_TOL
    r = parity.check(name, ys[-1].cpu(), refs[-1], "argmax", abs_tol=TF32_TOL, rms_rel=1e-3, max_rel=4e-3, all_px=0.9995, decided=1.0,
                     min_std=min_std)
    assert r["max_abs_err"] < TF32_TOL
    return r


def test_forward_within_1e3_and_matches_emulator():
    net = _net()
    x1, x2 = synth.image_pairs(3, 256, 256)
    with torch.no_grad():
        ref = nets.changeformer_forward(net.state_dict(), x1, x2)
    emu = emulate.run_program(net.lower(256, 256), x1, x2, chunk=2)
    net = net.cuda()
    net.chunk_pairs = 2                      # 3 pairs -> one full chunk + a ragged one
    ys = net(x1.cuda(), x2.cuda())
    _check("tf32:changeformer_v6:3x256x256", ys, ref)
    for y, e in zip(ys, emu):
        assert (y.cpu() - e).abs().max().item() < 2e-4, "kernel vs emulator (same split points, fp32 accumulation order differs)"


def test_layerwise_against_emulator():
    """Every plan tensor (hi + lo) against the emulator's: a wrong split kernel variant shows up at its own tensor."""
    net = _net()
    x1, x2 = synth.image_pairs(1, 256, 256, seed=9)
    keep = {}
    emulate.run_program(net.lower(256, 256), x1, x2, chunk=1, keep=keep)
    net = net.cuda()
    net.chunk_pairs = 1
    net(x1.cuda(), x2.cuda())
    torch.cuda.synchronize()
    plan = net.plan_for(x1.cuda())
    worst = {}
    for name in plan.prog.tensors:
        got, want = plan.read_tensor(name), keep[name]
        half = got.shape[-1] // 2
        got, want = got[..., :half] + got[..., half:], want[..., :half] + want[..., half:]
        worst[name] = ((got - want).abs().mean() / (want.abs().mean() + 1e-6)).item()
    bad = {k: v for k, v in worst.items() if v > 1e-4}
    assert not bad, bad


def test_config_c5_within_1e3():
    """Config C5 exactly (32 pairs of 256 x 256, chunk 32): four pairs against the oracle, bit-identical at chunk 8, deterministic."""
    net = _net()
    x1, x2 = synth.image_pairs(32, 256, 256, seed=5)
    with torch.no_grad():
        ref = nets.changeformer_forward(net.state_dict(), x1[:4], x2[:4])
    net = net.cuda()
    a, b = x1.cuda(), x2.cuda()
    ys = net(a, b)
    _check("tf32:changeformer_v6:C5 32x256x256 (pairs 0-3 vs oracle)", [y[:4] for y in ys], ref)
    assert all(torch.equal(u, v) for u, v in zip(ys, net(a, b))), "deterministic"
    net.chunk_pairs = 8
    assert all(torch.equal(u, v) for u, v in zip(ys, net(a, b))), "pairs are independent of the chunking"


def test_golden_within_1e3(golden_dir):
    """The reference's own outputs (changeformer_v6.npz, registry gain 0.5: full-resolution logit std 0.158, so the spread floor
    of the other tests does not apply)."""
    g = np.load(os.path.join(golden_dir, "changeformer_v6.npz"))
    assert float(g["gain"]) == synth.GAINS["ChangeFormerV6"]
    net = synth.prepare_(changeformer.ChangeFormerV6().eval(), "ChangeFormerV6")
    net.precision = "tf32"
    net = net.cuda()
    x1, x2 = synth.image_pairs(int(g["batch"]), int(g["h"]), int(g["w"]), seed=int(g["data_seed"]))
    ys = net(x1.cuda(), x2.cuda())
    refs = [torch.from_numpy(g[f"out{i}"]) for i in range(5)]
    assert abs(refs[-1].std().item() - 0.158) < 0.005
    _check("tf32:changeformer_v6:golden (std 0.158)", ys, refs, min_std=0.15)


def test_bf16_and_tf32_side_by_side():
    net = _net()
    x1, x2 = synth.image_pairs(2, 256, 256, seed=7)
    with torch.no_grad():
        ref = nets.changeformer_forward(net.state_dict(), x1, x2)[-1]
    net = net.cuda()
    a, b = x1.cuda(), x2.cuda()
    net.precision = "bf16"
    y16 = net(a, b)
    net.precision = "tf32"
    y32 = net(a, b)
    e16 = parity.report("bf16:changeformer_v6:2x256x256 (for the comparison)", y16[-1].cpu(), ref, "argmax")["max_abs_err"]
    e32 = (y32[-1].cpu() - ref).abs().max().item()
    assert e32 < TF32_TOL and e16 > 10 * e32, (e16, e32)
    net.precision = "bf16"
    assert all(torch.equal(u, v) for u, v in zip(y16, net(a, b))), "the bf16 plan is unchanged by the tf32 one"


def test_define_G_tf32():
    from types import SimpleNamespace
    from stcd_b200 import networks
    net = networks.define_G(SimpleNamespace(net_G="ChangeFormerV6", n_class=2, embed_dim=256, img_size=256, precision="tf32"), gpu_ids=[0])
    assert isinstance(net, changeformer.ChangeFormerV6) and net.plan_precision == "split"
    x1, x2 = synth.image_pairs(1, 256, 256)
    ys = net.eval()(x1.cuda(), x2.cuda())
    assert ys[-1].shape == (1, 2, 256, 256) and all(torch.isfinite(y).all() for y in ys)
