"""The oracle (oracle/nets.py, oracle/metric.py) against the reference's own outputs: tests/golden/*.npz, generated
from the UNMODIFIED reference by oracle/make_golden.py.
"""
import os

import numpy as np
import pytest
import torch

from oracle import metric as ometric
from oracle import nets
from oracle.make_golden import CASES
from stcd_b200 import synth
from stcd_b200.networks import CLASSES


def _our_net(case):
    mod, cls, args, b, h, w = CASES[case]
    return synth.prepare_(CLASSES[cls](*args).eval(), cls)


def _oracle_forward(case, sd, x1, x2):
    cls = CASES[case][1]
    if cls == "SiamUnet_diff":
        return [nets.siamunet_forward(sd, x1, x2, "diff")]
    if cls == "SiamUnet_conc":
        return [nets.siamunet_forward(sd, x1, x2, "conc")]
    if cls in ("SiamUnet_sub", "SiamUnet_cross_conc", "Unet"):
        return [nets.siamunet_forward(sd, x1, x2, {"SiamUnet_sub": "sub", "SiamUnet_cross_conc": "cross", "Unet": "ef"}[cls])]
    if cls == "SNUNet_ECAM":
        return [nets.snunet_forward(sd, x1, x2)]
    if cls == "SegCD":
        return list(nets.segcd_forward(sd, x1, x2))
    if cls == "ChangeGNNV1":
        return nets.changegnn_forward(sd, x1, x2)
    if cls == "ChangeFormerV6":
        return nets.changeformer_forward(sd, x1, x2)
    if cls == "CDNet_model":
        return [nets.dtcdscn_forward(sd, x1, x2)]
    if cls == "BASE_Transformer":
        return [nets.bit_forward(sd, x1, x2, stages=4)]
    if cls == "ResNet":
        return [nets.bit_forward(sd, x1, x2, stages=5)]
    if cls == "DSIFN":
        return [nets.dsifn_forward(sd, x1, x2)]
    if cls == "ChangeFormerV1":
        return [nets.changeformer_v1_forward(sd, x1, x2)]
    if cls == "ChangeFormerV2":
        return [nets.changeformer_v2_forward(sd, x1, x2)]
    if cls == "ChangeFormerV3":
        return [nets.changeformer_v3_forward(sd, x1, x2)]
    if cls == "VIG_V20_2":
        return nets.vig_v20_forward(sd, x1, x2)
    if cls == "ChangeGNNV2":
        return nets.changegnn_v2_forward(sd, x1, x2, "cross")
    if cls == "ChangeGNNV2_Compare":
        return nets.changegnn_v2_forward(sd, x1, x2, CASES[case][2][6])
    raise KeyError(cls)


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_matches_golden(case, golden_dir):
    g = np.load(os.path.join(golden_dir, f"{case}.npz"))
    x1, x2 = synth.image_pairs(int(g["batch"]), int(g["h"]), int(g["w"]), seed=int(g["data_seed"]))
    assert abs(float(x1.double().sum()) - float(g["x1_sum"])) < 1e-6, "synthetic inputs are not reproducible"
    net = _our_net(case)          # same seed + same module order as the reference => same weights
    with torch.no_grad():
        outs = _oracle_forward(case, net.state_dict(), x1, x2)
    assert len(outs) == int(g["n_out"])
    for i, y in enumerate(outs):
        ref = torch.from_numpy(g[f"out{i}"])
        assert y.shape == ref.shape
        # same fp32 ops, possibly different threading/accumulation order
        assert (y - ref).abs().max().item() < 1e-4


def test_metric_oracle_matches_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "segmentation_metric.npz"))
    cm = ometric.confusion_matrix(g["pred"], g["label"]) + ometric.confusion_matrix(g["pred2"], g["label"])
    assert np.array_equal(cm.astype(np.float64), g["cm"])
    s = ometric.scores(cm)
    np.testing.assert_allclose(s["F1"], g["f1"], rtol=0, atol=1e-15)
    np.testing.assert_allclose(s["IoU"], g["iou"], rtol=0, atol=1e-15)
    np.testing.assert_allclose(s["OA"], g["oa"], rtol=0, atol=1e-15)
    np.testing.assert_allclose(s["Precision"], g["precision"], rtol=0, atol=1e-15)
    np.testing.assert_allclose(s["Recall"], g["recall"], rtol=0, atol=1e-15)


def test_binarise_semantics():
    x = np.array([[[[0.0, 1e-8, 1e-6, -1.0, 2.0]]]], dtype=np.float32)
    # sigmoid(x) > 0.5 is NOT x > 0 in fp32: tiny positive logits round to exactly 0.5 (SURVEY §7.3-3)
    assert ometric.binarise(x, "sigmoid").ravel().tolist() == [0, 0, 1, 0, 1]
    assert ometric.binarise(x, "raw_ge", 0.5).ravel().tolist() == [0, 0, 0, 0, 1]
    two = np.stack([np.zeros((1, 1, 3)), np.array([[[0.0, 1.0, -1.0]]])], axis=1).astype(np.float32).reshape(1, 2, 1, 3)
    assert ometric.binarise(two, "argmax").ravel().tolist() == [0, 1, 0]     # ties -> class 0


def test_cm2score_matches_independent_statement():
    """ConfuseMatrixMeter's score dict (models/evaluator.py:150-167; misc/metric_tool.py absent upstream: parity unpinned)."""
    import numpy as np
    from oracle import metric as ometric
    from stcd_b200.metric import cm2score
    g = np.random.default_rng(4)
    pr = (g.random((3, 32, 32)) < 0.4).astype(np.int64)
    gt = (g.random((3, 32, 32)) < 0.25).astype(np.int64)
    cm = ometric.confusion_matrix(pr, gt)
    got, want = cm2score(cm), ometric.confuse_matrix_meter_scores(pr, gt)
    assert set(got) == set(want)
    for k in want:
        assert abs(got[k] - want[k]) < 1e-12, k
    absent = cm2score(np.array([[10.0, 0.0], [0.0, 0.0]]))      # class 1 absent: eps keeps every score finite (0, not NaN)
    assert absent["F1_1"] == 0.0 and absent["iou_1"] == 0.0 and np.isfinite(absent["mf1"])
