"""RPN proposal path (SURVEY.md section 8(f) rank 1): decode_bbox_target + ProposalLayer.

CPU: the numpy oracle (oracle/proposal.py) against the golden outputs of the reference's own Python
(tests/golden/proposal_layer.npz, written by oracle/make_golden_proposal.py).
GPU: the device path (pointrcnn_b200/rpn/proposal_layer.py -> csrc/proposal.cu) against the same golden vectors and the
oracle, bit for bit."""
import os
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.append(os.path.join(ROOT, "oracle"))
from make_golden_proposal import CASES, rpn_outputs  # noqa: E402
from oracle import proposal as P  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "proposal_layer.npz")
ANCHOR = np.array([1.52563191462, 1.62856739989, 3.88311640418], dtype=np.float32)     # tools/cfgs/default.yaml:19
MODES = {"TEST": dict(pre_nms_top_n=9000, post_nms_top_n=100, nms_thresh=0.8),           # default.yaml:163-165
         "TRAIN": dict(pre_nms_top_n=9000, post_nms_top_n=512, nms_thresh=0.85)}         # default.yaml:156-158


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN)


def test_decode_oracle_matches_reference_python(gold):
    _, reg, xyz = rpn_outputs(2, 4096, 106)
    d = P.decode_bbox_target(xyz.reshape(-1, 3), reg.reshape(-1, 76), ANCHOR, 3.0, 0.5, 12, True)
    assert np.array_equal(d, gold["decode_boxes"])


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_proposal_oracle_matches_reference_python(gold, case):
    name, mode, nms_type, dist_based, B, N, seed = case
    scores, reg, xyz = rpn_outputs(B, N, seed, far_empty=name.endswith("far_area_empty"))
    b, s = P.proposal_layer(scores, reg, xyz, ANCHOR, nms_type=nms_type, distance_based=dist_based, **MODES[mode])
    assert np.array_equal(b, gold[name + "_boxes"]) and np.array_equal(s, gold[name + "_scores"])


def _cfg(nms_type, dist_based):
    ns = types.SimpleNamespace
    cfg = {"TEST": ns(RPN_PRE_NMS_TOP_N=9000, RPN_POST_NMS_TOP_N=100, RPN_NMS_THRESH=0.8, RPN_DISTANCE_BASED_PROPOSE=dist_based),
           "TRAIN": ns(RPN_PRE_NMS_TOP_N=9000, RPN_POST_NMS_TOP_N=512, RPN_NMS_THRESH=0.85, RPN_DISTANCE_BASED_PROPOSE=True)}

    class Cfg(dict):
        __getattr__ = dict.__getitem__
    c = Cfg(cfg)
    c["CLS_MEAN_SIZE"] = ANCHOR[None]
    c["RPN"] = ns(LOC_SCOPE=3.0, LOC_BIN_SIZE=0.5, NUM_HEAD_BIN=12, LOC_XZ_FINE=True, NMS_TYPE=nms_type)
    return c


@pytest.mark.gpu
def test_decode_kernel_bit_exact(cuda, gold):
    from pointrcnn_b200.rpn.proposal_layer import decode_rpn_proposals
    _, reg, xyz = rpn_outputs(2, 4096, 106)
    got = decode_rpn_proposals(torch.from_numpy(xyz).to(cuda), torch.from_numpy(reg).to(cuda), ANCHOR, 3.0, 0.5, 12, True)
    want = gold["decode_boxes"].copy()
    want[:, 1] = want[:, 1] + want[:, 3] / np.float32(2)             # proposal_layer.py:32 is fused into the kernel
    assert np.array_equal(got.cpu().numpy().reshape(-1, 7), want)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_proposal_layer_bit_exact(cuda, gold, case):
    from pointrcnn_b200.rpn.proposal_layer import ProposalLayer
    name, mode, nms_type, dist_based, B, N, seed = case
    scores, reg, xyz = rpn_outputs(B, N, seed, far_empty=name.endswith("far_area_empty"))
    layer = ProposalLayer(mode=mode, cfg=_cfg(nms_type, dist_based))
    b, s = layer(torch.from_numpy(scores).to(cuda), torch.from_numpy(reg).to(cuda), torch.from_numpy(xyz).to(cuda))
    assert tuple(b.shape) == gold[name + "_boxes"].shape
    assert np.array_equal(s.cpu().numpy(), gold[name + "_scores"]), "kept scores differ from the reference's proposal layer"
    assert np.array_equal(b.cpu().numpy(), gold[name + "_boxes"]), "proposals differ from the reference's proposal layer"


@pytest.mark.gpu
def test_proposal_layer_few_points_and_empty_ranges(cuda):
    """fewer candidates than the quotas, survivors < post_nms_top_n (zero rows behind them), nothing in the far range"""
    from pointrcnn_b200.rpn.proposal_layer import ProposalLayer
    for seed, N, far_empty in ((7, 700, False), (8, 150, True), (9, 40, False)):
        scores, reg, xyz = rpn_outputs(3, N, seed, far_empty=far_empty)
        want_b, want_s = P.proposal_layer(scores, reg, xyz, ANCHOR, nms_type="rotate", distance_based=True, **MODES["TRAIN"])
        layer = ProposalLayer(mode="TRAIN", cfg=_cfg("rotate", True))
        b, s = layer(torch.from_numpy(scores).to(cuda), torch.from_numpy(reg).to(cuda), torch.from_numpy(xyz).to(cuda))
        assert np.array_equal(s.cpu().numpy(), want_s) and np.array_equal(b.cpu().numpy(), want_b)


@pytest.mark.gpu
@pytest.mark.parametrize("n_pts,with_twin", [(5000, False), (16384, True)])
def test_fused_rpn_heads_match_torch(cuda, n_pts, with_twin):
    """cls [128,128,1] + reg [128,128,76] head stacks (lib/net/rpn.py:19-47) as one two-layer tensor-core launch"""
    import torch.nn as nn
    from pointrcnn_b200.pointnet2 import pytorch_utils as pt_utils
    from pointrcnn_b200.pointnet2 import pointnet2_modules as pm
    from pointrcnn_b200.rpn.heads import rpn_heads
    torch.manual_seed(5)

    class Heads(nn.Module):
        def __init__(self):
            super().__init__()
            self.rpn_cls_layer = nn.Sequential(pt_utils.Conv1d(128, 128, bn=True), nn.Dropout(0.5), pt_utils.Conv1d(128, 1, activation=None))
            self.rpn_reg_layer = nn.Sequential(pt_utils.Conv1d(128, 128, bn=True), nn.Dropout(0.5), pt_utils.Conv1d(128, 76, activation=None))
    h = Heads().to(cuda).eval()
    g = torch.Generator().manual_seed(3)
    for m in h.modules():
        if isinstance(m, nn.BatchNorm1d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.2)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)
    nn.init.normal_(h.rpn_cls_layer[2].conv.bias, mean=-2.0, std=0.1)
    f = torch.randn(2, 128, n_pts, device=cuda)
    if with_twin:
        f = pm._attach_pm(f, f.transpose(1, 2).contiguous())
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            want_c = h.rpn_cls_layer(f).transpose(1, 2).contiguous()
            want_r = h.rpn_reg_layer(f).transpose(1, 2).contiguous()
            got_c, got_r = rpn_heads(h, f)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert got_c.shape == want_c.shape == (2, n_pts, 1) and got_r.shape == want_r.shape == (2, n_pts, 76)
    assert got_c.is_contiguous() and got_r.is_contiguous()
    assert (got_r.min() < 0) and (got_c.min() < 0), "the last layer is linear: negative outputs must survive"
    for got, want in ((got_c, want_c), (got_r, want_r)):
        assert (got - want).abs().max().item() <= 1e-2 * want.abs().max().item()
    # grad-enabled / training calls take the reference-shaped torch path
    h.train()
    c2, r2 = rpn_heads(h, f)
    assert c2.requires_grad and r2.shape == (2, n_pts, 76)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_golden_holds_with_the_reference_nms_kernel(cuda, gold, case, monkeypatch):
    """The golden vectors were produced by the reference's own Python with the CPU oracle standing in for its NMS
    extension (no GPU in the build container).  Here every NMS call of that pipeline is served by the reference's OWN
    kernel + host scan (oracle/_ref: nmsLauncher / nmsNormalLauncher, iou3d.cpp:73-170) on the B200 and the result must
    be the committed golden, rotated cases included -- i.e. the goldens are what the reference produces end to end.
    Without oracle/_ref the committed golden is checked against the recorded output of that run (tests/refstore.py)."""
    import refstore as REF
    from oracle import refgpu as R
    name, mode, nms_type, dist_based, B, N, seed = case

    def ref_nms(boxes_bev, scores, thresh, nms_t):
        order = np.argsort(-scores, kind="stable")
        keep = R.nms(torch.from_numpy(np.ascontiguousarray(boxes_bev[order])).to(cuda), float(thresh), normal=(nms_t == "normal"))
        return order[keep.numpy()]

    def ref_flow():
        with monkeypatch.context() as m:
            m.setattr(P, "_nms", ref_nms)
            scores, reg, xyz = rpn_outputs(B, N, seed, far_empty=name.endswith("far_area_empty"))
            return P.proposal_layer(scores, reg, xyz, ANCHOR, nms_type=nms_type, distance_based=dist_based, **MODES[mode])
    REF.equal("scores", gold[name + "_scores"], lambda: ref_flow()[1], "the golden scores are not what the reference produces")
    REF.equal("boxes", gold[name + "_boxes"], lambda: ref_flow()[0], "the golden boxes are not what the reference produces")


# ------------------------------------------------------------------------------------------------ RCNN target layer (8(f) rank 2)
TARGET_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "proposal_target_layer.npz")


def _target_cfg(aug_times, aug_data):
    from pointrcnn_b200.rpn import proposal_target_layer as ptl
    d = dict(ptl.DEFAULT_CFG, AUG_DATA=aug_data)
    d["RCNN"] = dict(d["RCNN"], ROI_FG_AUG_TIMES=aug_times)
    return ptl._ns(d)


@pytest.mark.gpu
def test_proposal_target_layer_matches_reference_python(cuda):
    """deterministic configuration (no jitter loop, no augmentation): the device layer against the outputs of the reference's
    own Python (oracle/make_golden_proposal_target.py), same numpy / torch seeds -> same sampled RoIs, labels and pooled points"""
    from make_golden_proposal_target import SEED, expand, inputs
    from pointrcnn_b200.rpn.proposal_target_layer import ProposalTargetLayer
    g = expand(np.load(TARGET_GOLDEN), inputs())
    layer = ProposalTargetLayer(cfg=_target_cfg(0, False))
    inp = {k: torch.from_numpy(v).to(cuda) for k, v in inputs().items()}
    np.random.seed(SEED)
    torch.manual_seed(SEED)
    with torch.no_grad():
        out = layer(inp)
    assert np.array_equal(out["roi_boxes3d"].cpu().numpy(), g["roi_boxes3d"]), "sampled RoIs differ"
    assert np.array_equal(out["cls_label"].cpu().numpy(), g["cls_label"]) and np.array_equal(out["reg_valid_mask"].cpu().numpy(), g["reg_valid_mask"])
    np.testing.assert_allclose(out["gt_iou"].cpu().numpy(), g["gt_iou"], rtol=1e-4, atol=1e-6)       # CPU libm vs device in the overlap
    np.testing.assert_allclose(out["gt_of_rois"].cpu().numpy(), g["gt_of_rois"], rtol=1e-5, atol=2e-5)
    # pooled rows: the golden's point-in-box flags come from the CPU oracle (host libm sin/cos): a point on a box face may
    # fall on the other side on the device, which shifts that RoI's rows -- RoI by RoI, nearly all must be identical
    pf, gf = out["pts_feature"].cpu().numpy().copy(), g["pts_feature"].copy()
    # column 1 is pts_depth / 70 - 0.5 computed by torch: on CUDA a division by a scalar is a multiplication by its reciprocal,
    # the golden was computed on the CPU (true division) -> compare that column with a one-ulp tolerance, the rest exactly
    np.testing.assert_allclose(pf[..., 1], gf[..., 1], rtol=0, atol=1e-6)
    pf[..., 1] = gf[..., 1] = 0
    same = np.all(pf.reshape(pf.shape[0], -1) == gf.reshape(gf.shape[0], -1), axis=1)
    assert same.mean() >= 0.95, "pooled features differ for %d of %d RoIs" % ((~same).sum(), same.size)
    np.testing.assert_allclose(out["sampled_pts"].cpu().numpy()[same], g["sampled_pts"][same], rtol=0, atol=3e-5)


@pytest.mark.gpu
def test_proposal_target_layer_jitter_loop_properties(cuda):
    """batched jitter loop (ROI_FG_AUG_TIMES = 10) + augmentation: every reported IoU is the true IoU of the returned (pre-
    augmentation) RoI with its GT, foreground jitter stops at the threshold, labels follow the IoU rules"""
    from make_golden_proposal_target import inputs
    from pointrcnn_b200.ext import iou3d_cuda
    from pointrcnn_b200.rpn.proposal_target_layer import ProposalTargetLayer
    layer = ProposalTargetLayer(cfg=_target_cfg(10, False))
    inp = {k: torch.from_numpy(v).to(cuda) for k, v in inputs().items()}
    np.random.seed(3)
    torch.manual_seed(3)
    with torch.no_grad():
        rois, gts, iou = layer.sample_rois_for_rcnn(inp["roi_boxes3d"], inp["gt_boxes3d"])
    true_iou = iou3d_cuda.boxes_iou3d_aligned(rois.reshape(-1, 7).contiguous(), gts.reshape(-1, 7).contiguous()).view(iou.shape)
    assert torch.allclose(iou, true_iou, rtol=1e-6, atol=1e-7), "reported IoU is not the IoU of the returned RoI"
    B, Rn = iou.shape
    assert Rn == 64 and (iou[:, :32] >= 0).all()
    # jittered boxes differ from every source RoI for most samples (p = 0.8 per draw), but stay near their GT cluster
    src = inp["roi_boxes3d"]
    same = (rois.unsqueeze(2) == src.unsqueeze(1)).all(dim=3).any(dim=2).float().mean().item()
    assert same < 0.6, "the jitter loop left %.0f%% of the RoIs untouched" % (100 * same)
    layer2 = ProposalTargetLayer(cfg=_target_cfg(10, True))
    with torch.no_grad():
        out = layer2(inp)
    assert out["sampled_pts"].shape == (B * 64, 512, 3) and torch.isfinite(out["sampled_pts"]).all()
    lab, giou = out["cls_label"], out["gt_iou"]
    assert ((lab == 1) <= (giou > 0.6)).all() and ((giou < 0.45) <= (lab <= 0)).all()
