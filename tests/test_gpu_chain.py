"""End-to-end chain (BASELINE configs[3]/[4], VERDICT r1 item 6): RPN backbone -> heads -> proposal layer -> roipool3d
(+ canonical transform) -> RCNN SA stack -> decode -> final rotated NMS, from the repo's own modules on the B200
natives, against the SAME chain on the reference's own kernels (oracle/_ref) + stock torch ops: their recorded outputs
(tests/refstore.py), and the live kernels as well when oracle/_ref is present.

MLP outputs carry TF32 rounding, so stage N+1 of both chains is fed THIS repo's stage-N output: every index / keep /
flag output is then compared exactly, every floating-point output within the stated tolerance.
Reference: lib/net/point_rcnn.py:26-70, lib/net/rcnn_net.py:115-190, tools/eval_rcnn.py:459-640.
"""
import functools
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.append(os.path.join(ROOT, "oracle"))
import refstore as REF  # noqa: E402
import synth  # noqa: E402
from oracle import oracle as O  # noqa: E402
from oracle import proposal as P  # noqa: E402
from oracle import refgpu as R  # noqa: E402

pytestmark = pytest.mark.gpu
TOL = 2e-3
TOL_BACKBONE = 5e-3


def _randomise_bn(module, seed):
    g = torch.Generator().manual_seed(seed)
    for m in module.modules():
        if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm1d)):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)


def _fp32(fn):
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        return fn()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.fixture(scope="module")
def chain(cuda):
    from pointrcnn_b200.point_rcnn import PointRCNNInference
    torch.manual_seed(21)
    model = PointRCNNInference(input_channels=1).to(cuda).eval()
    _randomise_bn(model, 22)
    with torch.no_grad():
        # heads that produce a usable score spread / box sizes on random weights
        model.rpn.rpn_reg_layer[-1].conv.weight.mul_(0.2)
    B, N = 8, 16384                                               # BASELINE configs[4]: batch 8
    pc = torch.from_numpy(np.concatenate([synth.u_kitti(1, N, 5000 + i, channels=4) for i in range(B)], 0)).to(cuda)
    with torch.no_grad():
        out = model(pc)
        dets, pred = model.detections(out)
    return model, pc, out, dets, pred


def test_rpn_stage_against_reference_kernels(cuda, chain):
    from oracle.ref_backbone import backbone as ref_backbone
    from pointrcnn_b200.rpn.stage import CLS_MEAN_SIZE
    model, pc, out, _, _ = chain
    with torch.no_grad():
        ref = functools.lru_cache(None)(lambda: _fp32(lambda: ref_backbone(model.rpn.backbone_net, pc)))
        REF.equal("xyz", out["backbone_xyz"], lambda: ref()[0], "backbone xyz differ from the reference kernels")
        idx, want, absmax = REF.sample("features", lambda: ref()[1])
        got = out["backbone_features"].reshape(-1)[torch.from_numpy(idx).to(cuda)].cpu().numpy()
        rel = np.abs(got - want).max() / absmax
        assert rel <= TOL_BACKBONE, "backbone features vs reference kernels + fp32 cuDNN (stored sample): %g" % rel
        if REF.live():
            rfeats = ref()[1]
            rel = (out["backbone_features"] - rfeats).abs().max().item() / rfeats.abs().max().item()
            assert rel <= TOL_BACKBONE, "backbone features vs reference kernels + fp32 cuDNN: %g" % rel
        # heads on OUR features: fused tcgen05 heads vs the torch modules
        cls_t = _fp32(lambda: model.rpn.rpn_cls_layer(out["backbone_features"]).transpose(1, 2).contiguous())
        reg_t = _fp32(lambda: model.rpn.rpn_reg_layer(out["backbone_features"]).transpose(1, 2).contiguous())
    assert (out["rpn_cls"] - cls_t).abs().max().item() <= TOL * cls_t.abs().max().item()
    assert (out["rpn_reg"] - reg_t).abs().max().item() <= TOL * reg_t.abs().max().item()
    # proposal layer on OUR cls / reg / xyz: device path vs the reference-shaped flow with the reference's NMS kernel
    def ref_nms(boxes_bev, scores, thresh, nms_t):
        order = np.argsort(-scores, kind="stable")
        keep = R.nms(torch.from_numpy(np.ascontiguousarray(boxes_bev[order])).to(cuda), float(thresh), normal=(nms_t == "normal"))
        return order[keep.numpy()]
    @functools.lru_cache(None)
    def ref_flow():
        old = P._nms
        P._nms = ref_nms
        try:
            return P.proposal_layer(out["rpn_cls"][:, :, 0].cpu().numpy(), out["rpn_reg"].cpu().numpy(), out["backbone_xyz"].cpu().numpy(),
                                    CLS_MEAN_SIZE[0], pre_nms_top_n=9000, post_nms_top_n=100, nms_thresh=0.8, nms_type="normal",
                                    distance_based=True)
        finally:
            P._nms = old
    REF.equal("scores", out["roi_scores_raw"], lambda: ref_flow()[1], "proposal scores differ from the reference flow")
    REF.equal("rois", out["rois"], lambda: ref_flow()[0], "proposals differ from the reference flow")
    b = out["rois"].cpu().numpy()
    assert (np.abs(b).sum(axis=2) > 0).sum() >= 8 * 50, "degenerate proposals: the test would not exercise the RCNN stage"


def test_roipool_and_rcnn_stage_against_reference_kernels(cuda, chain):
    from pointrcnn_b200 import config, kitti_utils
    model, pc, out, _, _ = chain
    rcnn = model.rcnn_net
    xyz, feats, rois = out["backbone_xyz"], out["backbone_features"], out["rois"]
    seg_mask = out["seg_result"]
    depth = torch.norm(xyz, p=2, dim=2)
    pts_feature = torch.cat((seg_mask.unsqueeze(2), (depth / 70.0 - 0.5).unsqueeze(2), feats.permute(0, 2, 1)), dim=2).contiguous()
    with torch.no_grad():
        pts_input, empty = rcnn.pool(xyz, feats.permute(0, 2, 1), seg_mask, depth, rois)
        # reference kernel on the enlarged boxes, then the reference's canonical transform in torch (rcnn_net.py:146-152)
        big = kitti_utils.enlarge_box3d(rois.view(-1, 7), 1.0).view(rois.shape[0], -1, 7).contiguous()

        @functools.lru_cache(None)
        def ref_pool():
            rp, re = R.roipool3d(xyz, pts_feature, big, 512)
            rp[..., 0:3] -= rois[:, :, None, 0:3]
            for k in range(rois.shape[0]):
                rp[k, :, :, 0:3] = kitti_utils.rotate_pc_along_y_torch(rp[k, :, :, 0:3], rois[k, :, 6])
            return rp, re
        got = pts_input.view(rois.shape[0], rois.shape[1], 512, -1)
        REF.equal("empty", empty, lambda: ref_pool()[1], "empty flags differ from the reference kernel")
        REF.equal("features", got[..., 3:], lambda: ref_pool()[0][..., 3:], "pooled features differ from the reference kernel")
        idx, want, _ = REF.sample("canonical_xyz", lambda: ref_pool()[0][..., 0:3])
        got_xyz = got[..., 0:3].reshape(-1)[torch.from_numpy(idx).to(cuda)].cpu().numpy()
        assert np.abs(got_xyz - want).max() <= 2e-5, "canonical xyz differ (stored sample)"
        if REF.live():
            assert (got[..., 0:3] - ref_pool()[0][..., 0:3]).abs().max().item() <= 2e-5, "canonical xyz differ"
        nonempty = int((empty == 0).sum())
        assert nonempty >= 8 * 20, "too few non-empty RoIs (%d) for a meaningful stage-2 check" % nonempty
        # RCNN SA stack on OUR pooled points: fused tcgen05 path vs the op-by-op path (our index natives + fp32 cuDNN)
        cls_f, reg_f = rcnn.forward_pts(pts_input)
        with config.override(disable_fused=True):
            cls_u, reg_u = _fp32(lambda: rcnn.forward_pts(pts_input))
        assert (cls_f - cls_u).abs().max().item() <= TOL_BACKBONE * cls_u.abs().max().item()
        assert (reg_f - reg_u).abs().max().item() <= TOL_BACKBONE * reg_u.abs().max().item()
        assert torch.equal(cls_f, out["rcnn_cls"]) and torch.equal(reg_f, out["rcnn_reg"])
        # sampling inside the RCNN stage: our FPS on the pooled clouds (duplicate-heavy: k % cnt padding) vs the reference kernel
        pooled_xyz = pts_input[..., 0:3].contiguous()
        from pointrcnn_b200.pointnet2 import pointnet2_utils as pu
        sub = pooled_xyz[:256]
        REF.equal("fps", pu.furthest_point_sample(sub, 128), lambda: R.fps(sub, 128), "RCNN SA1 sampling differs")


def test_final_detections_against_reference_nms(cuda, chain):
    from pointrcnn_b200 import kitti_utils
    model, pc, out, dets, pred = chain
    B = pred.shape[0]
    raw = out["rcnn_cls"].view(B, -1)
    total = 0
    for k in range(B):
        sel = torch.sigmoid(raw[k]) > model.rcnn_score_thresh
        boxes_k, raw_k = pred[k][sel], raw[k][sel]
        if boxes_k.shape[0] == 0:
            assert dets[k][0].shape[0] == 0
            continue
        order = raw_k.sort(0, descending=True)[1]

        def want(k=k, boxes_k=boxes_k, order=order):
            keep_ref = R.nms(kitti_utils.boxes3d_to_bev_torch(boxes_k)[order].contiguous(), model.rcnn_nms_thresh, normal=False)
            return order[keep_ref.to(order.device)]
        REF.equal("scene%d_boxes" % k, dets[k][0], lambda: boxes_k[want()], "scene %d: kept detections differ" % k)
        REF.equal("scene%d_scores" % k, dets[k][1], lambda: raw_k[want()], "scene %d: kept detections differ" % k)
        total += dets[k][0].shape[0]
    assert total > 0, "no detections at all: the final NMS was not exercised"


def test_batched_detections_and_kitti_writer_equal_the_per_scene_path(cuda, chain, tmp_path):
    """detections_device (no host round trip) selects exactly detections()'s boxes in the same order; write_kitti_batch writes
    what save_kitti_format writes scene by scene"""
    from pointrcnn_b200.datasets import kitti_output
    from oracle import kitti_io as KO
    model, pc, out, dets, _ = chain
    with torch.no_grad():
        boxes, raw, select = model.detections_device(out)
    B = boxes.shape[0]
    assert sum(int(d[0].shape[0]) for d in dets) > 0, "the fixture must produce detections"
    for k in range(B):
        sel = select[k]
        assert torch.equal(boxes[k][sel], dets[k][0]), "scene %d: batched detections differ" % k
        assert torch.equal(raw[k][sel], dets[k][1])
    texts = kitti_output.write_kitti_batch(range(B), [KO.CALIB] * B, [KO.IMG_SHAPE] * B, boxes, raw, select, str(tmp_path))
    for k in range(B):
        single = tmp_path / "single"
        single.mkdir(exist_ok=True)
        path = kitti_output.save_kitti_format(k, KO.CALIB, dets[k][0], str(single), dets[k][1], KO.IMG_SHAPE)
        assert open(path).read() == texts[k] == open(tmp_path / ("%06d.txt" % k)).read()


def test_batched_detections_with_nothing_above_the_threshold(cuda, chain):
    from pointrcnn_b200.datasets import kitti_output
    from oracle import kitti_io as KO
    model, pc, out, _, _ = chain
    out2 = dict(out)
    out2["rcnn_cls"] = torch.full_like(out["rcnn_cls"], -20.0)          # sigmoid ~ 0: every box is under the score threshold
    with torch.no_grad():
        boxes, raw, select = model.detections_device(out2)
        dets, _ = model.detections(out2)
    assert int(select.sum()) == 0 and all(d[0].shape[0] == 0 for d in dets)
    B = boxes.shape[0]
    texts = kitti_output.write_kitti_batch(range(B), [KO.CALIB] * B, [KO.IMG_SHAPE] * B, boxes, raw, select)
    assert texts == [""] * B
