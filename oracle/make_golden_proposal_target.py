"""oracle/make_golden_proposal_target.py -- golden vectors for the RCNN target layer (SURVEY 8(f) rank 2).

Runs the reference's OWN lib/rpn/proposal_target_layer.py (imported unchanged from /root/reference) on this container's CPU
with its two GPU extension entry points served by the CPU oracle (boxes_iou3d_gpu -> oracle.boxes_iou3d, roipool3d_gpu ->
oracle.roipool3d), in the deterministic configuration (ROI_FG_AUG_TIMES = 0, AUG_DATA = False: the random jitter loop draws
from the CUDA generator in the reference and cannot be reproduced off-device), and writes
tests/golden/proposal_target_layer.npz (pooled rows stored as the indices of the input points they copy: see compact()).
TEST INFRASTRUCTURE ONLY.   python oracle/make_golden_proposal_target.py
"""
import hashlib
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import synth  # noqa: E402

REF = "/root/reference"
SEED = 7


def inputs(B=2, N=4096, M=512, C=8, n_gt=7, seed=300):
    """RoIs clustered around `centres` objects; the first n_gt cluster centres are the GT boxes (zero-padded to 12 rows)"""
    rng = np.random.default_rng(seed)
    rois = np.zeros((B, M, 7), np.float32)
    gts = np.zeros((B, 12, 7), np.float32)
    xyz = np.zeros((B, N, 3), np.float32)
    for b in range(B):
        r, _ = synth.boxes3d(M, seed + 1 + b, centres=16)
        rois[b] = r
        # GT = the median box of each of the first n_gt clusters (RoIs were jittered around the same centres)
        rr = np.random.default_rng(seed + 1 + b)
        cx = rr.uniform(-35, 35, 16); cz = rr.uniform(5, 65, 16); cy = rr.uniform(1.2, 2.0, 16); ry = rr.uniform(-np.pi, np.pi, 16)
        for g in range(n_gt - b):
            gts[b, g] = [cx[g], cy[g], cz[g], 1.526, 1.629, 3.883, ry[g]]
        which = rng.integers(0, M, N)
        p = r[which, :3] + rng.normal(0, 1.0, (N, 3))
        p[:, 1] -= r[which, 3] / 2
        xyz[b] = p
    feat = rng.standard_normal((B, N, C)).astype(np.float32)
    seg = (rng.random((B, N)) > 0.5).astype(np.float32)
    depth = np.linalg.norm(xyz, axis=2).astype(np.float32)
    return dict(roi_boxes3d=rois, gt_boxes3d=gts, rpn_xyz=xyz, rpn_features=feat, seg_mask=seg, pts_depth=depth)


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _pooled(idx, inp, rois):
    """pts_feature and sampled_pts of the layer's output from the pooled point indices: each pooled row is an input point
    (seg_mask, pts_depth / 70 - 0.5, rpn_features) and its coordinates relative to the RoI, rotated by -ry about y
    (proposal_target_layer.py:48-54, kitti_utils.rotate_pc_along_y_torch), computed with the same torch CPU ops"""
    R = idx.shape[0]
    b = (np.arange(R) // (R // inp["rpn_xyz"].shape[0]))[:, None]
    depth = (torch.from_numpy(inp["pts_depth"]) / 70.0 - 0.5).numpy()
    feature = np.concatenate([inp["seg_mask"][b, idx][..., None], depth[b, idx][..., None], inp["rpn_features"][b, idx]], 2)
    r = torch.from_numpy(rois)
    pc = torch.from_numpy(inp["rpn_xyz"][b, idx]) - r[:, None, 0:3]
    cosa, sina = torch.cos(r[:, 6]).view(-1, 1), torch.sin(r[:, 6]).view(-1, 1)
    rot = torch.cat((torch.cat([cosa, -sina], 1).unsqueeze(1), torch.cat([sina, cosa], 1).unsqueeze(1)), 1)
    pc[:, :, [0, 2]] = torch.matmul(pc[:, :, [0, 2]], rot.permute(0, 2, 1))
    return feature, pc.numpy()


def compact(res, inp):
    """the stored form of the layer's output (the pooled arrays as int16 point indices + the SHA-256 of each)"""
    R, S = res["pts_feature"].shape[:2]
    B = inp["rpn_xyz"].shape[0]
    rows = [{inp["rpn_features"][b][i].tobytes(): i for i in range(inp["rpn_features"].shape[1])} for b in range(B)]
    idx = np.array([[rows[r // (R // B)][res["pts_feature"][r, s, 2:].tobytes()] for s in range(S)] for r in range(R)], np.int16)
    out = {k: v for k, v in res.items() if k not in ("pts_feature", "sampled_pts")}
    out.update(pooled_index=idx, pts_feature_sha256=np.array(_sha(res["pts_feature"])), sampled_pts_sha256=np.array(_sha(res["sampled_pts"])))
    assert all(np.array_equal(expand(out, inp)[k], res[k]) for k in res)
    return out


def expand(g, inp):
    """the layer's output from its stored form, checked bit for bit against the stored SHA-256"""
    out = {k: g[k] for k in ("cls_label", "reg_valid_mask", "gt_of_rois", "gt_iou", "roi_boxes3d")}
    out["pts_feature"], out["sampled_pts"] = _pooled(g["pooled_index"].astype(np.int64), inp, g["roi_boxes3d"])
    for k in ("pts_feature", "sampled_pts"):
        assert _sha(out[k]) == str(g[k + "_sha256"]), "%s does not rebuild from the stored indices" % k
    return out


def main():
    from oracle import oracle as O
    from pointrcnn_b200 import dropin
    dropin._install_compat()
    sys.path.insert(0, REF)
    # stubs for the two GPU extension wrappers the layer calls
    iou_stub = types.ModuleType("lib.utils.iou3d.iou3d_utils")
    iou_stub.boxes_iou3d_gpu = lambda a, b: torch.from_numpy(O.boxes_iou3d(a.numpy(), b.numpy()))
    rp_stub = types.ModuleType("lib.utils.roipool3d.roipool3d_utils")

    def roipool3d_gpu(pts, pts_feature, boxes3d, pool_extra_width, sampled_pt_num=512):
        big = O.enlarge_box3d(boxes3d.numpy().reshape(-1, 7), pool_extra_width).reshape(boxes3d.shape)
        pooled, empty = O.roipool3d(pts.numpy(), pts_feature.numpy(), big, sampled_pt_num)
        return torch.from_numpy(pooled), torch.from_numpy(empty)
    rp_stub.roipool3d_gpu = roipool3d_gpu
    import lib.utils  # noqa: F401
    for name, mod in (("lib.utils.iou3d", None), ("lib.utils.iou3d.iou3d_utils", iou_stub), ("lib.utils.roipool3d", None),
                      ("lib.utils.roipool3d.roipool3d_utils", rp_stub)):
        if mod is None:
            mod = types.ModuleType(name)
            mod.__path__ = []
        sys.modules[name] = mod
    sys.modules["lib.utils.iou3d"].iou3d_utils = iou_stub
    sys.modules["lib.utils.roipool3d"].roipool3d_utils = rp_stub
    from lib.config import cfg, cfg_from_file
    cfg_from_file(os.path.join(REF, "tools/cfgs/default.yaml"))
    cfg.RCNN.ROI_FG_AUG_TIMES = 0
    cfg.AUG_DATA = False
    from lib.rpn.proposal_target_layer import ProposalTargetLayer
    layer = ProposalTargetLayer()
    inp = inputs()
    np.random.seed(SEED)
    torch.manual_seed(SEED)
    with torch.no_grad():
        out = layer({k: torch.from_numpy(v) for k, v in inp.items()})
    res = {k: v.numpy() for k, v in out.items()}
    print({k: (v.shape, v.dtype) for k, v in res.items()})
    print("cls_label counts", {int(c): int((res["cls_label"] == c).sum()) for c in (-1, 0, 1)}, "reg_valid", int(res["reg_valid_mask"].sum()),
          "iou range", float(res["gt_iou"].min()), float(res["gt_iou"].max()))
    path = os.path.join(ROOT, "tests", "golden", "proposal_target_layer.npz")
    np.savez_compressed(path, **compact(res, inp))
    print("wrote", path, os.path.getsize(path))


if __name__ == "__main__":
    main()
