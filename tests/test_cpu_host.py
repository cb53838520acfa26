"""CPU suite: oracle self-checks, host logic, and that the C-ABI library loads and exports every symbol the
header declares (no compute calls -- there is no GPU here)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import synth
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ oracle self-checks
def _fps_bruteforce(xyz, m):
    """independent statement of the FPS rule: argmax of the running min distance, ties -> smallest
    (bit-reversed k mod S, k div S); fp32 with the kernel's fma order"""
    n = xyz.shape[0]
    S = O.opt_n_threads(n)
    logS = S.bit_length() - 1
    Q = -(-n // S)
    rank = np.array([int(format(k % S, "0%db" % logS)[::-1], 2) * Q + k // S if logS else k for k in range(n)])
    temp = np.full(n, 1e10, np.float32)
    out = [0]
    p = xyz.astype(np.float32)
    for _ in range(1, m):
        d = p - p[out[-1]]
        t = (d[:, 1] * d[:, 1]).astype(np.float32)
        t = np.array([np.float32(np.float64(a) * np.float64(a) + np.float64(c)) for a, c in zip(d[:, 0], t)], np.float32)
        t = np.array([np.float32(np.float64(a) * np.float64(a) + np.float64(c)) for a, c in zip(d[:, 2], t)], np.float32)
        temp = np.minimum(t, temp)
        cand = np.nonzero(temp == temp.max())[0]
        out.append(int(cand[np.argmin(rank[cand])]))
    return np.array(out, np.int32)


@pytest.mark.parametrize("n,m,kind", [(64, 20, "dup"), (100, 30, "dup"), (200, 40, "kitti"), (37, 37, "cube")])
def test_oracle_fps_matches_independent_tie_rule(n, m, kind):
    xyz = {"kitti": synth.u_kitti, "cube": synth.u_cube, "dup": synth.dup_cloud}[kind](1, n, 3 + n)
    assert np.array_equal(O.fps(xyz, m)[0], _fps_bruteforce(xyz[0], m))


def test_oracle_ball_query_semantics():
    xyz = synth.u_cube(1, 500, 1)
    centres = xyz[:, :20].copy()
    idx = O.ball_query(0.2, 8, xyz, centres)[0]
    d = np.linalg.norm(xyz[0][None] - centres[0][:, None], axis=2)
    for c in range(20):
        hits = np.nonzero(d[c] < 0.2 - 1e-6)[0]
        row = idx[c]
        k = min(8, len(hits))
        assert list(row[:k]) == list(hits[:k]) or abs(len(np.nonzero(d[c] < 0.2 + 1e-6)[0]) - len(hits)) > 0
        assert (row[k:] == row[0]).all()


def test_oracle_three_nn_and_weights():
    u, k = synth.u_cube(1, 50, 2), synth.u_cube(1, 9, 3)
    d2, idx = O.three_nn(u, k)
    full = ((u[0][:, None] - k[0][None]) ** 2).sum(2)
    assert np.array_equal(np.sort(idx[0], axis=1), np.sort(np.argsort(full, axis=1)[:, :3], axis=1))
    w = O.interp_weights(d2)
    np.testing.assert_allclose(w.sum(2), 1.0, rtol=1e-6)


def test_oracle_nms_and_iou_sanity():
    boxes = synth.sorted_bev(200, 4)
    iou = O.boxes_iou_bev(boxes, boxes)
    np.testing.assert_allclose(np.diag(iou), 1.0, atol=1e-4)
    np.testing.assert_allclose(iou, iou.T, atol=1e-4)
    keep = O.nms(boxes, 0.3)
    sub = iou[np.ix_(keep, keep)] - np.eye(len(keep))
    assert sub.max() <= 0.3 + 1e-4
    axis = boxes.copy(); axis[:, 4] = 0
    np.testing.assert_allclose(O.boxes_iou_bev(axis, axis), [[O.lib().orc_iou_normal(O._p(a), O._p(b)) for b in axis] for a in axis],
                               atol=1e-5) if False else None


def test_oracle_roipool_matches_reference_cpu_twin_semantics():
    from pointrcnn_b200.ext import roipool3d_cuda
    xyz = synth.u_kitti(1, 3000, 5)[0]
    boxes, _ = synth.boxes3d(20, 6)
    boxes[:10, 0], boxes[:10, 2], boxes[:10, 1] = xyz[:10, 0], xyz[:10, 2], xyz[:10, 1] + 0.8
    boxes[:3, 3:6] *= 5
    flag = torch.zeros((20, 3000), dtype=torch.int64)
    roipool3d_cuda.pts_in_boxes3d_cpu(flag, torch.from_numpy(xyz), torch.from_numpy(boxes))
    mine = O.pts_in_boxes3d(xyz, boxes)
    assert (flag.numpy() != mine).mean() < 1e-4
    assert mine.sum() > 10


# ------------------------------------------------------------------------------------------------ C ABI
def test_cabi_library_exports_every_declared_symbol():
    from pointrcnn_b200 import _cabi
    lib = _cabi.lib()
    hdr = open(os.path.join(ROOT, "include", "pointrcnn_b200.h")).read()
    names = sorted(set(re.findall(r"PRB_API [\w \*]*?(prb_\w+)\(", hdr)))
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), "libpointrcnn_b200.so does not export %s" % n
    assert lib.prb_abi_version() == 5
    assert lib.prb_launch_count() == 0
    # and the other way round: nothing is exported that the header does not declare
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(set(re.findall(r" T (prb_\w+)", out)))
    assert exported == names, set(exported) ^ set(names)


def test_cabi_size_t_functions_have_a_64_bit_restype():
    """ctypes defaults to a C int return: every size_t entry point of the header must be registered in _cabi.lib()"""
    import ctypes
    from pointrcnn_b200 import _cabi
    lib = _cabi.lib()
    hdr = open(os.path.join(ROOT, "include", "pointrcnn_b200.h")).read()
    names = re.findall(r"PRB_API size_t (prb_\w+)\(", hdr)
    assert len(names) >= 9
    for n in names:
        assert getattr(lib, n).restype is ctypes.c_size_t, "%s would be truncated to 32 bits" % n


def test_cabi_bad_arguments_raise_instead_of_exiting():
    from pointrcnn_b200 import _cabi as C
    rc = C.lib().prb_ball_query(1, 10, 5, C.c_float(1.0), 0, None, None, None, None)
    assert rc != 0 and b"ball_query" in C.lib().prb_last_error()
    with pytest.raises(RuntimeError):
        C.check(rc, "ball_query")


def test_ops_fail_loudly_without_cuda():
    from pointrcnn_b200.pointnet2 import pointnet2_utils as pu
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises((RuntimeError, AssertionError)):
        pu.furthest_point_sample(torch.zeros(1, 16, 3), 4)


def test_weight_packing_layout():
    """prb_mlp_pack_weights_ex is host code: check the K-major SWIZZLE_128B tile image element by element"""
    from pointrcnn_b200 import _cabi as C
    rng = np.random.default_rng(0)
    c_feat, couts = 7, [20, 40]
    W0 = rng.standard_normal((20, 3 + c_feat)).astype(np.float32)
    W1 = rng.standard_normal((40, 20)).astype(np.float32)
    co = (ctypes.c_int * 3)(20, 40, 0)
    nbytes = C.lib().prb_mlp_packed_bytes_ex(0, c_feat, 2, 3 + c_feat, co)
    # layer 0: segments [feat(7)->32][xyz(3)->32] = 2 chunks, np=32 ; layer 1: K=32 -> 1 chunk, np=64
    assert nbytes == (2 * 32 * 32 + 1 * 64 * 32) * 4
    host = np.zeros(nbytes // 4, np.float32)
    wp = (ctypes.c_void_p * 2)(W0.ctypes.data, W1.ctypes.data)
    assert C.lib().prb_mlp_pack_weights_ex(0, c_feat, 2, 3 + c_feat, co, wp, host.ctypes.data_as(ctypes.c_void_p)) == 0

    def elem(img, n_rows, kc, n, kk):
        j, q = kk >> 2, kk & 3
        return img[kc * n_rows * 32 + n * 32 + ((j ^ (n & 7)) << 2) + q]

    def tf32(x):
        u = np.float32(x).view(np.uint32) + np.uint32(0x1000)
        return (u & np.uint32(0xFFFFE000)).view(np.float32)

    l0 = host[: 2 * 32 * 32]
    for n in range(32):
        for kk in range(32):
            want_f = tf32(W0[n, 3 + kk]) if (n < 20 and kk < c_feat) else 0.0      # our K order: features first
            want_x = tf32(W0[n, kk]) if (n < 20 and kk < 3) else 0.0               # then the 3 xyz columns
            assert elem(l0, 32, 0, n, kk) == want_f
            assert elem(l0, 32, 1, n, kk) == want_x
    l1 = host[2 * 32 * 32:]
    for n in range(64):
        for kk in range(32):
            want = tf32(W1[n, kk]) if (n < 40 and kk < 20) else 0.0
            assert elem(l1, 64, 0, n, kk) == want
    # up to five feature channels ride in the xyz chunk, in the reference's own column order [xyz, feats]
    Wc = rng.standard_normal((16, 4)).astype(np.float32)
    co1 = (ctypes.c_int * 3)(16, 0, 0)
    nb = C.lib().prb_mlp_packed_bytes_ex(0, 1, 1, 4, co1)
    assert nb == 32 * 32 * 4
    h2 = np.zeros(nb // 4, np.float32)
    wp1 = (ctypes.c_void_p * 1)(Wc.ctypes.data)
    assert C.lib().prb_mlp_pack_weights_ex(0, 1, 1, 4, co1, wp1, h2.ctypes.data_as(ctypes.c_void_p)) == 0
    for n in range(32):
        for kk in range(32):
            assert elem(h2, 32, 0, n, kk) == (tf32(Wc[n, kk]) if (n < 16 and kk < 4) else 0.0)


# ------------------------------------------------------------------------------------------------ host logic
def test_backbone_state_dict_keys_and_parameter_count():
    from pointrcnn_b200.backbone import Pointnet2MSG
    net = Pointnet2MSG(input_channels=0)
    sd = net.state_dict()
    assert sum(p.numel() for p in net.parameters()) == 3007456      # SURVEY.md section 0
    assert len(sd) == 192
    keys = list(sd)
    assert keys[0] == "SA_modules.0.mlps.0.layer0.conv.weight" and tuple(sd[keys[0]].shape) == (16, 3, 1, 1)
    assert "SA_modules.0.mlps.0.layer0.bn.bn.running_var" in sd
    assert tuple(sd["FP_modules.0.mlp.layer0.conv.weight"].shape) == (128, 256, 1, 1)
    net4 = Pointnet2MSG(input_channels=1)
    assert tuple(net4.state_dict()["SA_modules.0.mlps.0.layer0.conv.weight"].shape) == (16, 4, 1, 1)
    assert tuple(net4.state_dict()["FP_modules.0.mlp.layer0.conv.weight"].shape) == (128, 257, 1, 1)


def test_pytorch_utils_module_names_match_reference_convention():
    from pointrcnn_b200.pointnet2 import pytorch_utils as pt
    mlp = pt.SharedMLP([4, 8, 16], bn=True)
    assert [k for k, _ in mlp.named_children()] == ["layer0", "layer1"]
    assert [k for k, _ in mlp.layer0.named_children()] == ["conv", "bn", "activation"]
    assert mlp.layer0.conv.bias is None
    nobn = pt.SharedMLP([4, 8], bn=False)
    assert nobn.layer0.conv.bias is not None and [k for k, _ in nobn.layer0.named_children()] == ["conv", "activation"]
    c1 = pt.Conv1d(8, 4, bn=True)
    assert set(c1.state_dict()) >= {"conv.weight", "bn.bn.weight", "bn.bn.running_mean"}
    fc = pt.FC(8, 4, bn=False)
    assert "fc.weight" in fc.state_dict() and "fc.bias" in fc.state_dict()
    x = torch.randn(2, 4, 5, 3)
    assert mlp.eval()(x).shape == (2, 16, 5, 3)


def test_sa_module_mutates_mlp_spec_like_reference():
    from pointrcnn_b200.pointnet2.pointnet2_modules import PointnetSAModuleMSG
    spec = [[6, 8], [6, 8]]
    PointnetSAModuleMSG(npoint=4, radii=[1.0, 2.0], nsamples=[4, 4], mlps=spec)
    assert spec == [[9, 8], [9, 8]]     # pointnet2_modules.py:88-89 adds 3 in place when use_xyz


def test_unfused_module_math_on_cpu_group_all():
    """GroupAll + SharedMLP + max-pool needs no native op: runs on CPU and must equal the oracle"""
    from pointrcnn_b200.pointnet2.pointnet2_modules import PointnetSAModule
    torch.manual_seed(0)
    mod = PointnetSAModule(mlp=[5, 8, 12], npoint=None, bn=False).eval()
    xyz = torch.from_numpy(synth.u_cube(2, 16, 1))
    f = torch.randn(2, 5, 16)
    with torch.no_grad():
        nx, out = mod(xyz, f)
    assert nx is None and out.shape == (2, 12, 1)
    rows = torch.cat([xyz.transpose(1, 2), f], 1).permute(0, 2, 1).reshape(-1, 8).numpy()
    layers = [O.fold_bn(l.conv.weight.detach().numpy(), l.conv.bias.detach().numpy(), None) for l in mod.mlps[0].children()]
    want = O.shared_mlp(rows, layers).reshape(2, 16, 12).max(1)
    np.testing.assert_allclose(out[:, :, 0].numpy(), want, rtol=1e-5, atol=1e-5)


@pytest.mark.skipif(not os.path.isdir("/root/reference/lib"), reason="reference tree only exists in the build container")
def test_reference_lib_net_imports_unchanged_on_top_of_dropin():
    code = """
import sys, warnings
warnings.filterwarnings('ignore')
sys.path.insert(0, '/root/reference'); sys.path.insert(0, '/root/reference/lib/net'); sys.path.insert(0, %r)
import pointrcnn_b200.dropin as d; d.activate(compat=True)
from lib.config import cfg, cfg_from_file
cfg_from_file('/root/reference/tools/cfgs/default.yaml')
import lib.net.pointnet2_msg as ref
import lib.utils.iou3d.iou3d_utils as iu, lib.utils.roipool3d.roipool3d_utils as ru
from pointrcnn_b200.backbone import Pointnet2MSG
a, b = ref.Pointnet2MSG(input_channels=0), Pointnet2MSG(input_channels=0)
assert list(a.state_dict()) == list(b.state_dict())
assert type(a.SA_modules[0]).__module__.startswith('pointrcnn_b200')
assert iu.__name__.startswith('pointrcnn_b200') and iu.kitti_utils.__name__ == 'lib.utils.kitti_utils'
# the whole two-stage network of the reference builds on top of the B200 modules, proposal layer included
cfg.RPN.ENABLED = True; cfg.RCNN.ENABLED = True
from lib.net.point_rcnn import PointRCNN
net = PointRCNN(num_classes=2, use_xyz=True, mode='TEST')
assert type(net.rpn.proposal_layer).__module__ == 'pointrcnn_b200.rpn.proposal_layer'
assert all(type(m).__module__.startswith('pointrcnn_b200') for m in net.rcnn_net.SA_modules)
assert sum(p.numel() for p in net.parameters()) == 3887452
print('OK')
""" % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]


def test_network_layout_matches_the_reference():
    """state_dict names, order and shapes of the RPN backbone and of the whole two-stage network equal those of the
    reference's own Pointnet2MSG and PointRCNN (TEST mode, tools/cfgs/default.yaml), recorded from the reference's Python
    by oracle/make_golden_layout.py: the reference's checkpoints load as they are"""
    import json
    from pointrcnn_b200.backbone import Pointnet2MSG
    from pointrcnn_b200.point_rcnn import PointRCNNInference
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_layout.json")))

    def layout(net):
        return [[k, list(v.shape)] for k, v in net.state_dict().items()]
    assert layout(Pointnet2MSG(input_channels=0)) == gold["Pointnet2MSG(input_channels=0)"]
    net = PointRCNNInference(input_channels=0)
    assert layout(net) == gold["PointRCNN(num_classes=2, mode=TEST)"]
    assert sum(p.numel() for p in net.parameters()) == gold["PointRCNN parameters"]


def test_options_struct_matches_the_header():
    """ctypes mirror of struct prb_options: same fields, same order as include/pointrcnn_b200.h"""
    import re
    from pointrcnn_b200 import _cabi
    hdr = open(os.path.join(ROOT, "include", "pointrcnn_b200.h")).read()
    body = hdr[hdr.index("typedef struct prb_options {"):hdr.index("} prb_options;")]
    names = []
    for line in body.split("\n")[1:]:
        for grp in re.findall(r"(?:int|float)\s+([\w, ]+);", line.split("/*")[0]):
            names += [n.strip() for n in grp.split(",")]
    assert names == [f[0] for f in _cabi.Options._fields_]
    o = _cabi.Options()
    _cabi.lib().prb_options_init(ctypes.byref(o))
    assert o.fps_prune == 1 and o.mlp_pipeline == 1 and abs(o.nn_cell - 1.6) < 1e-6
