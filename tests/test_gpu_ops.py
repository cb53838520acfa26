"""GPU parity tests (run with -m gpu on the B200 box): every native of the C ABI against
  (1) the CPU oracle (oracle/pointops_oracle.c, bit-exact for index work), and
  (2) the reference's own CUDA kernels rebuilt for sm_100a (oracle/_ref): their recorded outputs (tests/refstore.py), and
      the live kernels as well when that library is present.
Calls go through the reference-named extension modules / Python wrappers, i.e. through the C ABI.
"""
import os

import numpy as np
import pytest
import torch

import refstore as REF
import synth
from oracle import oracle as O
from oracle import refgpu as R

pytestmark = pytest.mark.gpu

from pointrcnn_b200.ext import iou3d_cuda, roipool3d_cuda  # noqa: E402
from pointrcnn_b200.iou3d import iou3d_utils  # noqa: E402
from pointrcnn_b200.pointnet2 import pointnet2_utils as pu  # noqa: E402
from pointrcnn_b200.roipool3d import roipool3d_utils  # noqa: E402


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ------------------------------------------------------------------------------------------------ FPS
FPS_CASES = [
    # (B, N, M, cloud)            what it exercises
    (2, 16384, 4096, "kitti"),    # pruned single-CTA kernel, 4095 rounds (RPN SA1 shape)
    (2, 16384, 2048, "cube"),     # pruned, uniform cloud
    (3, 10000, 700, "kitti"),     # pruned with 6384 pad points
    (2, 5000, 5000, "kitti"),     # pruned, 16 slots, m == n
    (2, 8192, 600, "dup"),        # pruned + ties
    (3, 4096, 1024, "kitti"),     # single CTA 512x8
    (3, 1024, 256, "cube"),
    (5, 256, 64, "kitti"),
    (7, 512, 128, "dup"),         # RCNN SA1 shape, duplicate-heavy (tie rule)
    (7, 128, 32, "dup"),
    (2, 300, 50, "kitti"),        # n not a power of two: S=256, Q=2, holes in the rank space
    (2, 1500, 100, "dup"),        # S=1024, Q=2
    (1, 20000, 64, "kitti"),      # rank copy does not fit shared memory
    (2, 16384, 300, "dup"),       # cluster + ties
    (1, 70, 70, "cube"),          # m == n, tiny
]


def _cloud(kind, B, N, seed):
    return {"kitti": synth.u_kitti, "cube": synth.u_cube, "dup": synth.dup_cloud}[kind](B, N, seed)


@pytest.mark.parametrize("B,N,M,kind", FPS_CASES)
def test_fps_index_exact(cuda, B, N, M, kind):
    xyz = _cloud(kind, B, N, 11 + N)
    want, want_temp = O.fps(xyz, M, return_temp=True)
    x = T(xyz, cuda)
    got = pu.furthest_point_sample(x, M)
    assert got.dtype == torch.int32 and tuple(got.shape) == (B, M)
    assert np.array_equal(got.cpu().numpy(), want), "FPS indices differ from the oracle"
    idx2, new_xyz = pu.furthest_point_sample_xyz(x, M)
    assert np.array_equal(idx2.cpu().numpy(), want)
    exp_xyz = np.stack([xyz[b][want[b]] for b in range(B)])
    assert np.array_equal(new_xyz.cpu().numpy(), exp_xyz), "emitted new_xyz != xyz[idx]"
    REF.equal("idx", got, lambda: R.fps(x, M), "FPS indices differ from the reference kernel")
    REF.equal("temp", want_temp, lambda: R.fps(x, M, return_temp=True)[1], "oracle temp != reference temp")


@pytest.mark.parametrize("opt", [{"fps_cluster": 1}, {"fps_cluster": 2}, {"fps_cluster": 4}, {"fps_cluster": 8},
                                 {"fps_generic": 1}, {"fps_cluster": 1, "fps_threads": 1024}, {"fps_prune": 1},
                                 {"fps_prune": 2, "fps_threads": 1024}])     # pruned kernel, 32 warps x half the slots
def test_fps_all_kernel_variants_agree(cuda, opt):
    from pointrcnn_b200 import _cabi
    xyz = synth.dup_cloud(2, 8192, 5, unique=3000)
    want = O.fps(xyz, 512)
    opt = dict({"fps_prune": 0}, **opt)     # the cluster / generic kernels unless the case asks for pruning
    with _cabi.options(**opt):              # per-thread prb_options, not the process environment
        got = pu.furthest_point_sample(T(xyz, cuda), 512)
    assert np.array_equal(got.cpu().numpy(), want)


ORDERED_CASES = [
    # (B, N0, levels, cloud): nested sampling levels as the encoder runs them (pointnet2_msg.py:57-61)
    (3, 16384, [4096, 1024, 256, 64], "kitti"),   # the RPN encoder
    (2, 8192, [2048, 512, 100], "cube"),
    (2, 4096, [1024, 1024, 300], "kitti"),        # m == n at the second level
    (4, 2048, [1024, 600], "dup"),                 # 512 distinct points: picks beyond them have distance 0 -> no proof, kernels sample
]


@pytest.mark.parametrize("B,N0,levels,kind", ORDERED_CASES)
def test_fps_ordered_levels_identical_to_sampling(cuda, B, N0, levels, kind):
    """the proven-prefix shortcut returns exactly what the sampling kernels (and the oracle) return at every nested level"""
    from pointrcnn_b200.ext import pointnet2_cuda
    from pointrcnn_b200 import _cabi as C
    xyz = _cloud(kind, B, N0, 23 + N0)
    x = T(xyz, cuda)
    proven = []
    for li, m in enumerate(levels):
        n = x.size(1)
        idx_o, nx_o, todo = pu.furthest_point_sample_xyz(x, m, ordered=True, return_todo=True)
        idx_p, nx_p = pu.furthest_point_sample_xyz(x, m, ordered=False)
        assert torch.equal(idx_o, idx_p), "level %d: ordered path differs from the sampling kernels" % li
        assert torch.equal(nx_o, nx_p)
        want, want_temp = O.fps(x.cpu().numpy(), m, return_temp=True)
        assert np.array_equal(idx_o.cpu().numpy(), want), "level %d: differs from the oracle" % li
        # temp written by the proof == temp written by the kernels == the oracle's
        lib = C.lib()
        wsb = lib.prb_fps_ordered_workspace_bytes(B, n, m)
        ws = torch.empty(wsb, dtype=torch.uint8, device=cuda)
        temp = torch.full((B, n), 1e10, device=cuda)
        idx2 = torch.empty((B, m), dtype=torch.int32, device=cuda)
        C.check(lib.prb_furthest_point_sampling_ordered_ws(B, n, m, C.ptr(x), C.ptr(temp), C.ptr(idx2), None, None, C.ptr(ws),
                                                           C.c_size_t(wsb), C.stream()), "fps_ordered")
        assert np.array_equal(temp.cpu().numpy(), want_temp), "level %d: temp differs from the oracle" % li
        assert torch.equal(idx2, idx_p)
        proven.append(int((todo == 0).sum()))
        x = nx_o
    if kind in ("kitti", "cube"):
        assert proven[0] == 0, "raw clouds are not in sampling order"
        assert all(p == B for p in proven[1:]), "nested levels of a tie-free cloud must be answered by the proof: %s" % proven
    else:
        assert proven[-1] == 0, "a level that runs out of distinct points cannot be proven"


def test_fps_ordered_mixed_batch_and_caller_temp(cuda):
    """per-scene decision: scene 0 in sampling order, scene 1 shuffled, scene 2 ordered but with one exact tie;
    plus a caller-initialised temp (in/out contract) -- all identical to the plain entry"""
    from pointrcnn_b200 import _cabi as C
    base = synth.u_kitti(3, 4096, 77)
    order = O.fps(base, 1024)
    lvl = np.stack([base[b][order[b]] for b in range(3)])          # (3,1024,3) in sampling order
    rng = np.random.default_rng(3)
    lvl[1] = lvl[1][rng.permutation(1024)]
    lvl[2][200] = lvl[2][100]                                       # duplicate of an early pick: v_200 == 0
    x = T(lvl, cuda)
    for t0 in (None, (rng.random((3, 1024)) * 50.0 + 1.0).astype(np.float32)):
        lib = C.lib()
        m = 256
        wsb = lib.prb_fps_ordered_workspace_bytes(3, 1024, m)
        ws = torch.empty(wsb, dtype=torch.uint8, device=cuda)
        temp = torch.full((3, 1024), 1e10, device=cuda) if t0 is None else T(t0.copy(), cuda)
        idx = torch.empty((3, m), dtype=torch.int32, device=cuda)
        nx = torch.empty((3, m, 3), device=cuda)
        todo = torch.empty(3, dtype=torch.int32, device=cuda)
        C.check(lib.prb_furthest_point_sampling_ordered_ws(3, 1024, m, C.ptr(x), C.ptr(temp), C.ptr(idx), C.ptr(nx), C.ptr(todo),
                                                           C.ptr(ws), C.c_size_t(wsb), C.stream()), "fps_ordered")
        want, want_temp = O.fps(lvl, m, return_temp=True, temp0=t0)
        assert np.array_equal(idx.cpu().numpy(), want)
        assert np.array_equal(temp.cpu().numpy(), want_temp)
        assert np.array_equal(nx.cpu().numpy(), np.stack([lvl[b][want[b]] for b in range(3)]))
        if t0 is None:
            assert todo.tolist() == [0, 1, 1]


@pytest.mark.parametrize("case", ["nan", "inf", "tiny", "all_equal", "single_scene"])
def test_fps_ordered_degenerate_inputs_equal_the_plain_entry(cuda, case):
    """whatever the input, the ordered entry returns what the sampling kernels return (the proof simply fails)"""
    base = synth.u_kitti(3, 1024, 91)
    order = O.fps(base, 256)
    lvl = np.stack([base[b][order[b]] for b in range(3)])
    m = 64
    if case == "nan":
        lvl[0, 100, 1] = np.nan
        lvl[1, 10, :] = np.nan
    elif case == "inf":
        lvl[0, 7, 0] = np.inf
        lvl[2, 200, 2] = -np.inf
    elif case == "tiny":
        lvl, m = lvl[:, :2].copy(), 2
    elif case == "all_equal":
        lvl[1] = lvl[1, 0]
    elif case == "single_scene":
        lvl = lvl[:1].copy()
    x = T(lvl, cuda)
    idx_o, nx_o, todo = pu.furthest_point_sample_xyz(x, m, ordered=True, return_todo=True)
    idx_p, nx_p = pu.furthest_point_sample_xyz(x, m, ordered=False)
    assert torch.equal(idx_o, idx_p)
    assert np.array_equal(nx_o.cpu().numpy(), nx_p.cpu().numpy(), equal_nan=True)
    if case == "all_equal":
        assert todo[1].item() == 1
    if case in ("tiny", "single_scene"):
        assert int(todo.sum()) == 0


def test_fps_ordered_settles_exact_ties_with_the_reference_rank_rule(cuda):
    """~2 % of uniform 4096-point levels hold an exact fp32 tie between two consecutive picks k, k+1.  The proof applies the
    sampling kernels' tie rule (smaller reference rank wins): scene A (tie at even k = 718: rank(k) < rank(k+1)) is proven,
    scene B (tie at odd k = 679: pick k+1 wins the tie) goes to the kernels; both equal the plain entry and the oracle."""
    import bench
    scenes = []
    for first, s in ((32, 1), (96, 7)):                  # bench pool scenes found by replaying the proof on the CPU
        pc = bench.make_scenes(first, 16)[s:s + 1, :, :3].copy()
        idx = O.fps(np.ascontiguousarray(pc), 4096)
        scenes.append(pc[0][idx[0]])
    lvl = np.stack(scenes)
    x = T(lvl, cuda)
    idx_o, nx_o, todo = pu.furthest_point_sample_xyz(x, 1024, ordered=True, return_todo=True)
    idx_p, nx_p = pu.furthest_point_sample_xyz(x, 1024, ordered=False)
    want = O.fps(lvl, 1024)
    assert torch.equal(idx_o, idx_p) and torch.equal(nx_o, nx_p)
    assert np.array_equal(idx_o.cpu().numpy(), want)
    assert np.array_equal(want[0], np.arange(1024)), "scene A: the tie is won by pick k"
    assert want[1][679] == 680 and want[1][680] == 679, "scene B: the tie is won by pick k+1 (a transposition)"
    assert todo.tolist() == [0, 1]


def test_backbone_takes_the_ordered_shortcut(cuda):
    """SA levels 2..4 of the fused encoder receive tagged coordinates; switching the shortcut off changes nothing"""
    from pointrcnn_b200 import backbone, config
    torch.manual_seed(0)
    net = backbone.get_model(input_channels=0).to(cuda).eval()
    pc = T(synth.u_kitti(2, 16384, 5), cuda)
    with torch.no_grad():
        xyz_a, f_a = net(pc)
        with config.override(fps_ordered=False):
            xyz_b, f_b = net(pc)
    assert torch.equal(f_a, f_b) and torch.equal(xyz_a, xyz_b)


def test_options_are_thread_local(cuda):
    """SURVEY 8(b): natives are re-entered from nn.DataParallel worker threads; one thread's prb_options must not leak"""
    import threading
    from pointrcnn_b200 import _cabi
    seen = {}

    def worker():
        o = _cabi.Options()
        _cabi.lib().prb_get_thread_options(ctypes.byref(o))
        seen["worker"] = (o.fps_cluster, o.fps_prune)
    import ctypes
    with _cabi.options(fps_cluster=8, fps_prune=0):
        t = threading.Thread(target=worker); t.start(); t.join()
        o = _cabi.Options()
        _cabi.lib().prb_get_thread_options(ctypes.byref(o))
        seen["main"] = (o.fps_cluster, o.fps_prune)
    assert seen["main"] == (8, 0) and seen["worker"] != (8, 0)


def test_fps_temp_writeback_and_m_edge(cuda):
    from pointrcnn_b200.ext import pointnet2_cuda
    xyz = synth.u_kitti(2, 2048, 3)
    x = T(xyz, cuda)
    temp = torch.full((2, 2048), 1e10, device=cuda)
    idx = torch.empty((2, 100), dtype=torch.int32, device=cuda)
    pointnet2_cuda.furthest_point_sampling_wrapper(2, 2048, 100, x, temp, idx)
    _, want_temp = O.fps(xyz, 100, return_temp=True)
    assert np.array_equal(temp.cpu().numpy(), want_temp)
    one = pu.furthest_point_sample(x, 1)
    assert torch.count_nonzero(one) == 0


@pytest.mark.parametrize("N,M,prune", [(6000, 300, 1), (16384, 1000, 1), (3000, 200, 2)])
def test_fps_pruned_kernel_resumes_from_caller_temp(cuda, N, M, prune):
    """temp is in/out (sampling_gpu.cu:105-111): a caller-initialised temp steers the sampling and gets the final minima"""
    from pointrcnn_b200.ext import pointnet2_cuda
    xyz = synth.u_kitti(2, N, 17)
    rng = np.random.default_rng(5)
    t0 = (rng.random((2, N)) * 30.0).astype(np.float32)
    t0[:, ::7] = 1e10
    want, want_temp = O.fps(xyz, M, return_temp=True, temp0=t0)
    x = T(xyz, cuda)
    temp = T(t0.copy(), cuda)
    idx = torch.empty((2, M), dtype=torch.int32, device=cuda)
    from pointrcnn_b200 import _cabi
    with _cabi.options(fps_prune=prune):
        pointnet2_cuda.furthest_point_sampling_wrapper(2, N, M, x, temp, idx)
    assert np.array_equal(idx.cpu().numpy(), want)
    assert np.array_equal(temp.cpu().numpy(), want_temp)
    def ref_fps():
        rt = T(t0.copy(), cuda)
        ridx = torch.empty((2, M), dtype=torch.int32, device=cuda)
        R.fps_raw(x, rt, ridx)
        return ridx, rt
    REF.equal("idx", idx, lambda: ref_fps()[0])
    REF.equal("temp", temp, lambda: ref_fps()[1])


# ------------------------------------------------------------------------------------------------ ball query / grouping
@pytest.mark.parametrize("kind,N,M,r,ns", [("cube", 16384, 4096, 0.1, 32), ("kitti", 16384, 4096, 0.5, 32),
                                           ("kitti", 4096, 1024, 1.0, 16), ("cube", 1000, 77, 0.3, 64),
                                           ("dup", 512, 128, 0.2, 64), ("kitti", 256, 64, 4.0, 32)])
def test_ball_query_exact(cuda, kind, N, M, r, ns):
    xyz = _cloud(kind, 2, N, 21 + N)
    fidx = O.fps(xyz, M)
    new_xyz = np.stack([xyz[b][fidx[b]] for b in range(2)])
    want = O.ball_query(r, ns, xyz, new_xyz)
    x, c = T(xyz, cuda), T(new_xyz, cuda)
    got = pu.ball_query(r, ns, x, c)
    assert np.array_equal(got.cpu().numpy(), want)
    REF.equal("idx", got, lambda: R.ball_query(r, ns, x, c))


def test_ball_query_no_hit_rows_stay_zero_and_msg2(cuda):
    xyz = synth.u_kitti(2, 4096, 9)
    centres = xyz[:, :128].copy()
    centres[:, ::2] += 500.0   # every other centre is far from everything
    x, c = T(xyz, cuda), T(centres, cuda)
    a = pu.ball_query(0.5, 16, x, c)
    assert torch.count_nonzero(a[:, ::2]) == 0
    assert np.array_equal(a.cpu().numpy(), O.ball_query(0.5, 16, xyz, centres))
    i0, i1 = pu.ball_query_msg2((0.5, 1.0), (16, 32), x, c)
    assert torch.equal(i0, a)
    assert torch.equal(i1, pu.ball_query(1.0, 32, x, c))


def test_group_gather_and_grads(cuda):
    rng = np.random.default_rng(0)
    B, C, N, M, S = 2, 19, 777, 60, 16
    feats = rng.standard_normal((B, C, N)).astype(np.float32)
    idx = rng.integers(0, N, (B, M, S)).astype(np.int32)
    f, i = T(feats, cuda), T(idx, cuda)
    got = pu.grouping_operation(f, i)
    assert np.array_equal(got.cpu().numpy(), O.group(feats, idx))
    gidx = idx[:, :, 0].copy()
    g2 = pu.gather_operation(f, T(gidx, cuda))
    assert np.array_equal(g2.cpu().numpy(), O.gather(feats, gidx))
    # backward: scatter-add (atomic order differs -> tolerance)
    fr = f.clone().requires_grad_(True)
    go = rng.standard_normal((B, C, M, S)).astype(np.float32)
    pu.grouping_operation(fr, i).backward(T(go, cuda))
    np.testing.assert_allclose(fr.grad.cpu().numpy(), O.group_grad(go, idx, N), rtol=1e-5, atol=1e-5)
    fr2 = f.clone().requires_grad_(True)
    go2 = rng.standard_normal((B, C, M)).astype(np.float32)
    pu.gather_operation(fr2, T(gidx, cuda)).backward(T(go2, cuda))
    np.testing.assert_allclose(fr2.grad.cpu().numpy(), O.gather_grad(go2, gidx, N), rtol=1e-5, atol=1e-5)
    REF.equal("group", got, lambda: R.group(f, i))


# ------------------------------------------------------------------------------------------------ three_nn / interpolate
@pytest.mark.parametrize("n,m,kind", [(16384, 4096, "kitti"), (1024, 256, "cube"), (256, 64, "dup"), (100, 2, "kitti"), (33, 3, "cube")])
def test_three_nn_exact(cuda, n, m, kind):
    unknown = _cloud(kind, 2, n, 31 + n)
    known = np.ascontiguousarray(unknown[:, ::max(1, n // m)][:, :m])
    d2, idx = O.three_nn(unknown, known)
    u, k = T(unknown, cuda), T(known, cuda)
    dist, gi = pu.three_nn(u, k)
    assert np.array_equal(gi.cpu().numpy(), idx)
    got_d2, _, w = pu.three_nn_weights(u, k)
    assert np.array_equal(got_d2.cpu().numpy(), d2)
    np.testing.assert_allclose(dist.cpu().numpy(), np.sqrt(d2), rtol=1e-6)
    if m >= 3:
        np.testing.assert_allclose(w.cpu().numpy(), O.interp_weights(d2), rtol=2e-6, atol=1e-7)
    REF.equal("idx", gi, lambda: R.three_nn(u, k)[1])
    REF.equal("dist2", got_d2, lambda: R.three_nn(u, k)[0])


def test_three_interpolate_and_grad(cuda):
    rng = np.random.default_rng(1)
    B, C, M, N = 2, 37, 300, 1000
    feats = rng.standard_normal((B, C, M)).astype(np.float32)
    idx = rng.integers(0, M, (B, N, 3)).astype(np.int32)
    w = rng.random((B, N, 3)).astype(np.float32)
    w /= w.sum(axis=2, keepdims=True)
    f, i, ww = T(feats, cuda), T(idx, cuda), T(w, cuda)
    got = pu.three_interpolate(f, i, ww)
    want = O.three_interpolate(feats, idx, w)
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=1e-6)   # north_star: 1e-5 rel
    assert np.array_equal(got.cpu().numpy(), want), "same FMA order as the reference SASS -> expected bit-exact"
    fr = f.clone().requires_grad_(True)
    go = rng.standard_normal((B, C, N)).astype(np.float32)
    pu.three_interpolate(fr, i, ww).backward(T(go, cuda))
    np.testing.assert_allclose(fr.grad.cpu().numpy(), O.three_interpolate_grad(go, idx, w, M), rtol=1e-4, atol=1e-4)
    REF.equal("out", got, lambda: R.three_interpolate(f, i, ww))


# ------------------------------------------------------------------------------------------------ roipool3d
def _roi_scene(B, N, M, C, seed):
    rng = np.random.default_rng(seed)
    xyz = synth.u_kitti(B, N, seed)
    boxes = np.stack([synth.boxes3d(M, seed + b)[0] for b in range(B)])
    # make boxes land on points: move a third of them onto random points, blow some up to saturate 512
    for b in range(B):
        pick = rng.integers(0, N, M // 3)
        boxes[b, : M // 3, 0] = xyz[b, pick, 0]
        boxes[b, : M // 3, 2] = xyz[b, pick, 2]
        boxes[b, : M // 3, 1] = xyz[b, pick, 1] + 0.8
        boxes[b, : M // 8, 3:6] *= 6.0
        boxes[b, -max(2, M // 8):, 0] += 500.0      # far from every point -> empty boxes
    feat = rng.standard_normal((B, N, C)).astype(np.float32)
    return xyz, boxes.astype(np.float32), feat


@pytest.mark.parametrize("B,N,M,C,S", [(2, 16384, 64, 130, 512), (1, 4096, 33, 5, 128), (2, 2000, 16, 0, 64)])
def test_roipool3d_vs_reference_and_oracle(cuda, B, N, M, C, S):
    xyz, boxes, feat = _roi_scene(B, N, M, C, 41 + N)
    x, bx, f = T(xyz, cuda), T(boxes, cuda), T(feat, cuda)
    pooled = torch.zeros((B, M, S, 3 + C), device=cuda)
    empty = torch.zeros((B, M), dtype=torch.int32, device=cuda)
    roipool3d_cuda.forward(x, bx, f, pooled, empty)
    from pointrcnn_b200 import _cabi
    for alt in ({"roipool_direct": 1}, {"roipool_stage_kb": 8}, {"roipool_parts": 3}):   # scalar-gather path; tiny staging area
        p2 = torch.zeros_like(pooled); e2 = torch.zeros_like(empty)                       # (every box chunked); 3 CTAs per box
        with _cabi.options(**alt):
            roipool3d_cuda.forward(x, bx, f, p2, e2)
        assert torch.equal(p2, pooled) and torch.equal(e2, empty), "pass-B variant %r differs" % alt
    if C > 0:
        REF.equal("empty", empty, lambda: R.roipool3d(x, f, bx, S)[1], "empty flags differ from the reference kernel")
        REF.equal("pooled", pooled, lambda: R.roipool3d(x, f, bx, S)[0], "pooled rows differ from the reference kernel")
    # CPU oracle uses host libm for cos/sin: flags may differ only for points within 1e-4 m of a box face
    op, oe = O.roipool3d(xyz, feat, boxes, S)
    gp, ge = pooled.cpu().numpy(), empty.cpu().numpy()
    same = np.all(gp.reshape(B, M, -1) == op.reshape(B, M, -1), axis=2) & (ge == oe)
    assert same.mean() > 0.97, "too many boxes disagree with the CPU oracle: %f" % same.mean()
    assert ge.sum() > 0 and (1 - ge).sum() > 0, "test should cover empty and non-empty boxes"
    for b, m in zip(*np.nonzero(~same)):
        mg = O.pts_in_boxes3d_margin(xyz[b], boxes[b, m:m + 1])[0]
        assert mg.min() < 1e-4, "non-borderline roipool3d mismatch at scene %d box %d" % (b, m)


@pytest.mark.parametrize("case", ["duplicates", "degenerate_line", "nan_inf", "huge_boxes", "tiny", "odd_n", "far_coordinates"])
def test_roipool3d_binned_equals_exhaustive(cuda, case):
    """the x-z binned assign pass (default) must select exactly the rows of the exhaustive scan: same predicate, the
    footprint only prunes cells that cannot hold an inside point.  Degenerate clouds and boxes included."""
    from pointrcnn_b200 import _cabi as C
    rng = np.random.default_rng(len(case))
    B, N, M, Cf, S = 2, 5000, 40, 7, 64
    xyz, boxes, feat = _roi_scene(B, N, M, Cf, 300 + len(case))
    if case == "duplicates":
        xyz[:, N // 2:] = xyz[:, :N - N // 2]                      # every point twice: ties in every cell
    elif case == "degenerate_line":
        xyz[0, :, 0] = 3.0                                         # zero x extent: one grid column
        xyz[1, :, :] = xyz[1, 0, :]                                # a single location
        boxes[:, :10, 0:3] = xyz[:, :10, :] + np.float32(0.3)
    elif case == "nan_inf":
        xyz[0, ::7, 0] = np.nan; xyz[0, 3::11, 2] = np.inf; xyz[1, 5::13, 1] = -np.inf
        boxes[0, 0, 0] = np.nan; boxes[0, 1, 6] = np.inf; boxes[1, 2, 5] = np.nan
    elif case == "huge_boxes":
        boxes[:, :8, 3:6] = 500.0                                  # the |dx|, |dz| <= 10 m rule of pt_in_box3d caps them
        boxes[:, 8:12, 3:6] = -1.0                                 # negative sizes: nothing inside
    elif case == "tiny":
        N = 1
        xyz, feat = xyz[:, :1].copy(), feat[:, :1].copy()
        boxes[:, 0, 0:3] = xyz[:, 0, :] + np.array([0, 0.5, 0], dtype=np.float32)
    elif case == "odd_n":
        N = 4099
        xyz, feat = xyz[:, :N].copy(), feat[:, :N].copy()
    elif case == "far_coordinates":
        xyz += np.float32(30000.0); boxes[:, :, 0:3] += np.float32(30000.0)     # coarse fp32 spacing around the boxes
    x, bx, f = T(xyz, cuda), T(boxes, cuda), T(feat, cuda)
    out = []
    # binned as two kernels (default), exhaustive, binned with the assign pass fused into the copy kernel
    for opt in (dict(roipool_exhaustive=0, roipool_fused=0), dict(roipool_exhaustive=1), dict(roipool_exhaustive=0, roipool_fused=1)):
        pooled = torch.zeros((B, M, S, 3 + Cf), device=cuda)
        empty = torch.zeros((B, M), dtype=torch.int32, device=cuda)
        with C.options(**opt):
            roipool3d_cuda.forward(x, bx, f, pooled, empty)
        torch.cuda.synchronize()
        out.append((pooled.cpu().numpy(), empty.cpu().numpy()))
    assert np.array_equal(out[0][1], out[1][1]) and np.array_equal(out[2][1], out[1][1]), "empty flags differ"
    assert np.array_equal(out[0][0].view(np.uint32), out[1][0].view(np.uint32)), "pooled rows differ (bitwise)"
    assert np.array_equal(out[2][0].view(np.uint32), out[1][0].view(np.uint32)), "pooled rows differ (bitwise, fused form)"
    if case in ("duplicates", "huge_boxes", "odd_n", "far_coordinates"):
        assert (out[0][1] == 0).sum() > 0, "case should have non-empty boxes"


def test_roipool3d_utils_and_canonical(cuda):
    xyz, boxes, feat = _roi_scene(2, 8192, 48, 6, 77)
    x, bx, f = T(xyz, cuda), T(boxes, cuda), T(feat, cuda)
    pooled, empty = roipool3d_utils.roipool3d_gpu(x, f, bx, 1.0, sampled_pt_num=256)
    large = O.enlarge_box3d(boxes, 1.0)
    op, oe = O.roipool3d(xyz, feat, large, 256)
    ok = np.all(pooled.cpu().numpy().reshape(2, 48, -1) == op.reshape(2, 48, -1), axis=2)
    assert ok.mean() > 0.95
    pc, ec = roipool3d_utils.roipool3d_gpu(x, f, bx, 1.0, sampled_pt_num=256, canonical_rois=bx)
    assert torch.equal(ec, empty)
    # the reference transforms EVERY RoI's rows, empty ones (all-zero rows) included (rcnn_net.py:146-152): so does the fused form
    want = O.canonical_transform(pooled.cpu().numpy(), boxes)
    np.testing.assert_allclose(pc.cpu().numpy(), want, rtol=1e-5, atol=2e-5)
    em = empty.bool()
    assert int(em.sum()) > 0 and torch.count_nonzero(pc[em][..., 3:]) == 0 and torch.count_nonzero(pc[em][..., 0:3]) > 0


# ------------------------------------------------------------------------------------------------ iou3d
def test_overlap_and_iou_matrices(cuda):
    a = synth.sorted_bev(300, 5)
    b = synth.sorted_bev(217, 6)
    b[:100] = a[50:150] + np.float32(0.01)      # heavy overlaps
    b[100] = a[0]                               # identical boxes
    ta, tb = T(a, cuda), T(b, cuda)
    ov = torch.zeros((300, 217), device=cuda)
    iou = torch.zeros((300, 217), device=cuda)
    iou3d_cuda.boxes_overlap_bev_gpu(ta, tb, ov)
    iou3d_cuda.boxes_iou_bev_gpu(ta, tb, iou)
    want_ov, want_iou = O.boxes_overlap_bev(a, b), O.boxes_iou_bev(a, b)
    # north_star: IoU within 1e-5 rel of the reference; the CPU oracle differs by libm ulps in sin/cos/atan2
    np.testing.assert_allclose(ov.cpu().numpy(), want_ov, rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(iou.cpu().numpy(), want_iou, rtol=2e-4, atol=2e-5)
    assert (want_iou > 0.5).sum() > 50
    REF.equal("overlap", ov, lambda: R.boxes_overlap_bev(ta, tb), "overlap matrix not bit-identical to the reference kernel")
    REF.equal("iou", iou, lambda: R.boxes_iou_bev(ta, tb), "IoU matrix not bit-identical to the reference kernel")


@pytest.mark.parametrize("n,thresh,normal", [(100, 0.1, False), (1000, 0.3, False), (2700, 0.8, True), (6300, 0.8, True),
                                             (6300, 0.85, True), (65, 0.5, False), (64, 0.5, True), (1, 0.5, False),
                                             (15000, 0.7, True)])
def test_nms_keep_exact(cuda, n, thresh, normal):
    boxes = synth.sorted_bev(n, 100 + n)
    tb = T(boxes, cuda)
    keep = torch.zeros(n, dtype=torch.int64)
    num = (iou3d_cuda.nms_normal_gpu if normal else iou3d_cuda.nms_gpu)(tb, keep, thresh)
    got = keep[:num].numpy()
    REF.equal("keep", got, lambda: R.nms(tb, thresh, normal), "keep list differs from the reference nms")
    from pointrcnn_b200 import _cabi as C
    mask = torch.zeros((n, (n + 63) // 64), dtype=torch.int64, device=cuda)
    C.check(C.lib().prb_nms_mask(C.ptr(tb), n, C.c_float(thresh), int(normal), C.ptr(mask), C.stream()), "nms_mask")
    mm = mask.cpu().numpy().view(np.uint64)
    rows = np.arange(n)[:, None] // 64
    cols = np.arange(mm.shape[1])[None, :]
    upper = cols >= rows
    REF.equal("mask", mm[upper], lambda: R.nms_mask(tb, thresh, normal).cpu().numpy().view(np.uint64)[upper],
              "upper-triangle mask differs from the reference kernel")
    assert not mm[~upper].any()
    if normal:  # no transcendental in the axis-aligned IoU -> the CPU oracle is bit-exact too
        assert np.array_equal(got, O.nms(boxes, thresh, normal=True))
    else:
        want = O.nms(boxes, thresh, normal=False)
        agree = len(set(got.tolist()) & set(want.tolist())) / max(1, len(want))
        assert agree > 0.98


def test_iou3d_utils_api(cuda):
    b3, scores = synth.boxes3d(500, 9)
    tb, ts = T(b3, cuda), T(scores, cuda)
    iou = iou3d_utils.boxes_iou3d_gpu(tb[:200], tb[200:])
    np.testing.assert_allclose(iou.cpu().numpy(), O.boxes_iou3d(b3[:200], b3[200:]), rtol=3e-4, atol=3e-5)
    bev = T(synth.to_bev(b3), cuda)
    keep = iou3d_utils.nms_normal_gpu(bev, ts, 0.7)
    order = np.argsort(-scores, kind="stable")
    want = order[O.nms(synth.to_bev(b3)[order], 0.7, normal=True)]
    assert keep.dtype == torch.int64 and keep.is_cuda
    assert np.array_equal(keep.cpu().numpy(), want)
    keep_r = iou3d_utils.nms_gpu(bev, ts, 0.1)
    assert 0 < keep_r.numel() < 500
    bi = iou3d_utils.boxes_iou_bev(bev[:10], bev[:10])
    assert torch.allclose(torch.diagonal(bi), torch.ones(10, device=cuda), atol=1e-4)


# ------------------------------------------------------------------------------------------------ hash-grid paths
@pytest.mark.parametrize("kind,N,M,radii,nss", [
    ("kitti", 8192, 2048, (0.5, 1.0), (16, 32)),     # sparse: everything answered by the grid
    ("cube", 4096, 512, (0.1, 0.3), (16, 32)),       # dense: >128 candidates per ball -> overflow list -> scan kernel
    ("dup", 2048, 512, (0.3, 0.6), (8, 64)),         # exact duplicates share cells
    ("cube", 300, 40, (0.2,), (16,)),                # tiny set through the grid, single radius
    ("kitti", 5000, 777, (2.0, 4.0), (16, 32)),      # n not a power of two, big balls
])
@pytest.mark.parametrize("csr", [0, 1])                # linked lists (default) / CSR runs
def test_ball_query_grid_path_exact(cuda, kind, N, M, radii, nss, csr):
    from pointrcnn_b200 import _cabi
    xyz = _cloud(kind, 2, N, 51 + N)
    fidx = O.fps(xyz, M)
    new_xyz = np.stack([xyz[b][fidx[b]] for b in range(2)])
    x, c = T(xyz, cuda), T(new_xyz, cuda)
    old = pu.GRID_MIN_POINTS_BQ
    pu.GRID_MIN_POINTS_BQ = 1
    try:
        with _cabi.options(grid_csr=csr):
            if len(radii) == 2:
                got = pu.ball_query_msg2(radii, nss, x, c)
            else:
                got = [pu.ball_query(radii[0], nss[0], x, c)]
    finally:
        pu.GRID_MIN_POINTS_BQ = old
    for g, r, ns in zip(got, radii, nss):
        assert np.array_equal(g.cpu().numpy(), O.ball_query(r, ns, xyz, new_xyz)), "grid ball query differs (r=%g)" % r


@pytest.mark.parametrize("cell", [None, 0.5, 4.0])     # default edge; tiny cells (most queries go to the exhaustive scan); big cells
@pytest.mark.parametrize("kind,n,m", [("kitti", 8192, 2048), ("cube", 2000, 500), ("dup", 1024, 256), ("cube", 100, 5),
                                      ("kitti", 300, 3), ("dup", 4096, 64)])
@pytest.mark.parametrize("mode", ["sorted_queries", "plain", "cursor_loop", "csr"])     # queries grouped by cell; default; convergent cursor loop; CSR
def test_three_nn_grid_path_exact(cuda, kind, n, m, cell, mode):
    grid_opts = {"sorted_queries": {"nn_sort_queries": 1}, "plain": {}, "cursor_loop": {"nn_walk": 1}, "csr": {"grid_csr": 1}}[mode]
    unknown = _cloud(kind, 2, n, 61 + n)
    known = np.ascontiguousarray(unknown[:, ::max(1, n // m)][:, :m])
    if kind == "kitti":
        unknown[0, :10] += 300.0         # far-away queries: third neighbour beyond one cell -> brute-force list
    d2, idx = O.three_nn(unknown, known)
    from pointrcnn_b200 import _cabi
    old = pu.GRID_MIN_POINTS_NN
    pu.GRID_MIN_POINTS_NN = 1
    try:
        with _cabi.options(**grid_opts, **({} if cell is None else {"nn_cell": cell})):
            got_d2, got_idx, w = pu.three_nn_weights(T(unknown, cuda), T(known, cuda))
    finally:
        pu.GRID_MIN_POINTS_NN = old
    assert np.array_equal(got_idx.cpu().numpy(), idx)
    assert np.array_equal(got_d2.cpu().numpy(), d2)
    np.testing.assert_allclose(w.cpu().numpy(), O.interp_weights(d2), rtol=2e-6, atol=1e-7)


# ------------------------------------------------------------------------------------------------ fused 3D IoU (8(f) rank 2)
def _ref_iou3d(a, b):
    """iou3d_utils.boxes_iou3d_gpu (reference :21-53) op for op, with the reference's OWN overlap kernel (oracle/_ref)"""
    from pointrcnn_b200 import kitti_utils
    ov_bev = R.boxes_overlap_bev(kitti_utils.boxes3d_to_bev_torch(a).contiguous(), kitti_utils.boxes3d_to_bev_torch(b).contiguous())
    a_min, a_max = (a[:, 1] - a[:, 3]).view(-1, 1), a[:, 1].view(-1, 1)
    b_min, b_max = (b[:, 1] - b[:, 3]).view(1, -1), b[:, 1].view(1, -1)
    ov_h = torch.clamp(torch.min(a_max, b_max) - torch.max(a_min, b_min), min=0)
    ov3d = ov_bev * ov_h
    va, vb = (a[:, 3] * a[:, 4] * a[:, 5]).view(-1, 1), (b[:, 3] * b[:, 4] * b[:, 5]).view(1, -1)
    return ov3d / torch.clamp(va + vb - ov3d, min=1e-7)


@pytest.mark.parametrize("M,N", [(512, 20), (64, 64), (1, 1), (100, 7)])
def test_fused_iou3d_matches_the_reference_sequence(cuda, M, N):
    b3, _ = synth.boxes3d(M + N, 91 + M)
    rng = np.random.default_rng(M)
    b3[:, 1] += rng.normal(0, 0.3, M + N).astype(np.float32)           # height offsets: partial vertical overlap
    a, b = T(b3[:M].copy(), cuda), T(b3[M:].copy(), cuda)
    got = iou3d_cuda.boxes_iou3d(a, b)
    mirror = iou3d_utils.boxes_iou3d_gpu(a, b)                          # the op-by-op mirror on this repo's overlap kernel
    assert torch.equal(got, mirror), "fused IoU differs from the op-by-op sequence"
    REF.equal("iou3d", got, lambda: _ref_iou3d(a, b), "fused IoU differs from the reference sequence on the reference kernel")
    want = O.boxes_iou3d(b3[:M], b3[M:])
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=2e-4, atol=2e-6)      # CPU libm vs device sin/cos/atan2
    # batched form = per-scene calls; aligned form = the diagonal of the matrix
    a2 = torch.stack([a, a.flip(0)]); b2 = torch.stack([b, b.flip(0)])
    gb = iou3d_cuda.boxes_iou3d(a2.contiguous(), b2.contiguous())
    assert torch.equal(gb[0], got) and torch.equal(gb[1], iou3d_cuda.boxes_iou3d(a2[1].contiguous(), b2[1].contiguous()))
    K = min(M, N)
    al = iou3d_cuda.boxes_iou3d_aligned(a[:K].contiguous(), b[:K].contiguous())
    assert torch.equal(al, got[:K, :K].diagonal())
