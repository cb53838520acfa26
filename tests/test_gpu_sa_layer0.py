"""SA chains whose layer 0 the gather warps evaluate (prb_sa_group_mlp_max_l0, direct form for c_feat <= 5) against the
tensor-core form of the same chain (prb_sa_group_mlp_max_ws) on the same inputs, and the host-side weight split.

Both forms see the same operands (dxyz and features rounded to tf32, weights rounded at pack time with the BN scale folded
in); only the fp32 summation order of layer 0 differs.  A layer-0 activation on a tf32 rounding boundary may round the other
way and move the next layer a little, so the bound is the chain bound of test_gpu_mlp.py: 97 % of the outputs within
2e-4 (1 + |y|) and all of them within 5e-3 (1 + |y|).
"""
import ctypes

import numpy as np
import pytest
import torch

import synth
from pointrcnn_b200 import _cabi as C
from pointrcnn_b200.pointnet2 import pointnet2_modules as pm
from pointrcnn_b200.pointnet2 import pointnet2_utils as pu


def _randomise_bn(module, seed):
    g = torch.Generator().manual_seed(seed)
    for m in module.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)


def test_split_layer0_matches_numpy():
    """weights (c0, 8) = BN-folded W0 in the module's column order [xyz, feats], zero beyond 3 + c_feat; shift0 = BN shift;
    the chain left for the tensor core is layers 1 .. L-1 as plain rows with c_in = c0"""
    torch.manual_seed(4)
    for c_feat, widths in ((0, [16, 16, 32]), (1, [32, 32, 64]), (3, [24, 40]), (5, [64, 96, 128])):
        mod = pm.PointnetSAModuleMSG(npoint=8, radii=[0.2], nsamples=[16], mlps=[[c_feat] + widths], bn=True).eval()
        _randomise_bn(mod, 3 + c_feat)
        layers = list(mod.mlps[0].children())
        conv, bn = layers[0].conv, layers[0].bn.bn
        W = conv.weight.detach().numpy().reshape(widths[0], 3 + c_feat)
        inv = bn.weight.detach().numpy() / np.sqrt(bn.running_var.numpy() + np.float32(bn.eps))
        shift = bn.bias.detach().numpy() - bn.running_mean.numpy() * inv
        want_w = np.zeros((widths[0], 8), np.float32)
        want_w[:, :3 + c_feat] = W * inv[:, None]

        fused = pm._FusedMLP()
        desc = fused.get(mod.mlps[0], 0, c_feat, torch.device("cpu"), layer0=True)
        np.testing.assert_allclose(fused.l0["w"].numpy(), want_w, rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(fused.l0["shift"].numpy(), shift, rtol=1e-6, atol=1e-6)
        assert fused.l0["c0"] == widths[0] and fused.c_out == widths
        assert desc.num_layers == len(widths) - 1 and desc.c_in == widths[0] and not desc.scale
        assert list(desc.c_out)[:desc.num_layers] == widths[1:]
        # the packed chain is exactly what packing layers 1 .. L-1 on their own as plain rows gives
        ref = pm._FusedMLP()
        tail = torch.nn.Sequential(*layers[1:])
        ref_desc = ref.get(tail, 2, 0, torch.device("cpu"))
        assert torch.equal(fused.tensors[0], ref.tensors[0]) and torch.equal(fused.tensors[2], ref.tensors[2])
        assert ref_desc.c_in == desc.c_in


def _check(out, ref):
    err = np.abs(out - ref)
    bound = 1 + np.abs(ref)
    assert (err <= 5e-3 * bound).all(), err.max()
    assert (err <= 2e-4 * bound).mean() >= 0.97, (err <= 2e-4 * bound).mean()


CASES = [
    # B, N, npoint, nsample, c_feat, widths
    (2, 4096, 512, 16, 1, [16, 16, 32]),       # RPN SA1 scale 0
    (2, 4096, 512, 32, 1, [32, 32, 64]),       # RPN SA1 scale 1
    (2, 4096, 300, 64, 1, [32, 32, 64]),       # 64 samples: a centre spans two warps
    (3, 2500, 37, 16, 3, [24, 40, 48]),        # 1776 rows: a partial last tile; c_feat not a multiple of 4
    (2, 2000, 150, 32, 5, [64, 96, 128]),      # five feature channels: all eight inputs; two K chunks of layer 1
    (2, 2000, 100, 8, 0, [16, 200]),           # no features; one layer left for the tensor core, nsample 8
    (2, 1024, 128, 32, 2, [128, 128, 256]),    # RCNN SA widths
]


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,npoint,ns,c_feat,widths", CASES)
def test_layer0_entry_matches_tensor_core_form(cuda, B, N, npoint, ns, c_feat, widths):
    torch.manual_seed(ns + c_feat)
    mod = pm.PointnetSAModuleMSG(npoint=npoint, radii=[0.3], nsamples=[ns], mlps=[[c_feat] + widths], bn=True).to(cuda).eval()
    _randomise_bn(mod, 2 + ns)
    x = torch.from_numpy(synth.u_cube(B, N, 17 + N)).to(cuda)
    feats_pm = torch.randn(B, N, c_feat, device=cuda) if c_feat else None
    with torch.no_grad():
        _, centres = pu.furthest_point_sample_xyz(x, npoint)
        centres = centres.contiguous()
        idx = pu.ball_query(0.3, ns, x, centres)
    mlp = mod.mlps[0]
    lib = C.lib()
    outs = []
    for layer0 in (False, True):
        fused = pm._FusedMLP()
        desc = fused.get(mlp, 0, c_feat, cuda, layer0=layer0)
        c_last = widths[-1]
        out = torch.full((B, c_last + 5, npoint), float("nan"), device=cuda)
        out_pm = torch.full((B, npoint, c_last + 5), float("nan"), device=cuda)
        if layer0:
            l0 = fused.l0
            C.check(lib.prb_sa_group_mlp_max_l0(B, N, npoint, ns, c_feat, C.ptr(x), C.ptr(centres), C.ptr(feats_pm), C.ptr(idx),
                                                l0["c0"], C.ptr(l0["w"]), C.ptr(l0["shift"]), ctypes.byref(desc), C.ptr(out),
                                                C.ptr(out_pm), c_last + 5, 5, C.stream()), "sa_group_mlp_max_l0")
        else:
            co = (ctypes.c_int * 3)(*(widths + [0] * (3 - len(widths))))
            wsb = lib.prb_sa_workspace_bytes(B, npoint, ns, c_feat, len(widths), co)
            ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=cuda)
            C.check(lib.prb_sa_group_mlp_max_ws(B, N, npoint, ns, c_feat, C.ptr(x), C.ptr(centres), C.ptr(feats_pm), C.ptr(idx),
                                                ctypes.byref(desc), C.ptr(out), C.ptr(out_pm), c_last + 5, 5, C.ptr(ws),
                                                C.c_size_t(wsb), C.stream()), "sa_group_mlp_max_ws")
        torch.cuda.synchronize()
        assert torch.isnan(out[:, :5]).all() and torch.isnan(out_pm[:, :, :5]).all(), "channels before the offset written"
        assert torch.equal(out_pm[:, :, 5:], out[:, 5:].transpose(1, 2))
        outs.append(out[:, 5:].cpu().numpy())
    assert np.isfinite(outs[1]).all()
    _check(outs[1], outs[0])


@pytest.mark.gpu
@pytest.mark.parametrize("ns,widths", [(16, [16, 16, 32]), (32, [32, 32, 64])])
def test_layer0_builds_bit_identical(cuda, ns, widths):
    """every build of the chain kernel (CTAs per SM x row warps) computes the same bits with layer 0 in the gather warps"""
    torch.manual_seed(ns)
    mod = pm.PointnetSAModuleMSG(npoint=700, radii=[0.3], nsamples=[ns], mlps=[[1] + widths], bn=True).to(cuda).eval()
    _randomise_bn(mod, 9)
    x = torch.from_numpy(synth.u_cube(3, 4000, 13)).to(cuda)
    f = torch.randn(3, 1, 4000, device=cuda)
    outs = []
    for opt in ({"mlp_tune": 0}, {"mlp_occ": 3}, {"mlp_occ": 1}, {"mlp_occ": 1, "mlp_ne": 2, "mlp_ngw": 3}):
        with torch.no_grad(), C.options(**opt):
            outs.append(mod(x, f)[1].clone())
    assert mod._fused[0].l0 is not None, "the module did not take the layer-0 path"
    for k in range(1, len(outs)):
        assert torch.equal(outs[0], outs[k]), "build %d differs" % k
