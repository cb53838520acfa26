"""Mirror of pointnet2_lib/pointnet2/pointnet2_modules.py (reference :10-160): PointnetSAModuleMSG,
PointnetSAModule, PointnetFPModule -- same constructor arguments, sub-module names (`groupers`, `mlps`,
`mlp`) and forward signatures, so checkpoints and lib/net/*.py work unchanged.

Two execution paths per module, chosen per call:
  fused    (no autograd graph needed, BatchNorm in eval mode or absent, max-pool, power-of-two nsample):
           FPS(+new_xyz) -> [one ball-query scan for both radii] -> per scale ONE tensor-core kernel that
           gathers the neighbourhood, runs the whole SharedMLP and max-pools (csrc/mlp_tc.cu).  FP modules:
           three_nn(+weights) -> ONE kernel that interpolates, concatenates the skip features and runs the MLP.
  unfused  (training / anything else): the reference's op-by-op sequence on the B200 natives with
           torch.nn convolutions, full autograd support.
`config.override(disable_fused=True)` forces the unfused path (used by tests to cross-check the two).
"""
import ctypes
from typing import List

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _cabi as C
from .. import config
from .. import prof
from . import pointnet2_utils
from . import pytorch_utils as pt_utils


def _round_up(a, b):
    return (a + b - 1) // b * b


class _FusedMLP:
    """Device-side image of one SharedMLP for the tensor-core chain: packed weights + folded BN scale/shift.
    Rebuilt whenever a parameter / buffer version changes (optimizer step, load_state_dict, .to())."""

    def __init__(self):
        self.key = None
        self.desc = None
        self.tensors = None
        self.c_out = None
        self.proj = None
        self.l0 = None

    @staticmethod
    def supported(mlp: nn.Sequential):
        layers = list(mlp.children())
        if not 1 <= len(layers) <= 3:
            return False
        for layer in layers:
            names = [k for k, _ in layer.named_children()]
            if names not in (["conv", "bn", "activation"], ["conv", "activation"]):
                return False
            if not isinstance(layer.activation, nn.ReLU):
                return False
            conv = layer.conv
            if tuple(conv.kernel_size) not in ((1, 1), (1,)) or conv.out_channels > 512:
                return False
            if "bn" in names and layer.bn.bn.training:
                return False
        return True

    def get(self, mlp: nn.Sequential, kind: int, split: int, device, project_known: bool = False, layer0: bool = False):
        """layer0 (SA chains, kind 0, split = c_feat <= 5): layer 0 is taken out of the tensor-core chain -- the gather warps
        evaluate relu(W0 . [dxyz, f] + shift0) themselves (`self.l0`: weights (c0, 8) with the BN scale folded, shift0 (c0,))
        and the returned desc is the chain of layers 1 .. L-1 packed as plain rows (kind 2, c_in = c0).
        project_known (FP chains, kind 1): layer 0 is split by linearity -- interp(known) @ W0k^T == interp(known @ W0k^T) --
        into a per-KNOWN-point projection (a separate, 4x smaller row GEMM: `self.proj`, linear, no shift) and a main chain
        whose layer 0 reads [interp(projected rows) | skip] through the weight [I | W0s]: the gather moves c_out0 instead of
        c_known floats per neighbour and layer 0 contracts over c_out0 + c_skip instead of c_known + c_skip columns."""
        layers = list(mlp.children())
        tensors = []
        for layer in layers:
            tensors += [layer.conv.weight, layer.conv.bias]
            if hasattr(layer, "bn"):
                bn = layer.bn.bn
                tensors += [bn.weight, bn.bias, bn.running_mean, bn.running_var]
        key = (kind, split, str(device), _fold_scale(), project_known, layer0) + tuple((id(t), t._version) if t is not None else None for t in tensors)
        if key == self.key:
            return self.desc
        L = len(layers)
        c_in = layers[0].conv.in_channels
        c_out = [layer.conv.out_channels for layer in layers]
        ws, scales, shifts = [], [], []
        with torch.no_grad():
            for layer in layers:
                conv = layer.conv
                W = conv.weight.detach().reshape(conv.out_channels, -1).float().cpu().contiguous()
                co = conv.out_channels
                if hasattr(layer, "bn"):
                    bn = layer.bn.bn
                    inv = (bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)).cpu()
                    sh = (bn.bias.detach().float().cpu() - bn.running_mean.detach().float().cpu() * inv)
                    if conv.bias is not None:
                        sh = sh + inv * conv.bias.detach().float().cpu()
                else:
                    inv = torch.ones(co)
                    sh = conv.bias.detach().float().cpu() if conv.bias is not None else torch.zeros(co)
                pad = _round_up(co, 32) - co
                if _fold_scale():
                    W = (W * inv[:, None]).contiguous()     # BN scale folded into the weights before TF32 rounding
                ws.append(W)
                scales.append(F.pad(inv, (0, pad)))
                shifts.append(F.pad(sh, (0, pad)))
        lib = C.lib()
        self.proj = None
        self.l0 = None
        if layer0:
            assert _fold_scale() and L >= 2 and kind == 0 and c_in == 3 + split <= L0_IN
            w0, sh0 = split_layer0(ws[0], shifts[0][:c_out[0]])
            self.l0 = dict(w=w0.to(device), shift=sh0.to(device), c0=c_out[0])
            ws, scales, shifts = ws[1:], scales[1:], shifts[1:]
            kind, split, c_in, L = 2, 0, c_out[0], L - 1
            c_out_chain = c_out[1:]
        else:
            c_out_chain = c_out
        if project_known:
            # ws[0] is (c_out0, c_known + c_skip) with the BN scale already folded in: W0k -> projection, W0s stays
            W0 = ws[0]
            c1, c_known = W0.shape[0], split
            self.proj = self._pack(lib, 2, 0, c_known, [c1], [W0[:, :c_known].contiguous()], torch.zeros(_round_up(c1, 32)), device, flags=1)
            ws[0] = torch.cat([torch.eye(c1), W0[:, c_known:]], dim=1).contiguous()
            c_in, split = c1 + (c_in - c_known), c1
        co_arr = (ctypes.c_int * 3)(*(c_out_chain + [0] * (3 - L)))
        nbytes = lib.prb_mlp_packed_bytes_ex(kind, split, L, c_in, co_arr)
        host = np.zeros(nbytes // 4, dtype=np.float32)
        wp = (ctypes.c_void_p * L)(*[w.data_ptr() for w in ws])
        C.check(lib.prb_mlp_pack_weights_ex(kind, split, L, c_in, co_arr, wp, host.ctypes.data_as(ctypes.c_void_p)), "mlp_pack")
        packed = torch.from_numpy(host).to(device)
        scale = torch.cat(scales).contiguous().to(device)
        shift = torch.cat(shifts).contiguous().to(device)
        desc = C.MlpDesc()
        desc.num_layers, desc.c_in = L, c_in
        for i in range(3):
            desc.c_out[i] = c_out_chain[i] if i < L else 0
        desc.packed_w, desc.scale, desc.shift = packed.data_ptr(), (None if _fold_scale() else scale.data_ptr()), shift.data_ptr()
        self.key, self.desc, self.tensors, self.c_out = key, desc, (packed, scale, shift), c_out
        return desc

    @staticmethod
    def _pack(lib, kind, split, c_in, c_out, ws, shift, device, flags=0):
        """pack a chain whose scale is already folded into `ws`; returns dict(desc, keep-alive tensors, c_out)"""
        L = len(ws)
        co_arr = (ctypes.c_int * 3)(*(c_out + [0] * (3 - L)))
        nbytes = lib.prb_mlp_packed_bytes_ex(kind, split, L, c_in, co_arr)
        host = np.zeros(nbytes // 4, dtype=np.float32)
        wp = (ctypes.c_void_p * L)(*[w.data_ptr() for w in ws])
        C.check(lib.prb_mlp_pack_weights_ex(kind, split, L, c_in, co_arr, wp, host.ctypes.data_as(ctypes.c_void_p)), "mlp_pack")
        packed = torch.from_numpy(host).to(device)
        shift = shift.contiguous().to(device)
        desc = C.MlpDesc()
        desc.num_layers, desc.c_in = L, c_in
        for i in range(3):
            desc.c_out[i] = c_out[i] if i < L else 0
        desc.packed_w, desc.scale, desc.shift, desc.flags = packed.data_ptr(), None, shift.data_ptr(), flags
        return dict(desc=desc, keep=(packed, shift, ws), c_out=c_out, co_arr=co_arr)


L0_IN = 8   # layer-0 inputs of the direct form: [dx, dy, dz, up to 5 feature channels] (csrc/mlp_dev.cuh)


def split_layer0(w0: torch.Tensor, shift0: torch.Tensor):
    """layer 0 of an SA chain with c_feat <= 5 for the gather warps: w0 (c0, 3 + c_feat) in the module's column order
    [xyz, feats], BN scale already folded -> ((c0, L0_IN) zero-padded weights, (c0,) shift), float32, contiguous"""
    c0, c_in = w0.shape
    assert c_in <= L0_IN and shift0.shape == (c0,)
    w = torch.zeros((c0, L0_IN), dtype=torch.float32)
    w[:, :c_in] = w0.float()
    return w.contiguous(), shift0.float().contiguous()


def _layer0_direct(mlp: nn.Sequential, c_feat: int) -> bool:
    """SA chain whose layer 0 the gather warps evaluate (prb_sa_group_mlp_max_l0): at most 5 feature channels (a layer 0 of
    <= 8 FMAs per output, every operand already in the gathering lane), BN scale folded, at least one layer left for the
    tensor core, and layers 1 .. L-1 fit one launch (the entry does not split chains)"""
    if c_feat > L0_IN - 3 or not _fold_scale():
        return False
    c_out = [layer.conv.out_channels for layer in mlp.children()]
    if len(c_out) < 2:
        return False
    np_ = [_round_up(c, 32) for c in c_out[1:]]
    last = np_[-1]
    if last > 512 or sum(np_[:-1]) + (2 * min(last, 64) if len(np_) > 1 else 0) > 512:
        return False
    o = C.Options()
    C.lib().prb_get_thread_options(ctypes.byref(o))
    return o.mlp_pipeline != 0 and o.mlp_gather == 0      # the layer-0 gather exists in the pipelined kernel only


def _attach_pm(t, pm):
    """remember the point-major twin the kernel wrote next to `t`; valid while `t` is not modified in place"""
    t._prb_pm = (pm, t._version)
    return t


def _point_major(t):
    """(B,C,N) -> (B,N,C): the twin written by the producing kernel if it is still valid, else a transpose kernel"""
    twin = getattr(t, "_prb_pm", None)
    if twin is not None and twin[1] == t._version and twin[0].shape == (t.size(0), t.size(2), t.size(1)) and twin[0].device == t.device:
        return twin[0]
    return pointnet2_utils.transpose_bcn_to_bnc(t.contiguous())


def rows_mlp(fused: "_FusedMLP", mlp: nn.Sequential, a: torch.Tensor, b: torch.Tensor = None, tag="rows_mlp"):
    """SharedMLP over point rows on the tensor-core chain: `a` (rows, c_a) and optionally `b` (rows, c_b) are 2-D views with
    unit column stride and any row pitch (e.g. column slices of the pooled RoI rows); layer 0 reads [a | b] without the
    concatenation ever existing in memory.  Returns (rows, c_out) row-major.  Replaces pt_utils.SharedMLP on (B,C,N,1)
    tensors (lib/net/rcnn_net.py:58-66,171-175)."""
    lib = C.lib()
    dev = a.device
    rows, c_a = a.shape
    c_b = 0 if b is None else b.size(1)
    assert a.stride(1) == 1 and (b is None or (b.stride(1) == 1 and b.size(0) == rows))
    desc = fused.get(mlp, 1 if c_b else 2, c_a if c_b else 0, dev)
    c_out = fused.c_out
    pitch = _round_up(c_out[-1], 32)
    out = torch.empty((rows, pitch), dtype=torch.float32, device=dev)
    co_arr = (ctypes.c_int * 3)(*(c_out + [0] * (3 - len(c_out))))
    with torch.cuda.device(dev):
        wsb = lib.prb_rows2_workspace_bytes(C.c_long(rows), c_a, c_b, desc.num_layers, co_arr)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        with prof.region(tag, "%d [%d+%d]+%s" % (rows, c_a, c_b, c_out)):
            C.check(lib.prb_mlp_rows2(C.c_long(rows), c_a, C.ptr(a), a.stride(0), c_b, C.ptr(b) if c_b else None,
                                      b.stride(0) if c_b else 0, ctypes.byref(desc), C.ptr(out), pitch, C.ptr(ws), C.c_size_t(wsb),
                                      C.stream()), "mlp_rows2")
    return out if pitch == c_out[-1] else out[:, :c_out[-1]]


def _fold_scale():
    """config.fold_scale=False keeps the BN scale as a separate epilogue multiply (y = relu(s * (W x) + t))"""
    return config.get("fold_scale")


def _fused_enabled():
    return not config.get("disable_fused")


def _needs_graph(module, *tensors):
    if not torch.is_grad_enabled():
        return False
    if any(t is not None and t.requires_grad for t in tensors):
        return True
    return any(p.requires_grad for p in module.parameters())


class _PointnetSAModuleBase(nn.Module):
    def __init__(self):
        super().__init__()
        self.npoint = None
        self.groupers = None
        self.mlps = None
        self.pool_method = 'max_pool'
        self._fused = None

    def _apply(self, fn, *args, **kwargs):
        # .to() / .half() / .float() / .cuda() replace parameter storage without bumping tensor versions: drop the packed images
        self._fused = None
        return super()._apply(fn, *args, **kwargs)

    def invalidate_fused(self):
        """call after editing weights through `.data` (EMA, weight averaging): such writes do not bump the version counters the
        packed-weight cache keys on"""
        self._fused = None

    # ------------------------------------------------------------------ fused (tensor-core) path
    def _can_fuse(self, xyz, features, new_xyz):
        if not _fused_enabled() or not xyz.is_cuda or self.pool_method != 'max_pool':
            return False
        if _needs_graph(self, xyz, features, new_xyz):
            return False
        if xyz.dtype != torch.float32 or (features is not None and features.dtype != torch.float32):
            return False
        for g, mlp in zip(self.groupers, self.mlps):
            if not _FusedMLP.supported(mlp):
                return False
            if isinstance(g, pointnet2_utils.QueryAndGroup):
                ns = g.nsample
                if not g.use_xyz or ns < 4 or ns > 128 or (ns & (ns - 1)):
                    return False
            elif isinstance(g, pointnet2_utils.GroupAll):
                n = xyz.size(1)
                if not g.use_xyz or n < 4 or n > 128 or (n & (n - 1)):
                    return False
            else:
                return False
        return True

    def fused_geometry(self, xyz, new_xyz=None):
        """sampling + neighbour search of the fused path (depends on coordinates only, so a caller may run it on a side
        stream, ahead of the feature MLPs): returns (ret_xyz, centres (B,npoint,3), [idx per scale], [nsample per scale])"""
        B, N, _ = xyz.shape
        dev = xyz.device
        if self.npoint is None:
            centres = torch.zeros((B, 1, 3), dtype=torch.float32, device=dev)   # GroupAll: no centre subtraction
            ar = torch.arange(N, dtype=torch.int32, device=dev).view(1, 1, N).expand(B, 1, N).contiguous()
            return None, centres, [ar for _ in self.groupers], [N for _ in self.groupers]
        if new_xyz is None:
            _, new_xyz = pointnet2_utils.furthest_point_sample_xyz(xyz, self.npoint)
        centres = new_xyz.contiguous()
        if len(self.groupers) == 2:
            g0, g1 = self.groupers
            idxs = list(pointnet2_utils.ball_query_msg2((g0.radius, g1.radius), (g0.nsample, g1.nsample), xyz, centres))
        else:
            idxs = [pointnet2_utils.ball_query(g.radius, g.nsample, xyz, centres) for g in self.groupers]
        return new_xyz, centres, idxs, [g.nsample for g in self.groupers]

    def fused_mlp(self, xyz, features, centres, idxs, nss):
        """gather + SharedMLP + max-pool of every scale (one tensor-core kernel per scale) -> (B, sum C_out, npoint)"""
        lib = C.lib()
        B, N, _ = xyz.shape
        dev = xyz.device
        npoint = centres.size(1)
        c_feat = 0 if features is None else features.size(1)
        feats_pm = _point_major(features) if features is not None else None
        if self._fused is None or len(self._fused) != len(self.mlps):
            self._fused = [_FusedMLP() for _ in self.mlps]
        direct = [_layer0_direct(mlp, c_feat) for mlp in self.mlps]
        descs = [f.get(mlp, 0, c_feat, dev, layer0=d) for f, mlp, d in zip(self._fused, self.mlps, direct)]
        c_total = sum(f.c_out[-1] for f in self._fused)
        out = torch.empty((B, c_total, npoint), dtype=torch.float32, device=dev)
        out_pm = torch.empty((B, npoint, c_total), dtype=torch.float32, device=dev)   # twin for the next gather
        off = 0
        with torch.cuda.device(dev):
            for desc, fused, idx, ns in zip(descs, self._fused, idxs, nss):
                if fused.l0 is not None:
                    l0 = fused.l0
                    with prof.region("sa_mlp", "%dx%d [%d]+%s l0" % (B * npoint, ns, 3 + c_feat, fused.c_out)):
                        C.check(lib.prb_sa_group_mlp_max_l0(B, N, npoint, ns, c_feat, C.ptr(xyz), C.ptr(centres), C.ptr(feats_pm),
                                                            C.ptr(idx), l0["c0"], C.ptr(l0["w"]), C.ptr(l0["shift"]), ctypes.byref(desc),
                                                            C.ptr(out), C.ptr(out_pm), out.size(1), off, C.stream()), "sa_group_mlp_max_l0")
                    off += fused.c_out[-1]
                    continue
                co_arr = (ctypes.c_int * 3)(*(fused.c_out + [0] * (3 - len(fused.c_out))))
                wsb = lib.prb_sa_workspace_bytes(B, npoint, ns, c_feat, desc.num_layers, co_arr)
                ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
                with prof.region("sa_mlp", "%dx%d [%d]+%s" % (B * npoint, ns, 3 + c_feat, fused.c_out)):
                    C.check(lib.prb_sa_group_mlp_max_ws(B, N, npoint, ns, c_feat, C.ptr(xyz), C.ptr(centres), C.ptr(feats_pm),
                                                        C.ptr(idx), ctypes.byref(desc), C.ptr(out), C.ptr(out_pm), out.size(1), off,
                                                        C.ptr(ws), C.c_size_t(wsb), C.stream()), "sa_group_mlp_max")
                off += fused.c_out[-1]
        return _attach_pm(out, out_pm)

    def _forward_fused(self, xyz, features, new_xyz):
        xyz = xyz.contiguous()
        ret_xyz, centres, idxs, nss = self.fused_geometry(xyz, new_xyz)
        return ret_xyz, self.fused_mlp(xyz, features, centres, idxs, nss)

    # ------------------------------------------------------------------ reference-shaped path
    def forward(self, xyz: torch.Tensor, features: torch.Tensor = None, new_xyz=None) -> (torch.Tensor, torch.Tensor):
        """
        :param xyz: (B, N, 3) coordinates
        :param features: (B, C, N) descriptors (channel-major) or None
        :param new_xyz: optional externally chosen centres (B, npoint, 3)
        :return: new_xyz (B, npoint, 3), new_features (B, sum_k mlps[k][-1], npoint)
        """
        if self._can_fuse(xyz, features, new_xyz):
            return self._forward_fused(xyz, features, new_xyz)

        new_features_list = []
        if new_xyz is None and self.npoint is not None:
            xyz_flipped = xyz.transpose(1, 2).contiguous()
            new_xyz = pointnet2_utils.gather_operation(
                xyz_flipped, pointnet2_utils.furthest_point_sample(xyz, self.npoint)).transpose(1, 2).contiguous()
        for i in range(len(self.groupers)):
            new_features = self.groupers[i](xyz, new_xyz, features)      # (B, C, npoint, nsample)
            new_features = self.mlps[i](new_features)                    # (B, mlp[-1], npoint, nsample)
            if self.pool_method == 'max_pool':
                new_features = F.max_pool2d(new_features, kernel_size=[1, new_features.size(3)])
            elif self.pool_method == 'avg_pool':
                new_features = F.avg_pool2d(new_features, kernel_size=[1, new_features.size(3)])
            else:
                raise NotImplementedError
            new_features_list.append(new_features.squeeze(-1))           # (B, mlp[-1], npoint)
        return new_xyz, torch.cat(new_features_list, dim=1)


class PointnetSAModuleMSG(_PointnetSAModuleBase):
    """Pointnet set abstraction layer with multiscale grouping"""

    def __init__(self, *, npoint: int, radii: List[float], nsamples: List[int], mlps: List[List[int]], bn: bool = True,
                 use_xyz: bool = True, pool_method='max_pool', instance_norm=False):
        super().__init__()
        assert len(radii) == len(nsamples) == len(mlps)
        self.npoint = npoint
        self.groupers = nn.ModuleList()
        self.mlps = nn.ModuleList()
        for i in range(len(radii)):
            self.groupers.append(pointnet2_utils.QueryAndGroup(radii[i], nsamples[i], use_xyz=use_xyz)
                                 if npoint is not None else pointnet2_utils.GroupAll(use_xyz))
            mlp_spec = mlps[i]
            if use_xyz:
                mlp_spec[0] += 3   # in place, like the reference (pointnet2_modules.py:88-89): callers rely on it
            self.mlps.append(pt_utils.SharedMLP(mlp_spec, bn=bn, instance_norm=instance_norm))
        self.pool_method = pool_method


class PointnetSAModule(PointnetSAModuleMSG):
    """Pointnet set abstraction layer"""

    def __init__(self, *, mlp: List[int], npoint: int = None, radius: float = None, nsample: int = None, bn: bool = True,
                 use_xyz: bool = True, pool_method='max_pool', instance_norm=False):
        super().__init__(mlps=[mlp], npoint=npoint, radii=[radius], nsamples=[nsample], bn=bn, use_xyz=use_xyz,
                         pool_method=pool_method, instance_norm=instance_norm)


class PointnetFPModule(nn.Module):
    r"""Propagates the features of one set to another"""

    def __init__(self, *, mlp: List[int], bn: bool = True):
        super().__init__()
        self.mlp = pt_utils.SharedMLP(mlp, bn=bn)
        self._fused = None
        self.emit_point_major = True   # also write a (B,n,C) twin for the next FP level (skips its transpose kernel)
        self.project_known = True      # split layer 0 by linearity when it narrows the gathered rows (see _FusedMLP.get)

    def _apply(self, fn, *args, **kwargs):
        self._fused = None             # see _PointnetSAModuleBase._apply
        return super()._apply(fn, *args, **kwargs)

    def invalidate_fused(self):
        self._fused = None

    def _can_fuse(self, unknown, known, unknow_feats, known_feats):
        if not _fused_enabled() or known is None or not unknown.is_cuda:
            return False
        if _needs_graph(self, unknown, known, unknow_feats, known_feats):
            return False
        if known_feats.dtype != torch.float32 or (unknow_feats is not None and unknow_feats.dtype != torch.float32):
            return False
        return _FusedMLP.supported(self.mlp)

    def fused_geometry(self, unknown, known):
        """3-NN search + inverse-distance weights (coordinates only) -> (idx (B,n,3) int32, weight (B,n,3))"""
        _, idx, weight = pointnet2_utils.three_nn_weights(unknown.contiguous(), known.contiguous())
        return idx, weight

    def fused_mlp(self, n, idx, weight, unknow_feats, known_feats):
        lib = C.lib()
        dev = known_feats.device
        B, c_known, m = known_feats.shape
        c_skip = 0 if unknow_feats is None else unknow_feats.size(1)
        known_pm = _point_major(known_feats)
        skip = unknow_feats.contiguous() if unknow_feats is not None else None
        if self._fused is None:
            self._fused = _FusedMLP()
        c1 = list(self.mlp.children())[0].conv.out_channels
        # interpolation commutes with the (linear) first layer: project the m known points once instead of gathering
        # c_known floats for each of the 3 neighbours of every one of the n >= m unknown points
        # measured (profiles/r2_notes.md): pays at the finest level (262144 rows: 0.267 -> 0.231 ms incl. the projection launch),
        # not at the coarse ones, where the extra launch costs more than the narrower gather saves
        project = (self.project_known and config.get("fp_project") and _fold_scale() and c1 < c_known and n >= m
                   and B * n >= config.get("fp_project_min_rows"))
        desc = self._fused.get(self.mlp, 1, c_known, dev, project_known=project)
        c_out = self._fused.c_out
        if project:
            pj = self._fused.proj
            pitch = _round_up(c1, 32)
            rows = B * m
            proj_rows = torch.empty((rows, pitch), dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                wsb = lib.prb_rows_workspace_bytes(C.c_long(rows), c_known, 1, pj["co_arr"])
                wsp = torch.empty(wsb, dtype=torch.uint8, device=dev)
                with prof.region("fp_mlp", "%d proj [%d]+[%d]" % (rows, c_known, c1)):
                    C.check(lib.prb_mlp_rows(C.c_long(rows), c_known, C.ptr(known_pm), ctypes.byref(pj["desc"]), C.ptr(proj_rows), pitch,
                                             C.ptr(wsp), C.c_size_t(wsb), C.stream()), "mlp_rows(fp projection)")
            known_pm = proj_rows if pitch == c1 else proj_rows[:, :c1].contiguous()
            c_known = c1
        out = torch.empty((B, c_out[-1], n), dtype=torch.float32, device=dev)
        out_pm = torch.empty((B, n, c_out[-1]), dtype=torch.float32, device=dev) if self.emit_point_major else None
        co_arr = (ctypes.c_int * 3)(*(c_out + [0] * (3 - len(c_out))))
        with torch.cuda.device(dev):
            wsb = lib.prb_fp_workspace_bytes(B, n, c_known, c_skip, desc.num_layers, co_arr)
            ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
            with prof.region("fp_mlp", "%d [%d+%d]+%s" % (B * n, c_known, c_skip, c_out)):
                C.check(lib.prb_fp_interp_mlp_ws(B, n, m, c_known, c_skip, C.ptr(known_pm), C.ptr(idx), C.ptr(weight), C.ptr(skip),
                                                 ctypes.byref(desc), C.ptr(out), C.ptr(out_pm), C.ptr(ws), C.c_size_t(wsb), C.stream()),
                        "fp_interp_mlp")
        return _attach_pm(out, out_pm) if out_pm is not None else out

    def _forward_fused(self, unknown, known, unknow_feats, known_feats):
        idx, weight = self.fused_geometry(unknown, known)
        return self.fused_mlp(unknown.size(1), idx, weight, unknow_feats, known_feats)

    def forward(self, unknown: torch.Tensor, known: torch.Tensor, unknow_feats: torch.Tensor,
                known_feats: torch.Tensor) -> torch.Tensor:
        """
        :param unknown: (B, n, 3) positions to propagate to
        :param known: (B, m, 3) positions to propagate from (None: broadcast known_feats)
        :param unknow_feats: (B, C1, n) skip features or None
        :param known_feats: (B, C2, m)
        :return: (B, mlp[-1], n)
        """
        if self._can_fuse(unknown, known, unknow_feats, known_feats):
            return self._forward_fused(unknown, known, unknow_feats, known_feats)

        if known is not None:
            dist, idx = pointnet2_utils.three_nn(unknown, known)
            dist_recip = 1.0 / (dist + 1e-8)
            norm = torch.sum(dist_recip, dim=2, keepdim=True)
            weight = dist_recip / norm
            interpolated_feats = pointnet2_utils.three_interpolate(known_feats, idx, weight)
        else:
            interpolated_feats = known_feats.expand(*known_feats.size()[0:2], unknown.size(1))
        if unknow_feats is not None:
            new_features = torch.cat([interpolated_feats, unknow_feats], dim=1)   # (B, C2 + C1, n)
        else:
            new_features = interpolated_feats
        new_features = self.mlp(new_features.unsqueeze(-1))
        return new_features.squeeze(-1)
