#!/usr/bin/env python
"""bench.py -- scenes/s of the RPN PointNet++ backbone forward (4 SA-MSG + 4 FP, tools/cfgs/default.yaml)
on synthetic 16384x4 clouds, batch 16 per GPU (BASELINE.json configs[1]).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the CPU restatement of the same path on the host cores

One JSON line on rank 0.  A "step" is one batch of 16 scenes per GPU.  Every timed region times EXACTLY K = --steps steps
between a barrier + synchronize on both sides (CUDA events, max over ranks), so the same arguments time the same steps on the
same inputs.  --dump-outputs DIR writes what the timed path (`value`) returned for its last step as DIR/<name>.npy.

  value         device-resident throughput: K steps through pointrcnn_b200.pipeline.BatchPipeline with `--inflight`
                independent batches in flight (one CUDA graph per slot); inputs rotate through a pool larger than L2.
  e2e           the whole RPN stage a caller runs (backbone -> fused cls/reg heads -> proposal layer, TEST quotas) from
                pinned HOST input: H2D of every step's points and D2H of every step's proposals (B,100,7)+(B,100)
                inside the timed region, handed to a host consumer per batch.
  e2e_features  backbone only, returning the full (B,128,16384) feature tensor to the host (PCIe bound; secondary).
  single_batch  one batch at a time on one stream with an L2 flush in between (per-batch latency view).
  roofline / kernels   per-kernel-family device times from CUDA events on the launching stream (sequential pass).
  ref_cuda      the reference's own CUDA kernels (oracle/_ref, rebuilt for sm_100a) + stock cuDNN MLP in the reference's
                call order, same process, same inputs: once single-stream, once with the same number of batches in
                flight; vs_ref_cuda = ours / theirs for both.
  strong_scaling  (N > 1) global batch 16: 16/N scenes per GPU per step, same pipeline.
  train_step    BASELINE configs[2]: RPN training step, 16 scenes per GPU, NCCL gradient all-reduce overlapped with backward.
  rcnn_stage    BASELINE configs[3]: roipool3d on 4 x 512 RoIs x 512 points + the RCNN PointNet++ stack (rank 0).
  eval_e2e      BASELINE configs[4]: raw scans -> input pipeline -> RPN -> RCNN -> rotated NMS -> KITTI result text, global
                batch 8 sharded over the ranks (8 / N scenes per GPU).
  cpu_baseline  oracle port on the host cores over a bounded sample of the same workload.
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

sys.dont_write_bytecode = True    # the tree may be read-only: nothing is written there
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

POINTS, CHANNELS, BATCH = 16384, 4, 16
CONFIG_SEED = 2000  # seed = 1000*config + scene index (SURVEY.md 8d)
METRIC = "scenes/sec RPN backbone fwd (16384 pts)"


def workload_config(world):
    """identical for the GPU arm and the reference (CPU) arm"""
    return {"workload": "RPN PointNet++ backbone fwd: 4 SA-MSG + 4 FP (tools/cfgs/default.yaml), 16384x4 uniform KITTI-scope "
                        "points, eval-mode BN (BASELINE configs[1])", "batch_per_gpu": BATCH, "global_batch": BATCH * world,
            "parallelism": "dp%d (scene sharding, no data-path collective)" % world}


def make_scenes(first, count):
    import synth
    return np.concatenate([synth.u_kitti(1, POINTS, CONFIG_SEED + first + i, channels=CHANNELS) for i in range(count)], 0)


def _randomise_bn(net):
    import torch
    g = torch.Generator().manual_seed(1)
    for m in net.modules():   # non-trivial eval-mode BN (SURVEY.md 8d)
        if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm1d)):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)


def build_model(device):
    import torch
    from pointrcnn_b200.backbone import Pointnet2MSG
    torch.manual_seed(0)
    net = Pointnet2MSG(input_channels=CHANNELS - 3).eval()
    _randomise_bn(net)
    return net.to(device)


def build_rpn_stage(device, backbone):
    """the RPN stage around the SAME backbone module (heads random-init, BN randomised)"""
    import torch
    from pointrcnn_b200.rpn.stage import RPNStage
    torch.manual_seed(2)
    stage = RPNStage(input_channels=CHANNELS - 3).eval()
    _randomise_bn(stage)
    stage.backbone_net = backbone
    stage.backbone_net.FP_modules[0].emit_point_major = True
    return stage.to(device)


def mlp_flops_per_scene(net):
    """2*MAC of every SA / FP SharedMLP per scene (algorithmic FLOPs of the tensor-core kernels)"""
    sa = fp = 0
    for mod in net.SA_modules:
        for grouper, mlp in zip(mod.groupers, mod.mlps):
            rows = mod.npoint * grouper.nsample
            sa += 2 * rows * sum(l.conv.in_channels * l.conv.out_channels for l in mlp.children())
    npts = [POINTS] + [m.npoint for m in net.SA_modules]
    for k, mod in enumerate(net.FP_modules):
        fp += 2 * npts[k] * sum(l.conv.in_channels * l.conv.out_channels for l in mod.mlp.children())
    return sa, fp


def folded_specs(net):
    from oracle import oracle as O

    def fold(mlp):
        out = []
        for layer in mlp.children():
            b = layer.bn.bn
            bn = dict(weight=b.weight.detach().cpu().numpy(), bias=b.bias.detach().cpu().numpy(),
                      running_mean=b.running_mean.cpu().numpy(), running_var=b.running_var.cpu().numpy(), eps=b.eps)
            out.append(O.fold_bn(layer.conv.weight.detach().cpu().numpy(), None, bn))
        return out
    sa = [dict(npoint=m.npoint, radii=[g.radius for g in m.groupers], nsamples=[g.nsample for g in m.groupers],
               mlps=[fold(x) for x in m.mlps]) for m in net.SA_modules]
    fp = [fold(m.mlp) for m in net.FP_modules]
    return sa, fp


def cpu_backbone(pc, sa, fp):
    """the CPU restatement of lib/net/pointnet2_msg.py:56-70 on top of the oracle ops"""
    from oracle import oracle as O
    xyz = np.ascontiguousarray(pc[..., :3])
    feats = np.ascontiguousarray(np.transpose(pc[..., 3:], (0, 2, 1))) if pc.shape[-1] > 3 else None
    l_xyz, l_f = [xyz], [feats]
    for s in sa:
        nx, nf, _ = O.sa_module_msg(l_xyz[-1], l_f[-1], s["npoint"], s["radii"], s["nsamples"], s["mlps"])
        l_xyz.append(nx)
        l_f.append(nf)
    for i in range(-1, -(len(fp) + 1), -1):
        l_f[i - 1] = O.fp_module(l_xyz[i - 1], l_xyz[i], l_f[i - 1], l_f[i], fp[i])
    return l_f[0]


def time_cpu(net_cpu_specs, scenes, steps=1, warmup=0):
    sa, fp = net_cpu_specs
    pc = make_scenes(0, scenes)
    for _ in range(warmup):
        cpu_backbone(pc, sa, fp)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_backbone(pc, sa, fp)
    dt = (time.perf_counter() - t0) / steps
    return scenes / dt, dt


class ClockSampler:
    """SM clock / throttle-reason samples every 100 ms while the timed regions run.  NVML is queried in-process
    (what nvidia-smi itself does) from a background thread: spawning nvidia-smi takes the driver lock for hundreds of
    milliseconds at start-up and occasionally stalled a timed region."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, index):
        import threading
        self.samples, self.stop_flag, self.h, self.nv = [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes CUDA_VISIBLE_DEVICES; map through it when it is set
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
        except Exception:
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, mx, rs))
            except Exception:
                pass
            time.sleep(0.1)

    def wait_started(self, timeout=5.0):
        t0 = time.time()
        while self.nv is not None and not self.samples and time.time() - t0 < timeout:
            time.sleep(0.02)

    def mark(self):
        """samples taken from here on belong to the timed regions"""
        self.first = len(self.samples)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "source": "nvml"}
        if self.nv is None:
            out["source"] = "unavailable"
            return out
        self.stop_flag = True
        self.t.join(timeout=2)
        rows = self.samples[getattr(self, "first", 0):] or self.samples
        if rows:
            out["sm_mhz"] = statistics.median(r[0] for r in rows)
            out["sm_max_mhz"] = max(r[1] for r in rows)
            out["samples"] = len(rows)
            seen = set()
            for r in rows:
                for name, bit in self.REASONS.items():
                    if r[2] & bit:
                        seen.add(name)
            out["reasons"] = sorted(seen)
        return out


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained"), src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


def ncu_traffic():
    """DRAM bytes per step of each kernel family, from the committed ncu --set full capture (profiles/r2_traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum summed over the family's launches of one step), or {}"""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        return json.load(open(path))
    except Exception:
        return {}


def run_reference_arm(args):
    """--impl reference: the reference has no CPU implementation of this path; the arm times the CPU restatement
    (oracle port) with all host threads on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import oracle as O
    net = build_model("cpu")
    specs = folded_specs(net)
    scenes = args.cpu_scenes
    steps, warm = max(1, args.steps), min(1, args.warmup)
    val, dt = time_cpu(specs, scenes, steps=steps, warmup=warm)
    cores = O.num_threads()
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "scenes/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "cpu_baseline": {"value": val, "unit": "scenes/s", "cores": cores, "kind": "port",
                             "sample": "%d scenes per step of the same workload (bounded sample of the batch of %d), oracle/pointops_oracle.c "
                                       "(OpenMP) + numpy fp32 MLP; the reference itself has no CPU implementation of this path" % (scenes, BATCH)},
            "e2e": {"value": val, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def tuned_plans():
    """measured build choice per chain shape (prb_debug_tuned_plans): CTAs per SM of the faster build"""
    import ctypes
    from pointrcnn_b200 import _cabi
    buf = (ctypes.c_int * (18 * 64))()
    n = _cabi.lib().prb_debug_tuned_plans(buf, 64)
    kinds_in, kinds_out = ("sa", "fp", "rows"), ("rows", "sa_max", "fp")
    builds = {2: "2 CTAs x (4 epilogue + 4 gather warps)", 1: "1 CTA x (8 + 8)", 3: "1 CTA x (8 + 12)", 4: "3 CTAs x (4 + 4)"}
    out = []
    for i in range(n):
        r = buf[18 * i:18 * i + 18]
        out.append({"in": kinds_in[r[0]], "out": kinds_out[r[1]], "nsample": r[3], "k_chunks": r[4], "tiles": r[5],
                    "np": [x for x in r[6:6 + r[2]]], "build": builds.get(r[9], r[9]),
                    "measured_us": {builds.get(r[10 + 2 * c], r[10 + 2 * c]): r[11 + 2 * c] for c in range(4) if r[10 + 2 * c]}})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-scenes", type=int, default=2, help="scenes per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip the reference-CUDA comparator leg")
    ap.add_argument("--no-train", action="store_true", help="skip the RPN training-step leg (BASELINE configs[2])")
    ap.add_argument("--no-rcnn", action="store_true", help="skip the RCNN stage-2 leg (BASELINE configs[3])")
    ap.add_argument("--no-eval", action="store_true", help="skip the end-to-end two-stage evaluation leg (BASELINE configs[4])")
    ap.add_argument("--inflight", type=int, default=6, help="independent batches in flight (CUDA streams); 1 = sequential")
    ap.add_argument("--graphs", type=int, default=1, help="1: one CUDA graph per pipeline slot (default), 0: eager launches")
    ap.add_argument("--pool", type=int, default=40, help="distinct input batches rotated through (40 x 4.2 MB > 126 MB L2)")
    ap.add_argument("--profile-out", default=None, help="write the line as indented JSON here as well")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the backbone features the timed path returned for its last step to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    from pointrcnn_b200 import _cabi, prof
    from pointrcnn_b200.parallel_utils import max_over_ranks
    from pointrcnn_b200.pipeline import BatchPipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W, K = max(3, args.warmup), max(1, args.steps)
    F = max(1, args.inflight)
    G = bool(args.graphs)

    net = build_model(dev)
    stage = build_rpn_stage(dev, net)
    # input pool: distinct batches, together larger than the 126 MB L2, rotated through -> no step finds its input in L2
    P = max(1, args.pool)
    host_pool = [torch.from_numpy(make_scenes((rank * P + i) * BATCH, BATCH)).pin_memory() for i in range(P)]
    dev_pool = [h.to(dev) for h in host_pool]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2 (sequential pass)
    pipe = BatchPipeline(lambda x: net(x)[1], inflight=F, device=dev, graphs=G)
    pipe_rpn = BatchPipeline(lambda x: stage(x), inflight=F, device=dev, graphs=G)
    pipe_feat = BatchPipeline(lambda x: net(x)[1], inflight=min(F, 3), device=dev, graphs=G)

    def barrier():
        if world > 1:
            dist.barrier()

    def timed(run_k):
        """time the K-step region once (barrier + sync on both sides, CUDA events, max over ranks); returns [ms per step]"""
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        t0.record()
        run_k(0)
        t1.record()
        torch.cuda.synchronize(); barrier()
        return [max_over_ranks(t0.elapsed_time(t1), device=dev) / K]

    def summary(ms_list):
        return {"n": len(ms_list), "ms_per_step_median": statistics.median(ms_list), "ms_per_step_min": min(ms_list),
                "ms_per_step_max": max(ms_list), "timed_seconds": sum(ms_list) * K * 1e-3}

    checksum = [0.0]

    def consume_rois(i, res):
        rois, scores = res
        checksum[0] += float(scores.numpy().sum())       # the host consumer: touches every batch's proposals
        return None

    def last_step_outputs():
        """the (B,128,16384) features the timed path returned for its last step (with graphs: the replay's static output
        of that step's slot), input batch (K-1) % P: all 16 scenes and channels at a fixed, seeded sample of 4096 points
        (32 MB), plus the scene-mean feature of every channel over all points"""
        feats = pipe.slots[(K - 1) % F].static_out[0] if G else pipe.run([dev_pool[(K - 1) % P]])[0]
        cols = torch.from_numpy(np.sort(np.random.default_rng(0).choice(POINTS, 4096, replace=False))).to(dev)
        return {"features_sample": feats.index_select(2, cols).float().cpu().numpy(),
                "features_mean": feats.double().mean(2).cpu().numpy()}

    sampler = ClockSampler(local) if rank == 0 else None
    with torch.no_grad():
        net(dev_pool[0])                                                    # first call: the chain plans are measured here
        torch.cuda.synchronize()
        launches0 = _cabi.launch_count()
        net(dev_pool[0])
        torch.cuda.synchronize()
        launches = _cabi.launch_count() - launches0                       # native kernels of one backbone forward
        for i in range(W):
            net(dev_pool[i % P])
            stage(dev_pool[i % P])
        pipe.run([dev_pool[i % P] for i in range(2 * F)], keep=False)       # captures the graphs
        pipe_rpn.run([host_pool[i % P] for i in range(2 * F)], to_host=True, consume=consume_rois)
        pipe_feat.run([host_pool[i % P] for i in range(4)], to_host=True, consume=lambda i, r: None)
        torch.cuda.synchronize()
        if sampler:
            sampler.wait_started()
            sampler.mark()

        # ---------------- device-resident throughput: K steps, F independent batches in flight
        ms_list = timed(lambda off: pipe.run([dev_pool[(off + i) % P] for i in range(K)], keep=False))
        ms = statistics.median(ms_list)
        dumped = last_step_outputs() if args.dump_outputs and rank == 0 else None

        # ---------------- end to end: pinned host input -> H2D -> backbone -> heads -> proposals -> D2H -> host consumer
        e2e_list = timed(lambda off: pipe_rpn.run([host_pool[(off + i) % P] for i in range(K)], to_host=True, consume=consume_rois))
        ms_e2e = statistics.median(e2e_list)
        d2h_bytes = BATCH * 100 * 7 * 4 + BATCH * 100 * 4

        # ---------------- secondary: the full feature tensor back on the host (PCIe bound)
        feat_list = timed(lambda off: pipe_feat.run([host_pool[(off + i) % P] for i in range(K)], to_host=True,
                                                    consume=lambda i, r: None))
        ms_feat = statistics.median(feat_list)

        # ---------------- strong scaling: global batch 16 -> 16/world scenes per GPU per step
        strong = None
        if world > 1 and BATCH % world == 0:
            bs = BATCH // world
            Fs = min(24, F * max(1, world // 2))
            pipe_s = BatchPipeline(lambda x: net(x)[1], inflight=Fs, device=dev, graphs=G)
            small = [d[:bs] for d in dev_pool]
            pipe_s.run([small[i % P] for i in range(2 * Fs)], keep=False)
            s_list = timed(lambda off: pipe_s.run([small[(off + i) % P] for i in range(K)], keep=False))
            ms_s = statistics.median(s_list)
            strong = {"global_batch": BATCH, "scenes_per_gpu_per_step": bs, "batches_in_flight": Fs, "ms_per_step": ms_s,
                      "value": BATCH / (ms_s * 1e-3), "unit": "scenes/s", "repeats": summary(s_list),
                      "note": "same K steps, each step = 16 scenes over all GPUs; efficiency = value / (N=1 value)"}

        # ---------------- sequential pass (one batch at a time, L2 flushed in between): per-batch latency and the
        # per-kernel-family breakdown (CUDA events on the launching stream)
        KS = K
        import gc
        gc.collect()                      # pinned buffers / graphs of the pipelined legs are released here, not inside a timed step
        for i in range(2):
            net(dev_pool[i % P])
        torch.cuda.synchronize()
        # every step is collected on its own and the MEDIAN step (by its total) is reported with its family breakdown: one
        # host-side hiccup (a deferred free, a page fault of the launch path) otherwise lands in whichever family it interrupts
        per_step = []
        for i in range(KS):
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            prof.enable()
            flush.fill_(1.0)
            a.record()
            net(dev_pool[i % P])
            b_.record()
            torch.cuda.synchronize()
            prof.disable()
            per_step.append((a.elapsed_time(b_), prof.collect()))
        per_step.sort(key=lambda t: t[0])
        ms_seq, fam = per_step[len(per_step) // 2]
        ms_seq_all = [t[0] for t in per_step]
        KS_FAM = 1                        # `fam` holds ONE step
        # the same single batch with the geometry chain (4 FPS levels, ball queries, 3-NN: coordinates only) on side
        # streams, overlapping the feature MLPs of the previous level (backbone._forward_planned): per-batch latency when
        # there is no second batch to overlap with
        from pointrcnn_b200 import config as prb_config
        ms_plan = None
        try:
            with prb_config.override(enable_plan=True):
                for i in range(2):
                    net(dev_pool[i % P])
                torch.cuda.synchronize()
                evp = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KS)]
                for i, (a, b_) in enumerate(evp):
                    flush.fill_(1.0)
                    a.record()
                    net(dev_pool[i % P])
                    b_.record()
                torch.cuda.synchronize()
                ms_plan = statistics.median(a.elapsed_time(b_) for a, b_ in evp)
        except Exception as e:
            ms_plan = None
    # ---------------- BASELINE configs[2]: RPN training step, data parallel over the ranks (16 scenes per GPU), gradient
    # all-reduce bucketed and overlapped with backward (parallel_utils.GradBucketReducer over NCCL)
    train = None
    if not args.no_train:
        from pointrcnn_b200.train.step import RPNTrainer, synthetic_labels
        tr = RPNTrainer(input_channels=CHANNELS - 3, device=dev, world=world)
        labels = [synthetic_labels(dev_pool[i], seed=rank * 100 + i) for i in range(4)]
        KT = K
        for i in range(2):
            tr.step(dev_pool[i % 4], *labels[i % 4], grad_norm_clip=1.0)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        t0.record()
        for i in range(KT):
            loss_t, _ = tr.step(dev_pool[i % 4], *labels[i % 4], grad_norm_clip=1.0)
        t1.record()
        torch.cuda.synchronize(); barrier()
        ms_t = max_over_ranks(t0.elapsed_time(t1) / KT, device=dev)
        train = {"what": "RPN training step (BASELINE configs[2]): train-mode forward on the index natives + cuDNN MLPs, bin-based loss, "
                         "backward (scatter kernels K3/K6/K9), bucketed NCCL all-reduce overlapped with backward, fused Adam",
                 "ms_per_step": ms_t, "value": BATCH * world / (ms_t * 1e-3), "unit": "scenes/s", "steps": KT, "batch_per_gpu": BATCH,
                 "allreduce_bytes_per_step": tr.reducer.bytes_per_step if world > 1 else 0, "buckets": len(tr.reducer.buckets),
                 "collective": "ncclAllReduce(sum) x %d buckets per step on a side stream" % len(tr.reducer.buckets) if world > 1 else None,
                 "final_loss": float(loss_t)}
        tr.reducer.remove()
        del tr
        torch.cuda.empty_cache()
        # second training phase (tools/train_rcnn.py --train_mode rcnn, RPN fixed): 4 scenes per GPU, 64 sampled RoIs per scene
        try:
            from pointrcnn_b200.train.step import RCNNTrainer
            rt = RCNNTrainer(input_channels=CHANNELS - 3, device=dev, world=world)
            with torch.no_grad():
                rt.rpn.rpn_reg_layer[-1].conv.weight.mul_(0.2)
            pcs = [dev_pool[i][:4].contiguous() for i in range(2)]
            gts = []
            for pc4 in pcs:                      # GT boxes = 8 of the scene's own proposals (foreground RoIs exist), 4 padding rows
                g4 = torch.zeros((4, 12, 7), device=dev)
                g4[:, :8] = rt.rpn_outputs(pc4, None)["roi_boxes3d"][:, ::60][:, :8]
                gts.append(g4)
            for i in range(2):
                rt.step(pcs[i % 2], gts[i % 2], grad_norm_clip=1.0)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier(); torch.cuda.synchronize()
            t0.record()
            for i in range(KT):
                loss_r, _ = rt.step(pcs[i % 2], gts[i % 2], grad_norm_clip=1.0)
            t1.record()
            torch.cuda.synchronize(); barrier()
            ms_r = max_over_ranks(t0.elapsed_time(t1) / KT, device=dev)
            train["rcnn_phase"] = {"what": "RCNN training step with the RPN fixed: fused RPN stage (no grad) -> target layer (64 RoIs per scene) -> RCNN "
                                           "network forward / backward -> get_rcnn_loss -> bucketed all-reduce -> fused Adam; 4 scenes per GPU",
                                   "ms_per_step": ms_r, "value": 4 * world / (ms_r * 1e-3), "unit": "scenes/s", "steps": KT,
                                   "allreduce_bytes_per_step": rt.reducer.bytes_per_step if world > 1 else 0, "final_loss": float(loss_r)}
            rt.reducer.remove()
            del rt
        except Exception as e:
            if world > 1:
                raise
            train["rcnn_phase"] = {"unavailable": "%s: %s" % (type(e).__name__, e)}
        torch.cuda.empty_cache()

    # ---------------- BASELINE configs[3]: RCNN stage 2 (roipool3d of 4 x 512 RoIs x 512 points + RCNN PointNet++), rank 0 only
    rcnn = None
    if not args.no_rcnn and rank == 0:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        try:
            import bench_rcnn_stage
            rcnn = bench_rcnn_stage.measure(dev, steps=K, warm=5)
        except Exception as e:
            rcnn = {"unavailable": "%s: %s" % (type(e).__name__, e)}
        torch.cuda.empty_cache()
    # ---------------- BASELINE configs[4]: end-to-end two-stage evaluation, global batch 8 sharded over the ranks
    eval_e2e = None
    if not args.no_eval:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        try:
            import bench_eval_e2e
            eval_e2e = bench_eval_e2e.measure(dev, rank=rank, world=world, steps=K, warm=3, barrier=barrier,
                                              max_over_ranks=max_over_ranks)
        except Exception as e:
            if world > 1:
                raise          # a rank that drops out of the barriers would hang the others
            eval_e2e = {"unavailable": "%s: %s" % (type(e).__name__, e)}
        torch.cuda.empty_cache()
    clocks = sampler.stop() if sampler else None

    # ---------------- the reference's CUDA-extension build (oracle/_ref kernels + cuDNN MLP), same process, same inputs
    ref_cuda = None
    if rank == 0 and world == 1 and not args.no_ref_cuda:
        try:
            from oracle import refgpu
            if not refgpu.available():
                ref_cuda = {"unavailable": "oracle/_ref/libref_pointops.so not built"}
            else:
                from oracle.ref_backbone import backbone as ref_backbone
                with torch.no_grad():
                    for i in range(3):
                        ref_backbone(net, dev_pool[i % P])
                    torch.cuda.synchronize()
                    KR = K
                    evr = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KR)]
                    for i, (a, b_) in enumerate(evr):
                        flush.fill_(1.0)
                        a.record()
                        ref_backbone(net, dev_pool[i % P])
                        b_.record()
                    torch.cuda.synchronize()
                    ms_ref_single = sum(a.elapsed_time(b_) for a, b_ in evr) / KR
                    pipe_ref = BatchPipeline(lambda x: ref_backbone(net, x)[1], inflight=F, device=dev, graphs=False)
                    pipe_ref.run([dev_pool[i % P] for i in range(F)], keep=False)
                    torch.cuda.synchronize()
                    KP = K
                    a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    pipe_ref.run([dev_pool[i % P] for i in range(KP)], keep=False)
                    b_.record()
                    torch.cuda.synchronize()
                    ms_ref_pipe = a.elapsed_time(b_) / KP
                ref_cuda = {"impl": "reference CUDA kernels (oracle/_ref, unmodified sources rebuilt for sm_100a) + torch cuDNN/cuBLAS MLP, "
                                    "reference call order (pointnet2_modules.py:19-55,127-156)",
                            "single_stream": {"ms_per_step": ms_ref_single, "value": BATCH / (ms_ref_single * 1e-3), "steps": KR},
                            "pipelined": {"ms_per_step": ms_ref_pipe, "value": BATCH / (ms_ref_pipe * 1e-3), "steps": KP,
                                          "batches_in_flight": F, "graphs": False},
                            "unit": "scenes/s", "cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32)}
        except Exception as e:      # the comparator must never take the bench line down
            ref_cuda = {"unavailable": "%s: %s" % (type(e).__name__, e)}

    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return

    pk = peaks()
    sa_flops, fp_flops = mlp_flops_per_scene(net)
    tf32_peak = pk["bf16"] / 2.0          # tcgen05 kind::tf32 runs at half the bf16 rate; bf16 figure is the measured one
    fam_ms = {k: v[0] / KS_FAM for k, v in fam.items()}
    traffic = ncu_traffic()
    kernels = []
    if "sa_mlp" in fam_ms:
        kernels.append({"name": "mlp_chain kernels (SA: gather + SharedMLP + max-pool)", "family": "sa_mlp", "ms_per_step": fam_ms["sa_mlp"],
                        "bound": "tensor", "achieved": sa_flops * BATCH / (fam_ms["sa_mlp"] * 1e-3) / 1e12, "peak": tf32_peak,
                        "unit": "TFLOP/s"})
    if "fp_mlp" in fam_ms:
        kernels.append({"name": "mlp_chain kernels (FP: interpolate + SharedMLP)", "family": "fp_mlp", "ms_per_step": fam_ms["fp_mlp"],
                        "bound": "tensor", "achieved": fp_flops * BATCH / (fam_ms["fp_mlp"] * 1e-3) / 1e12, "peak": tf32_peak,
                        "unit": "TFLOP/s"})
    if "fps" in fam_ms:
        rounds = sum(m.npoint - 1 for m in net.SA_modules)
        npts = [POINTS] + [m.npoint for m in net.SA_modules]
        fps_bytes = sum(npts[i] * 12 + npts[i + 1] * 16 for i in range(len(net.SA_modules))) * BATCH
        kernels.append({"name": "fps_pruned_kernel + fps_rank_kernel (dependency chain: %d serial rounds/scene)" % rounds, "family": "fps",
                        "ms_per_step": fam_ms["fps"], "bound": "hbm", "achieved": fps_bytes / (fam_ms["fps"] * 1e-3) / 1e9,
                        "peak": pk["hbm"], "unit": "GB/s", "us_per_round": fam_ms["fps"] * 1e3 / rounds})
    for name in ("ball_query", "three_nn", "transpose"):
        if name in fam_ms:
            kernels.append({"name": name, "family": name, "ms_per_step": fam_ms[name]})
    for name in sorted(fam_ms):                      # prof_detail: one line per chain launch shape
        if name.startswith(("sa_mlp ", "fp_mlp ")):
            kernels.append({"name": name, "ms_per_step": fam_ms[name]})
    for k in kernels:
        if "achieved" in k:
            k["frac"] = k["achieved"] / k["peak"]
        k["share"] = k["ms_per_step"] / ms_seq     # share of the sequential (single batch) step
        if k.get("family") in traffic:
            k["traffic"] = traffic[k["family"]]
    # Dominant kernel of the PIPELINED step = largest share of SM-time: a chain launch fills the GPU, while the
    # sampling kernels hold one CTA per scene (16 of the SMs) for their duration.
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    for k in kernels:
        if "achieved" in k:
            sm_frac = min(1.0, BATCH / n_sm) if k["name"].startswith("fps") else 1.0
            k["sm_time_ms"] = k["ms_per_step"] * sm_frac
    dom = max((k for k in kernels if "achieved" in k), key=lambda k: k["sm_time_ms"], default=None)
    roofline = None
    if dom:
        roofline = {"kernel": dom["name"], "bound": dom["bound"], "achieved": dom["achieved"], "peak": dom["peak"], "unit": dom["unit"],
                    "frac": dom["frac"], "traffic": dom.get("traffic"),
                    "traffic_source": traffic.get("_source") if dom.get("traffic") is not None else None,
                    "algorithmic_flops_per_step": (sa_flops if dom.get("family") == "sa_mlp" else fp_flops) * BATCH if dom["bound"] == "tensor" else None,
                    "peak_source": pk["src"] + (" bf16/2" if dom["bound"] == "tensor" else " copy"),
                    "share_of_step": dom["share"],
                    "share_of_sm_time": dom["sm_time_ms"] / sum(k.get("sm_time_ms", k["ms_per_step"]) for k in kernels if "family" in k),
                    "timing": "CUDA events around the family's launches, sequential pass with L2 flush (single_batch), median of %d steps" % KS}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        cval, cdt = time_cpu(folded_specs(net.cpu()), args.cpu_scenes)
        cpu = {"value": cval, "unit": "scenes/s", "cores": O.num_threads(), "kind": "port",
               "sample": "%d scenes of the same workload, %.1f s (oracle C/OpenMP ops + numpy fp32 MLP)" % (args.cpu_scenes, cdt)}

    scenes = BATCH * world
    value = scenes / (ms * 1e-3)
    single_val = BATCH / (ms_seq * 1e-3)
    vs_ref = None
    if ref_cuda and "pipelined" in ref_cuda:
        vs_ref = {"pipelined": value / ref_cuda["pipelined"]["value"], "single_stream": single_val / ref_cuda["single_stream"]["value"],
                  "note": "pipelined: both sides with %d batches in flight; single_stream: one batch at a time, L2 flushed" % F}
    line = {"metric": METRIC, "value": value, "unit": "scenes/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (tf32 tensor-core MLP, fp32 accumulate)", "data": "synthetic",
            "config": workload_config(world),
            "pipeline": {"batches_in_flight": F, "cuda_graphs": G,
                         "l2": "inputs rotate through %d distinct batches (%.0f MB > 126 MB L2)" % (P, P * BATCH * POINTS * CHANNELS * 4 / 1e6)},
            "repeats": summary(ms_list),
            "single_batch": {"ms_per_step": ms_seq, "value": single_val, "unit": "scenes/s", "ms_per_step_planned": ms_plan,
                             "ms_per_step_min_max": [min(ms_seq_all), max(ms_seq_all)],
                             "note": "one batch at a time on one stream (eager launches), 256 MB L2 flush write between steps"},
            "e2e": {"value": scenes / (ms_e2e * 1e-3), "unit": "scenes/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": host_pool[0].numel() * 4, "d2h_bytes_per_step": d2h_bytes,
                    "what": "RPN stage: pinned host points -> H2D -> backbone -> fused cls/reg heads -> proposal layer (TEST: 9000 pre-NMS, "
                            "100 post-NMS, thr 0.8) -> D2H of rois (B,100,7) + scores (B,100) -> host consumer per batch",
                    "repeats": summary(e2e_list), "consumer_checksum": checksum[0]},
            "e2e_features": {"value": scenes / (ms_feat * 1e-3), "unit": "scenes/s", "ms_per_step": ms_feat,
                             "h2d_bytes_per_step": host_pool[0].numel() * 4, "d2h_bytes_per_step": BATCH * 128 * POINTS * 4,
                             "what": "backbone only, full (B,128,16384) features copied to pinned host memory every step (PCIe bound)",
                             "repeats": summary(feat_list)},
            "gpu_launches": launches, "chain_plans": tuned_plans(), "clocks": clocks, "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu,
            "ref_cuda": ref_cuda, "vs_ref_cuda": vs_ref, "strong_scaling": strong, "train_step": train, "rcnn_stage": rcnn, "eval_e2e": eval_e2e}
    if args.profile_out:
        json.dump(line, open(args.profile_out, "w"), indent=1)
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
