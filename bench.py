"""bench.py -- scenes/sec of the PointNet++ SSG semseg SA+FP forward (8192-point ScanNet-shaped scenes).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the reference path on the host CPU cores
    python bench.py ... --dump-outputs DIR                   # also writes the last timed step's logits to DIR/logits.npy

A "step" is one forward of PointNet2SemSeg (model/pointnet2.py:131-162: 4 SA + 4 FP + head) over one batch
of `--batch` synthetic scenes per GPU (weak scaling: per-GPU work is fixed).  One JSON line is printed by
rank 0; see DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

NPOINTS = 8192
NUM_CLASSES = 21
METRIC = "scenes/sec PointNet++ SSG semseg SA+FP forward (8192 pts)"
# 2 * MACs of the C1 network per scene (SURVEY.md Appendix C)
FLOPS_PER_SCENE = 2 * 1250.6e6
FP1_HEAD_FLOPS_PER_SCENE = 2 * (405.8e6 + 156.2e6)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained"),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons; only samples that arrive inside a begin()..end() window are used
    (one window per timed region: the device-resident leg and the end-to-end legs).  Started well before the first
    timed region (nvidia-smi needs a few hundred ms to come up)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index, period_ms=20):
        self.rows, self.proc, self.windows = [], None, []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(period_ms)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def wait_ready(self, timeout=5.0):
        t = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t < timeout:
            time.sleep(0.02)

    def begin(self):
        self.windows.append([time.perf_counter(), None])

    def end(self):
        self.windows[-1][1] = time.perf_counter()

    def close(self):
        if self.proc is not None:
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if not any(a <= ts <= (b if b is not None else ts) + 0.03 for a, b in self.windows):
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out_dir, logits):
    """Writes the logits of one step (B, N, C) as out_dir/logits.npy in float32; above DUMP_LIMIT_BYTES only the first
    scenes that fit are kept (4 KB left for the .npy header)."""
    logits = np.ascontiguousarray(logits, dtype=np.float32)
    keep = (DUMP_LIMIT_BYTES - 4096) // logits[0].nbytes
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), logits[:keep])


def build_model(device):
    from pn2_b200.models import PointNet2SemSeg
    torch.manual_seed(0)
    return PointNet2SemSeg(NUM_CLASSES).eval().to(device)


def host_batches(rank, batch, count):
    """`count` distinct pinned host batches in the loader's layout (B, N, 6) [xyz | rgb]."""
    from pn2_b200 import scenes, sharding
    out = []
    for i in range(count):
        a = torch.from_numpy(scenes.scannet_batch(sharding.weak_scene_ids(rank, batch, i)[0], batch, NPOINTS))
        out.append(a.pin_memory() if torch.cuda.is_available() else a)
    return out


def cpu_reference_scenes_per_sec(steps, warmup, sample_scenes):
    """The reference path on the host: oracle geometry (C, OpenMP) + torch CPU conv/BN, all host threads."""
    from oracle import modules_ref
    from oracle import oracle as orc
    from pn2_b200 import scenes
    from pn2_b200.models import PointNet2SemSeg
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = PointNet2SemSeg(NUM_CLASSES).eval()
    pts = torch.from_numpy(scenes.scannet_batch(0, sample_scenes, NPOINTS)).permute(0, 2, 1).contiguous()
    xyz, rgb = pts[:, :3], pts[:, 3:]
    for _ in range(warmup):
        modules_ref.semseg_forward_ref(model, xyz, rgb)
    t0 = time.perf_counter()
    for _ in range(steps):
        modules_ref.semseg_forward_ref(model, xyz, rgb)
    dt = time.perf_counter() - t0
    return sample_scenes * steps / dt, dt / steps * 1e3, max(cores, orc.num_threads())


def workload_config(batch, world):
    """The `config` object shared by both arms (the driver compares them)."""
    return {"workload": "PointNet2SemSeg SSG forward (4 SA + 4 FP + head), ScanNet-shaped synthetic scenes drawn with "
                        "replacement, 8192 pts, batch %d per GPU, scene-sharded (no collective)" % batch,
            "npoints": NPOINTS, "batch_per_gpu": batch, "global_batch": batch * world, "parallelism": "scene-sharded x%d" % world}


def run_reference(args):
    """The reference arm: the reference ships no CPU implementation of this path (model/pointnet2_utils.py:7 hard-imports
    the CUDA extension), so this times the restated CPU path -- the C oracle's geometry (OpenMP over the clouds of the
    batch) + torch CPU conv/BN on all host threads -- on the SAME config as our arm: one step = one batch of `--batch`
    scenes.  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    sample = args.batch
    value, ms, cores = cpu_reference_scenes_per_sec(args.steps, args.warmup, sample)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "scenes/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.batch, max(world, args.gpus)),
        "cpu_baseline": {"value": value, "unit": "scenes/s", "cores": cores, "kind": "port",
                         "sample": "%d scenes per step (one full batch of the workload) x %d steps; restated CPU path (the reference "
                                   "ships no CPU implementation): C oracle geometry, OpenMP over the clouds of the batch, + torch CPU "
                                   "conv/BN on all host threads" % (sample, args.steps)},
        "e2e": {"value": value, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def time_ref_gpu(model, device, batch):
    """The reference's own CUDA kernels + cuDNN modules on this GPU (oracle/_ref), a few steps."""
    from oracle import ref_cuda
    if not ref_cuda.available():
        return None
    from oracle import ref_gpu_model
    x = host_batches(7, batch, 1)[0].to(device).permute(0, 2, 1).contiguous()
    xyz, rgb = x[:, :3], x[:, 3:]
    for _ in range(3):
        ref_gpu_model.semseg_forward(model, xyz, rgb)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        ref_gpu_model.semseg_forward(model, xyz, rgb)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 5
    return {"value": batch / ms * 1e3, "unit": "scenes/s", "ms_per_step": ms,
            "what": "reference CUDA kernels compiled verbatim (oracle/_ref/ref_cuda.so) + stock torch Conv/BN (cuDNN, "
                    "TF32 allowed as torch defaults), batch %d, inputs resident, 5 steps" % batch}


def time_train_step_msg(device, batch=4, steps=8, world=1, rank=0):
    """BASELINE config[1]: MSG semseg TRAIN step (forward + backward + Adam), `batch` scenes per GPU, scenes sharded over
    the ranks.  The step is replayed as CUDA graphs (pn2_b200.models.GraphedTrainStep); with several ranks the gradients
    live in one flat buffer that is all-reduced once per step (NCCL) between the backward graph and the optimizer
    graph -- the only collective of the whole path.  Returns (graph ms, eager ms), timed on the device (CUDA events);
    max over ranks by the caller."""
    import torch.nn.functional as F
    from pn2_b200 import scenes
    from pn2_b200.models import GraphedTrainStep, PointNet2Multiview2Msg
    torch.manual_seed(0)
    net = PointNet2Multiview2Msg(NUM_CLASSES).to(device).train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)
    pts = torch.from_numpy(scenes.scannet_batch(77 + 1000 * rank, batch, NPOINTS)).to(device)
    xyz = pts[:, :, :3].permute(0, 2, 1).contiguous()
    img = torch.randn(batch, 128, NPOINTS, device=device)
    target = (pts[:, :, 2].clamp(0, 2.69) / 2.7 * 20).long() + 1

    def loss_fn(logits, tgt):
        return F.cross_entropy(logits.reshape(-1, NUM_CLASSES), tgt.reshape(-1), ignore_index=0)

    def timed(fn, n):
        evs = []
        for _ in range(n + 2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return float(np.median([x.elapsed_time(y) for x, y in evs[2:]]))

    eager_ms = 0.0
    if world == 1:  # the eager loop as a data point (host-bound at this batch size)
        def eager():
            opt.zero_grad(set_to_none=True)
            loss_fn(net(xyz, img), target).backward()
            opt.step()
        eager_ms = timed(eager, 4)
        opt.zero_grad(set_to_none=True)
    stepper = GraphedTrainStep(net, opt, loss_fn, xyz, img, target)
    ms = timed(lambda: stepper.step(xyz, img, target), steps)
    del stepper, net, opt
    torch.cuda.empty_cache()
    return ms, eager_ms


def time_other_configs(device, B):
    """BASELINE configs 2-4 on one GPU as data points (inference, fused path, CUDA events): the MSG stack forward (config 2's
    network), multi-view lifting + point branch (config 3), the nuScenes backbone at 16 384 and 34 720 points (config 4)."""
    from pn2_b200 import scenes
    from pn2_b200.models import PipelinedForward, PointNet2Backbone, PointNet2Multiview2, PointNet2Multiview2Msg
    out = {}

    def eager_ms(fn, iters=5):
        with torch.no_grad():
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(iters):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fn(); b.record(); torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    def pipelined_ms(model, a, b_, n=40, depth=6):
        pipe = PipelinedForward(model, a, b_, depth=depth)
        for _ in range(2 * depth):
            pipe.submit(a, b_)
        pipe.join()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            pipe.submit(a, b_)
        pipe.join()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    torch.manual_seed(0)
    pts = scenes.scannet_batch(0, B, NPOINTS).astype(np.float32)
    xyz = torch.from_numpy(pts[:, :, :3]).to(device).permute(0, 2, 1).contiguous()
    img = torch.randn(B, 128, NPOINTS, device=device)
    msg = PointNet2Multiview2Msg(NUM_CLASSES).eval().to(device)
    ms = pipelined_ms(msg, xyz, img)
    out["config2_msg_forward"] = {"ms_per_step": ms, "value": B / ms * 1e3, "unit": "scenes/s", "batch": B,
                                  "what": "PointNet2Multiview2Msg point branch forward (MSG SA x6, FP x4, head; synthetic lifted features), "
                                          "6 graphs in flight"}
    del msg
    V = 3
    mv = [scenes.multiview_inputs(7000 + i, pts[i, :, :3], V, 128) for i in range(B)]
    feats = torch.from_numpy(np.stack([m[0] for m in mv])).to(device)
    depth = torch.from_numpy(np.stack([m[1] for m in mv])).to(device)
    poses = torch.from_numpy(np.stack([m[2] for m in mv]).astype(np.float32)).to(device)
    ssg = PointNet2Multiview2(NUM_CLASSES).eval().to(device)
    view_args = (scenes.SCANNET_INTRINSIC, 0.1, 4.0, scenes.SCANNET_IMAGE_DIMS, 0.05)
    ms_eager = eager_ms(lambda: ssg.forward_views(xyz, feats, depth, poses, *view_args))
    # the same call as CUDA graphs, 6 batches in flight on 6 streams (pn2_b200.models.GraphedViews)
    from pn2_b200.models import GraphedViews
    from pn2_b200.pointnet_util import fps_policy
    streams = [torch.cuda.Stream(device) for _ in range(6)]
    slots = []
    with fps_policy("throughput"):
        for st in streams:
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):
                slots.append(GraphedViews(ssg, xyz, feats, depth, poses, *view_args))
            torch.cuda.current_stream().wait_stream(st)

    def views_round(n):
        for k in range(n):
            st = streams[k % 6]
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):
                slots[k % 6].run(xyz, feats, depth, poses)
        for st in streams:
            torch.cuda.current_stream().wait_stream(st)

    views_round(12)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    views_round(30)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 30
    out["config3_forward_views"] = {"ms_per_step": ms, "value": B / ms * 1e3, "unit": "scenes/s", "batch": B, "eager_ms_per_step": ms_eager,
                                    "what": "PointNet2Multiview2.forward_views: lifting of 3 views (128 x 32 x 41 maps, ENet output as "
                                            "input, first-non-zero reduction) + point branch; CUDA graphs (GraphedViews), 6 batches in flight; "
                                            "inputs copied into the static buffers every step"}
    del slots
    ms = pipelined_ms(ssg, xyz, img)
    out["config3_point_branch"] = {"ms_per_step": ms, "value": B / ms * 1e3, "unit": "scenes/s", "batch": B,
                                   "what": "PointNet2Multiview2 point branch (lifted features resident), 6 graphs in flight"}
    del ssg, feats, depth, poses
    bb = PointNet2Backbone().eval().to(device)
    for n in (16384, 34720):
        sw = [scenes.lidar_sweep(50 + i, n) for i in range(16)]
        x3 = torch.from_numpy(np.stack([s_[0] for s_ in sw]).astype(np.float32)).to(device).permute(0, 2, 1).contiguous()
        f2 = torch.from_numpy(np.stack([s_[1] for s_ in sw]).astype(np.float32)).to(device).permute(0, 2, 1).contiguous()
        ms_eager = eager_ms(lambda: bb(x3, f2))
        # the sampling of a 16-sweep batch occupies 64 SMs (one 4-CTA cluster per sweep) for most of the forward: two graph
        # instances in flight let the second batch's sampling use the other half of the GPU
        ms = pipelined_ms(bb, x3, f2, n=12, depth=2)
        out["config4_backbone_n%d" % n] = {"ms_per_step": ms, "value": 16 / ms * 1e3, "unit": "sweeps/s", "batch": 16,
                                           "eager_ms_per_step": ms_eager,
                                           "what": "nuScenes backbone (model/pointmaskrcnn.py:8-32), batch 16 x %d points, CUDA "
                                                   "graphs with 2 batches in flight (eager, one batch at a time: eager_ms_per_step)" % n}
        del x3, f2
    del bb
    torch.cuda.empty_cache()
    return out


def ncu_traffic(kernel_substr="row_mlp_tc_kernel_bf16_fp(", grid=None):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed `ncu --set full` summary of this
    round (profiles/r2_tc_mlp_ncu_full_summary.csv, written by scripts/summarize_ncu_full.py from the .ncu-rep): the LAST
    matching launch of one forward (fp1 + head).  Returns (bytes or None, file name)."""
    import csv
    for name in ("r2_tc_mlp_ncu_full_summary.csv", "r1_tc_mlp_v5_ncu_full_summary.csv"):
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        try:
            rows = list(csv.reader(open(path)))
            head = rows[0]
            ir, iw = head.index("dram__bytes_read.sum"), head.index("dram__bytes_write.sum")
            units = rows[1]
            scale = {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}
            hit = [r for r in rows[2:] if r and kernel_substr in r[0]]
            if hit:
                r = hit[-1]
                return float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0), "profiles/" + name
        except (ValueError, IndexError, OSError):
            continue
    return None, None


def op_rooflines(device, batch, pk):
    """HBM-roofline figures of the standalone gather / interpolate kernels at the C1 shapes (timed alone -> burst peak)."""
    from pn2_b200 import _lib as _lib_mod
    from pn2_b200 import pointnet2_utils as pu
    from pn2_b200.pointnet_util import fps_gather_cl, three_nn_weights_cl
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    x = host_batches(5, batch, 1)[0].to(device)
    xyz = x[:, :, :3].contiguous()

    def t_ms(fn, iters=5):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    out = {}
    lib = _lib_mod.load()
    for mode, label in ((1, "fps_8192_to_1024_one_cta_per_cloud"), (2, "fps_8192_to_1024_cluster4_dsmem")):
        lib.pn2_debug_set_fps_mode(mode)
        ms = t_ms(lambda: fps_gather_cl(xyz, 1024))
        out[label] = {"ms": ms, "us_per_round": ms * 1e3 / 1023, "clouds_in_flight": batch,
                      "algorithmic_gbs": batch * (12 * NPOINTS + 16 * 1024) / ms / 1e6,
                      "note": "latency-bound: 1023 dependent rounds per cloud; HBM bytes are read once (cloud lives on chip)"}
    lib.pn2_debug_set_fps_mode(0)
    _, new_xyz = fps_gather_cl(xyz, 1024)
    i3, w3 = three_nn_weights_cl(xyz, new_xyz)
    for (C, m, n, bb) in ((128, 1024, NPOINTS, batch), (128, 4096, 16384, 64)):
        feats = torch.randn(bb, C, m, device=device)
        idx = torch.randint(0, m, (bb, n, 3), device=device, dtype=torch.int32)
        w = torch.rand(bb, n, 3, device=device)
        w = (w / w.sum(-1, keepdim=True)).contiguous()
        ms = t_ms(lambda: pu.three_interpolate(feats, idx, w))
        byts = bb * (24 * n + 4 * C * m + 4 * C * n)
        out["three_interpolate_b%d_c%d_m%d_n%d" % (bb, C, m, n)] = {"ms": ms, "gbs": byts / ms / 1e6, "frac_hbm": byts / ms / 1e6 / pk["hbm_gbs"]}
        del feats, idx, w
    for (C, N, M, K, bb) in ((64, NPOINTS, 1024, 32, batch), (128, 16384, 4096, 32, 64)):
        f = torch.randn(bb, C, N, device=device)
        idx = torch.randint(0, N, (bb, M, K), device=device, dtype=torch.int32)
        ms = t_ms(lambda: pu.grouping_operation(f, idx))
        byts = bb * (4 * M * K + 4 * C * min(N, M * K) + 4 * C * M * K)
        out["group_points_b%d_c%d_n%d_m%d_k%d" % (bb, C, N, M, K)] = {"ms": ms, "gbs": byts / ms / 1e6, "frac_hbm": byts / ms / 1e6 / pk["hbm_gbs"]}
        del f, idx
    # multi-view lifting (BASELINE config 3 shapes): V views of 128 x 32 x 41 feature maps onto 8192 points per scene
    from pn2_b200 import scenes as _sc
    from pn2_b200.projection import lift_views
    pts_np = x[:, :, :3].cpu().numpy()
    for V in (3, 5):
        mv = [_sc.multiview_inputs(7000 + i, pts_np[i], V, 128) for i in range(batch)]
        feats = torch.from_numpy(np.stack([m[0] for m in mv])).to(device)
        depth = torch.from_numpy(np.stack([m[1] for m in mv])).to(device)
        poses = torch.from_numpy(np.stack([m[2] for m in mv]).astype(np.float32)).to(device)
        for red in ("max", "first"):
            ms = t_ms(lambda: lift_views(xyz, feats, depth, poses, _sc.SCANNET_INTRINSIC, 0.1, 4.0, _sc.SCANNET_IMAGE_DIMS, 0.05, reduce=red))
            byts = batch * (12 * NPOINTS + V * (4 * 32 * 41 + 64) + 4 * 128 * min(V * 32 * 41, V * NPOINTS) + 4 * 128 * NPOINTS)
            out["lift_views_v%d_%s" % (V, red)] = {"ms": ms, "scenes_per_s": batch / ms * 1e3, "gbs": byts / ms / 1e6,
                                                   "frac_hbm": byts / ms / 1e6 / pk["hbm_gbs"]}
        del feats, depth, poses
    ms = t_ms(lambda: pu.ball_query(0.1, 32, xyz, new_xyz))
    out["ball_query_r0.1_k32_grid"] = {"ms": ms, "note": "grid build + query; brute force (first version) 0.345 ms"}
    return out


def run_ours(args):
    import torch.distributed as dist
    from pn2_b200 import _lib
    from pn2_b200 import pointnet_util as _pu
    from pn2_b200 import scenes as _scenes
    from pn2_b200 import sharding
    from pn2_b200.models import GraphedForward, PipelinedForward

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    pk = peaks()
    B = args.batch
    if args.fps_mode:
        _lib.load().pn2_debug_set_fps_mode(args.fps_mode)
    if args.tc_max_ctas > 0:
        _lib.load().pn2_debug_set_tc_max_ctas(args.tc_max_ctas)
    _pu.set_mlp_precision(args.precision)  # the drop-in modules default to fp32 (1e-5 parity); the benchmark path is bf16
    model = build_model(device)
    # rotating inputs: 24 distinct batches = 151 MB of input (+ the activations they produce) > the 126 MB L2
    n_rot = 24
    hosts = host_batches(rank, B, 8)
    devs = [torch.from_numpy(_scenes.scannet_batch(sharding.weak_scene_ids(rank, B, i)[0] + 1000, B, NPOINTS)).to(device).permute(0, 2, 1).contiguous()
            for i in range(n_rot)]  # (B, 6, N) resident, as the train script feeds it
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ex_xyz, ex_pts = devs[0][:, :3].contiguous(), devs[0][:, 3:].contiguous()
    graphed = None if args.no_graph else GraphedForward(model, ex_xyz, ex_pts)
    depth = 1 if args.no_graph else max(1, args.pipeline)
    pipe = PipelinedForward(model, ex_xyz, ex_pts, depth) if depth > 1 else None
    clocks = ClockSampler(local)

    def step(i):
        x = devs[i % n_rot]
        if graphed is not None:
            return graphed.run(x[:, :3], x[:, 3:])
        return model(x[:, :3], x[:, 3:])

    def run_e2e(pipe_, graphed_, out_shape, out_dtype, fwd, warm):
        """Pinned host (B, N, 6) -> H2D -> forward -> D2H of the result, every step.  `warm` untimed steps of the same
        protocol run first (pipeline fill, first touch of the pinned buffers), then exactly args.steps timed ones.  The
        read-back is split in two halves on two copy streams so that it overlaps the next batch's H2D and forward."""
        n_slots = max(depth, 1)
        stages = [torch.empty((B, NPOINTS, 6), dtype=torch.float32, device=device) for _ in range(n_slots)]
        outs_host = [torch.empty(out_shape, dtype=out_dtype).pin_memory() for _ in range(n_slots)]
        copy_in = torch.cuda.Stream(device)
        copy_out = [torch.cuda.Stream(device), torch.cuda.Stream(device)]
        slot_free = [None] * n_slots
        half = max(B // 2, 1)

        def one(i):
            k = i % n_slots
            with torch.cuda.stream(copy_in):
                if slot_free[k] is not None:
                    copy_in.wait_event(slot_free[k])   # the previous forward of this slot has consumed its staging buffer
                stages[k].copy_(hosts[i % len(hosts)], non_blocking=True)
                h2d = torch.cuda.Event()
                h2d.record(copy_in)
            x = stages[k].permute(0, 2, 1)
            if pipe_ is not None:
                y, done, st = pipe_.submit(x[:, :3], x[:, 3:], after=h2d)
            else:
                torch.cuda.current_stream().wait_event(h2d)
                y = graphed_.run(x[:, :3], x[:, 3:]) if graphed_ is not None else fwd(x[:, :3], x[:, 3:])
                done = torch.cuda.Event()
                done.record()
                st = torch.cuda.current_stream()
            slot_free[k] = done
            for c, (lo, hi) in enumerate(((0, half), (half, B))):
                if lo >= hi:
                    continue
                with torch.cuda.stream(copy_out[c]):
                    copy_out[c].wait_event(done)
                    outs_host[k][lo:hi].copy_(y[lo:hi], non_blocking=True)
                    d2h = torch.cuda.Event()
                    d2h.record(copy_out[c])
                st.wait_event(d2h)  # the slot's static output may only be overwritten after it has been read back

        def drain():
            if pipe_ is not None:
                pipe_.join()
            for c in copy_out:
                torch.cuda.current_stream().wait_stream(c)

        copy_in.wait_stream(torch.cuda.current_stream())
        for i in range(warm):
            one(i)
        drain()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        copy_in.wait_stream(torch.cuda.current_stream())
        for i in range(args.steps):
            one(warm + i)
        drain()
        b.record()
        barrier()
        return a.elapsed_time(b)

    with torch.no_grad():
        for i in range(args.warmup):
            step(i)
            if pipe is not None:
                pipe.submit(devs[i % n_rot][:, :3], devs[i % n_rot][:, 3:])
        if pipe is not None:
            pipe.join()
        barrier()
        # ---- (a) one step at a time, L2 flushed between steps: the latency of a single batch -----------------
        evs = []
        barrier()
        for i in range(args.steps):
            flush.zero_()  # L2 flush between timed steps (outside the timed events)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step(i)
            b.record()
            evs.append((a, b))
        barrier()
        serial_ms = sum(a.elapsed_time(b) for a, b in evs)
        # ---- (b) device-resident throughput: `depth` batches in flight, inputs rotate over a set larger than L2 ----
        launches0 = _lib.launch_count()
        clocks.wait_ready()
        barrier()
        clocks.begin()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(args.steps):
            x = devs[i % n_rot]
            if pipe is not None:
                last = pipe.submit(x[:, :3], x[:, 3:])[0]
            else:
                last = step(i)
        if pipe is not None:
            pipe.join()
        b.record()
        barrier()
        clocks.end()
        # a static graph output: copied now, before the legs below replay the same graphs
        last_logits = last.float().cpu().numpy() if args.dump_outputs else None
        total_ms = a.elapsed_time(b)
        launches = _lib.launch_count() - launches0
        if graphed is not None:
            launches = args.steps * graphed.kernels_per_replay
        # ---- the dominant kernel, timed with events inside eager steps of the same workload -------------
        timers = {}
        model.timers = timers
        model.single_stream = True   # nothing else on the GPU while the kernel is timed
        for i in range(max(3, min(args.steps, 10))):
            x = devs[i % n_rot]
            flush.zero_()
            model(x[:, :3], x[:, 3:])
        torch.cuda.synchronize()
        model.timers = None
        model.single_stream = False
        dom_ms = [a.elapsed_time(b) for a, b in timers.get("fp1_head", [])][1:]
        # ---- end to end: pinned host (B,N,6) -> H2D -> forward -> D2H of the result, every step ----------------------
        e2e_warm = max(args.warmup, 2 * depth)
        # (1) the reference protocol: the full fp32 logits come back (train_scannet_semseg.py:204 `pred.cpu().numpy()`)
        clocks.begin()
        e2e_ms = run_e2e(pipe, graphed, (B, NPOINTS, NUM_CLASSES), torch.float32, model, e2e_warm)
        clocks.end()
        # (2) predict(): the arg-max the evaluation loop takes from those logits, fused into the head kernel; 1 byte per point
        e2e_lab_ms = 0.0
        if model.can_fuse_labels() and not args.no_graph:
            pipe_l = PipelinedForward(model, ex_xyz, ex_pts, depth, labels=True) if depth > 1 else None
            graphed_l = GraphedForward(model, ex_xyz, ex_pts, labels=True) if depth <= 1 else None
            clocks.begin()
            e2e_lab_ms = run_e2e(pipe_l, graphed_l, (B, NPOINTS), torch.uint8, model.predict, e2e_warm)
            clocks.end()
            del pipe_l, graphed_l
        # (3) bf16 logits: the tensor-core head's outputs carry bf16-MMA precision; storing them as bf16 halves the read-back
        e2e_bf16_ms = 0.0
        if args.precision == "bf16" and model.can_fuse_labels() and not args.no_graph:
            pipe_h = PipelinedForward(model, ex_xyz, ex_pts, depth, logits_dtype=torch.bfloat16) if depth > 1 else None
            graphed_h = GraphedForward(model, ex_xyz, ex_pts, logits_dtype=torch.bfloat16) if depth <= 1 else None
            clocks.begin()
            e2e_bf16_ms = run_e2e(pipe_h, graphed_h, (B, NPOINTS, NUM_CLASSES), torch.bfloat16, None, e2e_warm)
            clocks.end()
            del pipe_h, graphed_h
        clocks.close()

        # ---- further legs of the same line (not the headline): fp32 MLP path, BASELINE config 1's batch of 2 ----------
        legs = {}
        if not args.no_graph and not args.no_extras:
            def pipelined_value(model_, xs, steps_, depth_):
                pp = PipelinedForward(model_, xs[0][:, :3].contiguous(), xs[0][:, 3:].contiguous(), depth_)
                for i in range(max(3, depth_)):
                    pp.submit(xs[i % len(xs)][:, :3], xs[i % len(xs)][:, 3:])
                pp.join()
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(steps_):
                    pp.submit(xs[i % len(xs)][:, :3], xs[i % len(xs)][:, 3:])
                pp.join()
                e1.record()
                barrier()
                return e0.elapsed_time(e1) / steps_

            def one_at_a_time_ms(model_, xs, steps_):
                g = GraphedForward(model_, xs[0][:, :3].contiguous(), xs[0][:, 3:].contiguous())
                ts = []
                for i in range(steps_ + 3):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    g.run(xs[i % len(xs)][:, :3], xs[i % len(xs)][:, 3:])
                    e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
                return float(np.median(ts[3:]))

            if args.precision == "bf16":
                prev = _pu.set_mlp_precision("fp32")
                try:
                    k32 = max(3, min(args.steps, 20))
                    ms32 = pipelined_value(model, devs, k32, depth)
                    legs["fp32"] = {"value": world * B / ms32 * 1e3, "unit": "scenes/s", "ms_per_step": ms32, "steps": k32, "dtype": "f32",
                                    "what": "the same workload on the fp32 FFMA shared-MLP kernels (row_mlp.cu; 1e-5 relative to the "
                                            "reference instead of the bf16 path's 2e-2), %d batches in flight" % depth}
                finally:
                    _pu.set_mlp_precision(prev)
            b2 = [d[:2].contiguous() for d in devs]   # BASELINE configs[0]: batch 2
            lat = one_at_a_time_ms(model, b2, 20)
            # a batch of 2 keeps two SMs busy in its sampling phase: four times as many graph instances in flight as for batch 32
            depth_b2 = 4 * depth
            thr = pipelined_value(model, b2, max(4 * depth_b2, min(args.steps, 200)), depth_b2)
            legs["batch2"] = {"latency_ms": lat, "value_one_at_a_time": world * 2 / lat * 1e3, "value": world * 2 / thr * 1e3, "unit": "scenes/s",
                              "ms_per_step": thr,
                              "what": "BASELINE configs[0] shape: batch 2 x 8192 points per GPU.  latency_ms = one CUDA-graph forward at a "
                                      "time, L2 flushed in between; value = %d graphs of batch 2 in flight" % depth_b2}

    # ---- BASELINE config[1]: the MSG train step, scenes sharded over the ranks, one gradient all-reduce -----------------
    train_ms, train_eager_ms = 0.0, 0.0
    if not args.no_extras:
        train_ms, train_eager_ms = time_train_step_msg(device, batch=4, world=world, rank=rank)

    t = torch.tensor([total_ms, e2e_ms, e2e_lab_ms, train_ms, e2e_bf16_ms] + [legs.get("fp32", {}).get("ms_per_step", 0.0),
                                                                 legs.get("batch2", {}).get("ms_per_step", 0.0)],
                     dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, e2e_lab_ms, train_ms, e2e_bf16_ms, ms32_max, msb2_max = t.tolist()
    if rank == 0:
        value = world * B * args.steps / (total_ms / 1e3)
        e2e_value = world * B * args.steps / (e2e_ms / 1e3)
        cfg = workload_config(B, world)
        line = {
            "metric": METRIC, "value": value, "unit": "scenes/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "ms_per_step_one_at_a_time": serial_ms / args.steps,
            "value_one_at_a_time": world * B * args.steps / (serial_ms / 1e3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": model.compute_dtype, "data": "synthetic",
            "config": cfg,
            "timing": {"l2": "inputs rotate over %d distinct batches (%.0f MB > L2); the one-at-a-time figure flushes L2 (256 MiB) "
                             "between steps" % (n_rot, n_rot * B * NPOINTS * 6 * 4 / 1e6),
                       "launch": "eager, 3 streams" if graphed is None else "CUDA graph replay (3 streams captured), %d batches in flight" % depth,
                       "e2e_warmup_steps": e2e_warm},
            "e2e": {"value": e2e_value, "unit": "scenes/s", "h2d_bytes_per_step": B * NPOINTS * 6 * 4,
                    "d2h_bytes_per_step": B * NPOINTS * NUM_CLASSES * 4, "ms_per_step": e2e_ms / args.steps,
                    "what": "pinned host (B, N, 6) -> H2D -> forward -> D2H of the (B, N, 21) fp32 logits every step (the reference's "
                            "evaluation protocol, train_scannet_semseg.py:204); %d untimed warm-up steps" % e2e_warm},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "tflops": value * FLOPS_PER_SCENE / 1e12,
        }
        if e2e_lab_ms > 0:
            line["e2e_labels"] = {"value": world * B * args.steps / (e2e_lab_ms / 1e3), "unit": "scenes/s",
                                  "h2d_bytes_per_step": B * NPOINTS * 6 * 4, "d2h_bytes_per_step": B * NPOINTS,
                                  "ms_per_step": e2e_lab_ms / args.steps,
                                  "what": "same protocol through PointNet2SemSeg.predict(): per-point class predictions (uint8) "
                                          "read back instead of fp32 logits; the arg-max is fused into the head kernel"}
        if e2e_bf16_ms > 0:
            line["e2e_bf16_logits"] = {"value": world * B * args.steps / (e2e_bf16_ms / 1e3), "unit": "scenes/s",
                                       "h2d_bytes_per_step": B * NPOINTS * 6 * 4, "d2h_bytes_per_step": B * NPOINTS * NUM_CLASSES * 2,
                                       "ms_per_step": e2e_bf16_ms / args.steps,
                                       "what": "same protocol with the (B, N, 21) logits stored and read back as bf16 (the tensor-core head "
                                               "computes them with bf16 operands; forward_fused(logits_dtype=torch.bfloat16))"}
        host_probe = os.path.join(ROOT, "profiles", "r2_host_link_probe.json")
        if os.path.exists(host_probe):
            line["e2e"]["host_link_ceiling"] = {"source": "profiles/r2_host_link_probe.json",
                                                "note": "measured pinned D2H bandwidth of this pool's boxes with all ranks copying at once "
                                                        "(GB/s aggregate): 56 / 75 / 80 / 109 at 1 / 2 / 4 / 8 GPUs, 76 with H2D running too; "
                                                        "fp32 logits need 41 GB/s per GPU at the device rate, so beyond 2 GPUs this leg is "
                                                        "bounded by the host links (8 GPUs: 126 k scenes/s = 87 GB/s D2H + 25 GB/s H2D)"}
        if "fp32" in legs:
            legs["fp32"]["ms_per_step"] = ms32_max
            legs["fp32"]["value"] = world * B / ms32_max * 1e3
            line["value_fp32"] = legs["fp32"]
        if "batch2" in legs:
            legs["batch2"]["ms_per_step"] = msb2_max
            legs["batch2"]["value"] = world * 2 / msb2_max * 1e3
            line["batch2"] = legs["batch2"]
            line["value_b2_latency_ms"] = legs["batch2"]["latency_ms"]
        extra = {}
        if train_ms > 0:
            extra["config2_msg_train_step"] = {
                "value": world * 4 / train_ms * 1e3, "unit": "scenes/s", "ms_per_step": train_ms, "batch_per_gpu": 4, "n_gpus": world,
                "launch": "CUDA graphs (pn2_b200.models.GraphedTrainStep)",
                "what": "BASELINE configs[1]: PointNet2Multiview2Msg point branch (model/pointnet2multiview.py:179-233), forward + "
                        "backward + Adam, 4 scenes per GPU, scene-sharded" + (", one NCCL all-reduce of the flat gradient buffer per step" if world > 1 else "")
                        + "; geometry and its backwards AND the shared MLPs (conv + batch-statistics BatchNorm + ReLU, forward and "
                          "backward: csrc/train_mlp.cu) on our kernels"}
            if train_eager_ms > 0:
                extra["config2_msg_train_step"]["eager_ms_per_step"] = train_eager_ms
        if dom_ms:
            ms = float(np.mean(dom_ms))
            achieved = B * FP1_HEAD_FLOPS_PER_SCENE / (ms / 1e3) / 1e12
            peak = pk["bf16_tflops_sustained"] or pk["bf16_tflops"]
            traffic, traffic_src = ncu_traffic() if B == 32 else (None, None)
            line["roofline"] = {"kernel": "row_mlp_tc_kernel (fused fp1 + head: 3-NN interpolation gather + 131-128-128-128-128-21 "
                                          "tcgen05 MLP over %d rows)" % (B * NPOINTS),
                                "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                                "traffic": traffic, "traffic_source": traffic_src,
                                "algorithmic_bytes": B * NPOINTS * (12 + 12 + 24 + 4 * NUM_CLASSES) + B * 1024 * 128 * 2,
                                "ms": ms, "share_of_step_one_at_a_time": ms / (serial_ms / args.steps),
                                "peak_source": pk["source"] + " bf16 sustained (kernel timed inside eager steps, alone on the GPU)"}
        if world == 1 and not args.no_extras:
            line["kernels"] = op_rooflines(device, B, pk)
            line["ref_gpu"] = time_ref_gpu(model, device, B)
            with torch.no_grad():
                extra.update(time_other_configs(device, B))
            cpu_steps = 3
            cpu_v, cpu_ms, cores = cpu_reference_scenes_per_sec(cpu_steps, 1, B)
            line["cpu_baseline"] = {"value": cpu_v, "unit": "scenes/s", "cores": cores, "kind": "port",
                                    "sample": "%d scenes per step (one full batch) x %d steps (+1 warm-up); restated CPU path (the reference "
                                              "ships no CPU implementation): C oracle geometry with OpenMP over the clouds + torch CPU "
                                              "conv/BN on all host threads" % (B, cpu_steps)}
        if extra:
            line["extra"] = extra
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_logits)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=32, help="scenes per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"],
                    help="shared-MLP arithmetic: bf16 tcgen05 tensor cores (2e-2, north_star) or fp32 FFMA (1e-5)")
    ap.add_argument("--pipeline", type=int, default=6, help="batches in flight (graph instances on separate streams)")
    ap.add_argument("--fps-mode", type=int, default=0, help="developer knob: 1 = one CTA per cloud, 2 = 4-CTA cluster per cloud")
    ap.add_argument("--tc-max-ctas", type=int, default=0, help="developer knob: cap resident CTAs/SM of the tensor-core MLP kernel")
    ap.add_argument("--no-graph", action="store_true", help="launch the forward eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-extras", action="store_true", help="skip the op rooflines / ref_gpu / cpu_baseline legs (for ncu runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the (B, N, 21) fp32 logits of the headline leg's last step as DIR/logits.npy "
                         "(rank 0; at most 64 MB: the first scenes of a larger batch); inputs and weights are seeded, so two "
                         "builds given the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
