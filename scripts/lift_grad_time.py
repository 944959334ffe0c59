"""Backward of the fused lifting (pn2_lift_views_grad) at the BASELINE config 3 shape: 32 scenes x 8192 points, V in {3, 5}
views of 128 x 32 x 41 maps from scenes.multiview_inputs, both reductions.

    python scripts/lift_grad_time.py [--out profiles/lift_grad_b200.json] [--batch 32]

Per (V, reduce): the forward lift_views; the backward alone (CUDA events around the ABI call, warmed up, a 256 MB buffer
overwritten before every timed call so that nothing is served from L2); its compulsory HBM traffic per scene
    4 C N (grad_out) + 4 V N (pix) + 4 V C H W (feats read; "first" reads them for the non-zero flags) + 4 V C H W (written)
as a fraction of the measured HBM copy figure 6 536.7 GB/s (BASELINE.md), the sort's traffic stated separately (an
estimate from the algorithm: cub's radix sort of 4-byte keys and payloads moves ~16 B per pair and pass over ceil(bits/8)
passes, plus the key kernel and the segment starts); the reference composition's backward on the same inputs
(Projection.apply per scene and view + F.max_pool1d / the fill loop, under autograd); and a torch.profiler breakdown of
one backward call by kernel.  The GPU name and power limit are read in the same run (nvidia-smi --query-gpu).
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import lift_grad_ref as lgr  # noqa: E402
from pn2_b200 import scenes  # noqa: E402
from pn2_b200.projection import lift_views, lift_views_grad  # noqa: E402

HBM_GBS = 6536.7  # measured HBM copy figure of one B200 (BASELINE.md), the denominator the project uses


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, flush, reps):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lift_grad_b200.json"))
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--reps", type=int, default=15)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    B, N, C = args.batch, 8192, 128
    W, H = scenes.SCANNET_IMAGE_DIMS
    HW = H * W
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = dict(gpu_info(), shape={"B": B, "N": N, "C": C, "H": H, "W": W}, hbm_gbs_denominator=HBM_GBS, runs=[])
    for V in (3, 5):
        pts = scenes.scannet_batch(7000, B, N)[:, :, :3].astype(np.float32)
        mv = [scenes.multiview_inputs(7000 + b, pts[b], V, C) for b in range(B)]
        feats = torch.from_numpy(np.stack([m[0] for m in mv])).to(dev)
        depth = torch.from_numpy(np.stack([m[1] for m in mv])).to(dev)
        poses = torch.from_numpy(np.stack([m[2] for m in mv]).astype(np.float32)).to(dev)
        p = torch.from_numpy(pts).to(dev)
        fargs = (p, feats, depth, poses, scenes.SCANNET_INTRINSIC, 0.1, 4.0, scenes.SCANNET_IMAGE_DIMS, 0.05)
        g = torch.randn(B, C, N, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
        for red in ("max", "first"):
            fwd = timed(lambda: lift_views(*fargs, reduce=red), flush, args.reps)
            _, pix, _ = lift_views(*fargs, reduce=red, return_pixels=True)
            bwd = timed(lambda: lift_views_grad(feats, pix, g, red), flush, args.reps)
            # the same backward through autograd (lift_views with feats.requires_grad), for the overhead of the Function
            f = feats.clone().requires_grad_(True)

            def autograd_bwd():
                out = lift_views(p, f, *fargs[2:], reduce=red)
                torch.autograd.grad(out, f, g)
            fwd_bwd = timed(autograd_bwd, flush, args.reps)
            compulsory = 4 * C * N + 4 * V * N + 2 * 4 * V * C * HW
            pairs = V * N if red == "max" else N
            keys = V * HW + 1
            bits = max(1, math.ceil(math.log2(B * keys)))
            sort_bytes = pairs * (16 * math.ceil(bits / 8) + 4 * V + 8 + 4) + 4 * keys
            # the reference composition's backward (Projection.apply per scene and view + reduction) on the same inputs
            ref_ms = []
            for _ in range(3):
                fr = feats.clone().requires_grad_(True)
                out_ref = lgr.composition_forward(fr, pix, red)
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                out_ref.backward(g)
                b.record()
                torch.cuda.synchronize()
                ref_ms.append(a.elapsed_time(b))
            # the two backwards agree (N(0,1) grad_out: only the summation order differs)
            ours = lift_views_grad(feats, pix, g, red)
            scale = float(fr.grad.abs().max())
            max_rel = float((ours - fr.grad).abs().max()) / scale
            # kernel breakdown of one backward call, in a profiler run of its own
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                lift_views_grad(feats, pix, g, red)
                torch.cuda.synchronize()
            kernels = {}
            for e in prof.key_averages():
                if e.device_type == torch.autograd.DeviceType.CUDA and getattr(e, "device_time_total", 0) > 0:
                    kernels[e.key[:90]] = round(e.device_time_total / 1e3, 4)
            run = {"V": V, "reduce": red, "forward_ms": fwd[0], "backward_ms": bwd[0], "backward_ms_min_max": bwd[1:],
                   "forward_plus_backward_through_autograd_ms": fwd_bwd[0], "backward_over_forward": bwd[0] / fwd[0],
                   "compulsory_bytes_per_scene": compulsory,
                   "backward_frac_hbm": B * compulsory / (bwd[0] * 1e-3) / (HBM_GBS * 1e9),
                   "sort_pairs_per_scene": pairs, "sort_bytes_per_scene_estimate": sort_bytes,
                   "backward_frac_hbm_with_sort_estimate": B * (compulsory + sort_bytes) / (bwd[0] * 1e-3) / (HBM_GBS * 1e9),
                   "reference_composition_backward_ms": float(np.median(ref_ms)),
                   "speedup_vs_reference_backward": float(np.median(ref_ms)) / bwd[0],
                   "max_rel_diff_vs_reference_backward": max_rel, "kernels_ms_one_call": kernels}
            print(json.dumps(run), flush=True)
            result["runs"].append(run)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
