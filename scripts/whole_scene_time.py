"""Whole-scene evaluation and labelling (pn2_b200/whole_scene.py) on synthetic rooms of 100 k - 400 k points, 5 - 12 m
across (scenes.scannet_room).

    python scripts/whole_scene_time.py OUT.json

a  block tiling: the host loop of the whole-scene loader (oracle/whole_scene_ref.scene_blocks, numpy, the same blocks)
   against scene_blocks on the device, alternating per room; host clock around work that ends in a device synchronise
b  evaluation end to end, scenes/s: scene_blocks + predict() in groups of 32 blocks + EvalCounters.update, per room
c  labelling end to end, scenes/s: segment_scene (scene_chunks + predict() in groups of 32 chunks + votes + arg-max)
b and c run under both set_mlp_precision settings, alternating, after a warm-up pass over every room.  Inputs start on
the device; the times include the one 40-byte read-back per pass.
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import whole_scene_ref  # noqa: E402
from pn2_b200 import pc_util, scenes, whole_scene  # noqa: E402
from pn2_b200.models import PointNet2SemSeg  # noqa: E402
from pn2_b200.pointnet_util import set_mlp_precision  # noqa: E402

dev = torch.device("cuda:0")
C = 21
ROOMS = [(0, 100_000, 5.0), (1, 200_000, 7.0), (2, 300_000, 9.5), (3, 400_000, 12.0)]
LABELWEIGHTS = (1.0 + np.arange(C) / 7.0).astype(np.float32) ** 1.5


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def evaluate(net, room):
    xyz, rgb, labels = room["dev"]
    blocks = whole_scene.scene_blocks(xyz, rgb, labels, room["lw"], seed=0)
    ctr = pc_util.EvalCounters(C, dev, res=0.02)
    with torch.no_grad():
        for s in range(0, blocks.points.shape[0], 32):
            pts = blocks.points[s:s + 32]
            x = pts.permute(0, 2, 1)
            ctr.update(pts, blocks.target[s:s + 32], net.predict(x[:, :3], x[:, 3:]), blocks.weights[s:s + 32])
    return blocks.points.shape[0]


def label(net, room):
    xyz, rgb, _ = room["dev"]
    labels, _ = whole_scene.segment_scene(net, xyz, rgb, batch=32)
    return labels


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "whole_scene_time.json"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    torch.manual_seed(0)
    net = PointNet2SemSeg(C).eval().to(dev)
    rooms = []
    for sid, n, ext in ROOMS:
        xyz, rgb, labels = scenes.scannet_room(sid, n, ext)
        rooms.append({"id": sid, "n": n, "extent": ext, "host": (xyz, rgb, labels),
                      "dev": (torch.from_numpy(xyz).to(dev), torch.from_numpy(rgb).to(dev), torch.from_numpy(labels).to(dev)),
                      "lw": torch.from_numpy(LABELWEIGHTS).to(dev)})
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "rooms": [], "reps": 5}

    # a: tiling only, host loop vs device
    for room in rooms:
        xyz, rgb, labels = room["host"]
        d_xyz, d_rgb, d_lab = room["dev"]
        whole_scene.scene_blocks(d_xyz, d_rgb, d_lab, room["lw"])  # warm-up
        host, device = [], []
        for _ in range(res["reps"]):
            t, want = timed(lambda: whole_scene_ref.scene_blocks(xyz, rgb, labels, LABELWEIGHTS, 8192, 0))
            host.append(t)
            t, got = timed(lambda: whole_scene.scene_blocks(d_xyz, d_rgb, d_lab, room["lw"]))
            device.append(t)
        same = bool(np.array_equal(got.points.cpu().numpy(), want["points"]) and np.array_equal(got.weights.cpu().numpy(), want["weights"]))
        room["blocks"] = int(got.points.shape[0])
        res["rooms"].append({"points": room["n"], "extent_m": room["extent"], "kept_blocks": room["blocks"],
                             "host_tiling_ms": 1e3 * float(np.median(host)), "device_tiling_ms": 1e3 * float(np.median(device)),
                             "host_tiling_std_ms": 1e3 * float(np.std(host)), "device_tiling_std_ms": 1e3 * float(np.std(device)),
                             "tiling_speedup": float(np.median(host) / np.median(device)), "identical_to_host": same})

    # b, c: end to end under both precisions (warm-up pass first)
    e2e = {}
    for precision in ("fp32", "bf16"):
        set_mlp_precision(precision)
        for room in rooms:
            evaluate(net, room)
            label(net, room)
    reps = 3
    times = {(p, k): [] for p in ("fp32", "bf16") for k in ("eval", "label")}
    chunks = {}
    for _ in range(reps):
        for precision in ("fp32", "bf16"):
            set_mlp_precision(precision)
            t, _ = timed(lambda: [evaluate(net, r) for r in rooms])
            times[(precision, "eval")].append(t)
            t, _ = timed(lambda: [label(net, r) for r in rooms])
            times[(precision, "label")].append(t)
    set_mlp_precision("fp32")
    for r in rooms:
        chunks[r["n"]] = int(whole_scene.scene_chunks(*r["dev"][:2])[2].shape[0])
    for (precision, kind), ts in times.items():
        e2e["%s_%s" % (kind, precision)] = {"scenes_per_s": len(rooms) / float(np.median(ts)), "ms_per_pass_of_4_rooms": 1e3 * float(np.median(ts)),
                                            "std_ms": 1e3 * float(np.std(ts))}
    res["end_to_end"] = e2e
    res["chunks_per_room"] = chunks
    res["blocks_per_room"] = {r["n"]: r["blocks"] for r in rooms}
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
