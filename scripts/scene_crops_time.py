"""Training crops (pn2_b200/whole_scene.py SceneBank.crops) on synthetic rooms of 100 k - 400 k points, 5 - 12 m across
(scenes.scannet_room), beside the host loop they replace and the train step they feed.

    python scripts/scene_crops_time.py OUT.json

a  warm: a bank of the three rooms (22 MB, L2-resident); B crops all from one room, B = 8 and 32.  CUDA events around
   50 back-to-back calls after a warm-up, median of 5 such windows; plus one call checked against the oracle.
b  cold: a bank of 64 rooms of 100 k - 400 k points (about 0.5 GB, four times the 126 MB L2); B random room ids per call.
c  host: the training loader's numpy loop per crop (oracle/scene_crops_ref.py, the same loop with the hash in place of
   np.random.choice), host clock, 5 crops per room.
d  a GraphedTrainStep step (zero-grad + forward + backward + Adam, replayed) of PointNet2SemSeg and of the MSG stack at
   the same B on 8192-point crops: CUDA events around 20 replays after 3, median per step.
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
import torch.nn.functional as F  # noqa: E402

from oracle import scene_crops_ref  # noqa: E402
from pn2_b200 import scenes, whole_scene  # noqa: E402
from pn2_b200.models import GraphedTrainStep, PointNet2Multiview2Msg, PointNet2SemSeg  # noqa: E402

dev = torch.device("cuda:0")
C, NPOINTS = 21, 8192
ROOMS = [(0, 100_000, 5.0), (1, 200_000, 8.0), (2, 400_000, 12.0)]


def make_bank(rooms):
    xyz, rgb, lab = (np.concatenate([r[i] for r in rooms]) for i in range(3))
    offsets = np.concatenate([[0], np.cumsum([len(r[0]) for r in rooms])]).astype(np.int64)
    t = [torch.from_numpy(a).to(dev) for a in (xyz, rgb, lab, offsets)]
    return whole_scene.SceneBank(*t), (xyz, rgb, lab, offsets)


def event_ms(fn, calls, windows=5):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / calls)
    return float(np.median(out)), float(np.std(out))


def train_step_ms(model, b, crops):
    torch.manual_seed(0)
    net = (PointNet2Multiview2Msg(C) if model == "msg" else PointNet2SemSeg(C)).to(dev).train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)
    w = crops.weights.clone()

    def loss_fn(pred, tgt):
        return (F.cross_entropy(pred.reshape(-1, C), tgt.reshape(-1), ignore_index=0, reduction="none") * w.reshape(-1)).mean()
    xyz = crops.points[..., :3].permute(0, 2, 1).contiguous()
    feats = (torch.randn(b, 128, NPOINTS, device=dev) if model == "msg" else crops.points[..., 3:].permute(0, 2, 1).contiguous())
    stepper = GraphedTrainStep(net, opt, loss_fn, xyz, feats, crops.target)
    ms, sd = event_ms(lambda: stepper.step(xyz, feats, crops.target), 20, windows=3)
    del stepper, net, opt
    torch.cuda.empty_cache()
    return ms, sd


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "scene_crops_time.json"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "npoints": NPOINTS, "warm": [], "cold": [], "host": [],
           "train_step": []}
    rooms = [scenes.scannet_room(*r) for r in ROOMS]
    bank, packed = make_bank(rooms)
    lw = bank.label_weights(C)
    lw_host = lw.cpu().numpy()

    # a: warm, one room per batch
    for k, (_, n, ext) in enumerate(ROOMS):
        for b in (8, 32):
            ids = torch.full((b,), k, dtype=torch.int32, device=dev)
            bank.step.zero_()
            got = bank.crops(ids, lw, NPOINTS)
            want = scene_crops_ref.scene_crops(*packed, [k] * b, lw_host, NPOINTS, 0, 0)
            same = all(np.array_equal(getattr(got, f).cpu().numpy(), want[f]) for f in ("point_index", "points", "weights", "tries"))
            ms, sd = event_ms(lambda: bank.crops(ids, lw, NPOINTS), 50)
            res["warm"].append({"points": n, "extent_m": ext, "B": b, "crop_batch_ms": ms, "std_ms": sd,
                                "tries_mean": float(got.tries.float().mean()), "identical_to_oracle": same})

    # c: the host loop per crop
    for k, (_, n, ext) in enumerate(ROOMS):
        ts = []
        for rep in range(5):
            t0 = time.perf_counter()
            scene_crops_ref.scene_crops(*packed, [k], lw_host, NPOINTS, 0, rep)
            ts.append(time.perf_counter() - t0)
        res["host"].append({"points": n, "extent_m": ext, "host_ms_per_crop": 1e3 * float(np.median(ts)), "std_ms": 1e3 * float(np.std(ts))})

    # b: cold, a bank larger than L2, random rooms per call
    del bank
    big = [scenes.scannet_room(100 + i, 100_000 * (1 + i % 4), 5.0 + 2.3 * (i % 4)) for i in range(64)]
    bank_big, _ = make_bank(big)
    del big
    bank_bytes = sum(t.numel() * t.element_size() for t in (bank_big.xyz, bank_big.feats, bank_big.labels))
    g = torch.Generator(device="cpu").manual_seed(0)
    for b in (8, 32):
        pool = [torch.randint(0, 64, (b,), generator=g, dtype=torch.int32).to(dev) for _ in range(16)]
        it = iter(range(1 << 30))
        ms, sd = event_ms(lambda: bank_big.crops(pool[next(it) % 16], lw, NPOINTS), 50)
        res["cold"].append({"bank_rooms": 64, "bank_MB": bank_bytes / 2 ** 20, "B": b, "crop_batch_ms": ms, "std_ms": sd})

    # d: the train step at the same B, from crops of the warm bank
    bank, _ = make_bank(rooms)
    for b in (8, 32):
        crops = bank.crops(torch.arange(b, dtype=torch.int32, device=dev) % 3, lw, NPOINTS)
        for model in ("ssg", "msg"):
            ms, sd = train_step_ms(model, b, crops)
            res["train_step"].append({"model": "PointNet2SemSeg" if model == "ssg" else "MSG", "B": b, "graphed_step_ms": ms, "std_ms": sd})
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
