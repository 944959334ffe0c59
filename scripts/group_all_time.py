"""group_all SA layer: the fused path (pn2_sa_all_mlp_max in eval, train_mlp.sa_all_train in training) against the
composition it replaced (sample_and_group_all -> cuDNN conv / BatchNorm / ReLU -> max in eval; sample_and_group_all ->
fused_mlp_train -> max(dim=2) in training), alternating in one process.

    python scripts/group_all_time.py OUT.json

Shapes (clouds x points, feature channels D, MLP):
  a  32 x 128,  D = 256, [256, 512, 1024]   the classification head's last SA layer
  b  32 x 512,  D = 5,   [32, 64]           the golden unit case, batched
  c  8 x 8192,  D = 64,  [64, 128]          many row tiles per cloud
Times are medians of CUDA-event windows after warm-up; every input fits the 126 MB L2, so these are warm-cache times.
The replaced path is selected by switching PointNetSetAbstraction._fused_ok / pointnet_util._train_blocks off (a developer
hook of this script only).  The eval composition runs cuDNN with its default TF32 setting, as the module did."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from pn2_b200 import pointnet_util  # noqa: E402
from pn2_b200.pointnet_util import PointNetSetAbstraction  # noqa: E402

dev = torch.device("cuda:0")
SHAPES = {"a": (32, 128, 256, [256, 512, 1024]), "b": (32, 512, 5, [32, 64]), "c": (8, 8192, 64, [64, 128])}
_FUSED_OK = PointNetSetAbstraction._fused_ok
_BLOCKS = pointnet_util._train_blocks


def use(new):
    PointNetSetAbstraction._fused_ok = _FUSED_OK if new else (lambda *a, **k: False)
    pointnet_util._train_blocks = _BLOCKS if new else (lambda *a, **k: False)


def events_ms(fns, reps):
    """Median ms of each fn over `reps` rounds, the fns alternating inside every round."""
    times = [[] for _ in fns]
    for _ in range(reps):
        for i, fn in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[i].append(a.elapsed_time(b))
    return [float(np.median(t)) for t in times], [float(np.std(t)) for t in times]


def shape_times(key, reps=50):
    B, N, D, mlp = SHAPES[key]
    torch.manual_seed(0)
    mod = PointNetSetAbstraction(None, None, None, 3 + D, mlp, True).to(dev)
    g = torch.Generator(device=dev).manual_seed(1)
    xyz = torch.randn(B, 3, N, device=dev, generator=g)
    feat_cl = torch.randn(B, N, D, device=dev, generator=g)
    gout = torch.randn(B, 1, mlp[-1], device=dev, generator=g).permute(0, 2, 1)

    def eval_fn(new):
        def run():
            use(new)
            with torch.no_grad():
                return mod(xyz, feat_cl.permute(0, 2, 1))[1]
        return run

    def train_fn(new):
        f = feat_cl.clone().requires_grad_(True)

        def run():
            use(new)
            for t in [f] + list(mod.parameters()):
                t.grad = None
            out = mod(xyz, f.permute(0, 2, 1))[1]
            out.backward(gout)
            return out, f.grad
        return run

    row = {"clouds": B, "points": N, "D": D, "mlp": mlp}
    mod.eval()
    ev = [eval_fn(False), eval_fn(True)]
    outs = [f() for f in ev]
    row["eval_rel_diff_new_vs_old"] = float((outs[1] - outs[0]).abs().max() / outs[0].abs().max())
    for f in ev:
        for _ in range(5):
            f()
    (old, new), (sd_old, sd_new) = events_ms(ev, reps)
    row.update(eval_old_ms=old, eval_new_ms=new, eval_old_std=sd_old, eval_new_std=sd_new, eval_speedup=old / new)
    mod.train()
    tr = [train_fn(False), train_fn(True)]
    (o0, g0), (o1, g1) = [(o.detach(), g) for o, g in (f() for f in tr)]
    row["train_out_rel_diff"] = float((o1 - o0).abs().max() / o0.abs().max())
    row["train_feat_grad_rel_diff"] = float((g1 - g0).abs().max() / g0.abs().max())
    for f in tr:
        for _ in range(5):
            f()
    (old, new), (sd_old, sd_new) = events_ms(tr, reps)
    row.update(train_old_ms=old, train_new_ms=new, train_old_std=sd_old, train_new_std=sd_new, train_speedup=old / new)
    use(True)
    return row


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "group_all_time.json"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0),
           "cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32),
           "shapes": {k: shape_times(k) for k in SHAPES}}
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(res["gpu"])
    for k, r in res["shapes"].items():
        print("%s  %d x %d, D=%d, %s: eval %.3f -> %.3f ms, train fwd+bwd %.3f -> %.3f ms, eval diff %.1e" % (
            k, r["clouds"], r["points"], r["D"], r["mlp"], r["eval_old_ms"], r["eval_new_ms"], r["train_old_ms"],
            r["train_new_ms"], r["eval_rel_diff_new_vs_old"]))


if __name__ == "__main__":
    main()
