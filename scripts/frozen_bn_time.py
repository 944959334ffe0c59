"""Running-statistics BatchNorm on the fused training kernels (eval() under autograd, frozen-BatchNorm fine-tuning) against
the path these calls took before: the reference's composition on torch conv / BatchNorm (cuDNN, its default TF32
setting), which set_fused_training(False) still selects.  Both alternate in one process.

    python scripts/frozen_bn_time.py OUT.json

Times (medians of CUDA-event windows after warm-up):
  a  PointNet2SemSeg, 8 x 8192 points, net.eval(): forward + backward of a loss
  b  PointNet2Multiview2Msg (the MSG stack), 4 x 8192 points, net.train() with every BatchNorm in eval: eager forward +
     backward, and the GraphedTrainStep step (forward + backward + Adam replayed as one CUDA graph; each path is captured
     under its own setting)
Beside the times: the largest difference between the two paths' outputs and input-feature gradients, relative to the
largest value, and the relative L2 difference of the gradients; once with the composition in its default TF32 and once
with TF32 off, which separates the composition's TF32 rounding from any difference of the new path.  (A max-pool routes
its whole gradient to one sample, so a TF32 perturbation that changes the winner moves an O(1) gradient to another
point.)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from pn2_b200 import scenes  # noqa: E402
from pn2_b200.models import GraphedTrainStep, PointNet2Multiview2Msg, PointNet2SemSeg  # noqa: E402
from pn2_b200.pointnet_util import set_fused_training  # noqa: E402

dev = torch.device("cuda:0")
N = 8192


def events_ms(fns, reps):
    """Median and standard deviation (ms) of each fn over `reps` rounds, the fns alternating inside every round."""
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


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max())


def rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def tf32(on):
    torch.backends.cudnn.allow_tf32 = on
    torch.backends.cuda.matmul.allow_tf32 = on


def inputs(B, seed, width):
    pts = torch.from_numpy(scenes.scannet_batch(seed, B, N)).to(dev)
    xyz = pts[:, :, :3].permute(0, 2, 1).contiguous()
    if width == 3:
        feat = pts[:, :, 3:].permute(0, 2, 1).contiguous()
    else:
        feat = torch.randn(B, width, N, device=dev, generator=torch.Generator(device=dev).manual_seed(seed))
    target = (pts[:, :, 2].clamp(0, 2.69) / 2.7 * 20).long() + 1
    return xyz, feat, target


def loss_fn(logits, tgt):
    return F.cross_entropy(logits.reshape(-1, 21), tgt.reshape(-1), ignore_index=0)


def frozen(net):
    net.train()
    for m in net.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            m.eval()
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    return net


def eager_fns(net, xyz, feat, target):
    f = feat.clone().requires_grad_(True)

    def fn(new):
        def run():
            set_fused_training(new)
            net.zero_grad(set_to_none=True)
            f.grad = None
            out = net(xyz, f)
            loss_fn(out, target).backward()
            return out.detach(), f.grad
        return run
    return [fn(False), fn(True)]


def compare_and_time(fns, reps):
    row = {}
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    for tag, on in (("", True), ("_tf32_off", False)):
        tf32(on)
        (o0, g0), (o1, g1) = [fn() for fn in fns]
        row.update({"out_rel_diff_new_vs_old" + tag: rel(o1, o0), "feat_grad_rel_diff_new_vs_old" + tag: rel(g1, g0),
                    "feat_grad_rel_l2_diff_new_vs_old" + tag: rel_l2(g1, g0)})
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    for fn in fns:
        for _ in range(3):
            fn()
    (old, new), (sd_old, sd_new) = events_ms(fns, reps)
    row.update(old_ms=old, new_ms=new, old_std=sd_old, new_std=sd_new, speedup=old / new)
    return row


def semseg_eval(reps=20):
    torch.manual_seed(0)
    net = PointNet2SemSeg(21).to(dev).eval()
    xyz, rgb, target = inputs(8, 1, 3)
    row = {"model": "PointNet2SemSeg", "scenes": 8, "points": N, "mode": "net.eval(), forward + backward"}
    row.update(compare_and_time(eager_fns(net, xyz, rgb, target), reps))
    return row


def msg_frozen_eager(reps=20):
    torch.manual_seed(0)
    net = frozen(PointNet2Multiview2Msg(21).to(dev))
    xyz, img, target = inputs(4, 2, 128)
    row = {"model": "PointNet2Multiview2Msg", "scenes": 4, "points": N, "mode": "frozen BatchNorm, eager forward + backward"}
    row.update(compare_and_time(eager_fns(net, xyz, img, target), reps))
    return row


def msg_frozen_graphed(reps=30):
    xyz, img, target = inputs(4, 2, 128)
    steppers = []
    for new in (False, True):
        set_fused_training(new)
        torch.manual_seed(0)
        net = frozen(PointNet2Multiview2Msg(21).to(dev))
        opt = torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)
        steppers.append(GraphedTrainStep(net, opt, loss_fn, xyz, img, target))
    set_fused_training(True)
    first = [float(s.step(xyz, img, target)) for s in steppers]
    fns = [lambda s=s: s.step(xyz, img, target) for s in steppers]
    for fn in fns:
        for _ in range(3):
            fn()
    (old, new), (sd_old, sd_new) = events_ms(fns, reps)
    return {"model": "PointNet2Multiview2Msg", "scenes": 4, "points": N, "mode": "frozen BatchNorm, GraphedTrainStep step",
            "first_loss_old": first[0], "first_loss_new": first[1], "old_ms": old, "new_ms": new, "old_std": sd_old,
            "new_std": sd_new, "speedup": old / new}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "frozen_bn_time.json"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    prev = set_fused_training(True)
    try:
        res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0),
               "cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32),
               "old_path": "set_fused_training(False): torch conv / BatchNorm composition",
               "a_semseg_eval": semseg_eval(), "b_msg_frozen_eager": msg_frozen_eager(),
               "b_msg_frozen_graphed": msg_frozen_graphed()}
    finally:
        set_fused_training(prev)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(res["gpu"])
    for k, r in res.items():
        if isinstance(r, dict):
            print("%s: %.3f -> %.3f ms (x%.3f, std %.3f / %.3f)%s" % (
                k, r["old_ms"], r["new_ms"], r["speedup"], r["old_std"], r["new_std"],
                ", out diff %.1e / %.1e (TF32 off), feat grad diff %.1e / %.1e, L2 %.1e / %.1e" % (
                    r["out_rel_diff_new_vs_old"], r["out_rel_diff_new_vs_old_tf32_off"], r["feat_grad_rel_diff_new_vs_old"],
                    r["feat_grad_rel_diff_new_vs_old_tf32_off"], r["feat_grad_rel_l2_diff_new_vs_old"],
                    r["feat_grad_rel_l2_diff_new_vs_old_tf32_off"])
                if "out_rel_diff_new_vs_old" in r else ""))


if __name__ == "__main__":
    main()
