"""Training-mode SA / FP blocks: the block Functions (train_mlp.sa_scale_train / fp_block_train) against the composition
they replaced (grouping / interpolation -> fused_mlp_train -> max), alternating in one process.

    python scripts/train_block_time.py OUT.json

Times, on the MSG multi-view network (PointNet2Multiview2Msg, 8192 points per scene):
  * forward + backward of every SA / FP module at 4 and 8 scenes, on the inputs it receives in the network;
  * the GraphedTrainStep step (forward + backward + Adam replayed as one CUDA graph) at 4 scenes;
  * the kernels one eager step issues (torch.profiler).
The replaced path is selected by switching pointnet_util._train_blocks off (a developer hook of this script only)."""
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

from pn2_b200 import pointnet_util, scenes  # noqa: E402
from pn2_b200.models import GraphedTrainStep, PointNet2Multiview2Msg  # noqa: E402

dev = torch.device("cuda:0")
N = 8192
_BLOCKS = pointnet_util._train_blocks


def use(new):
    pointnet_util._train_blocks = _BLOCKS if new else (lambda *a, **k: False)


def inputs(B, seed):
    pts = torch.from_numpy(scenes.scannet_batch(seed, B, N)).to(dev)
    xyz = pts[:, :, :3].permute(0, 2, 1).contiguous()
    img = torch.randn(B, 128, N, device=dev, generator=torch.Generator(device=dev).manual_seed(seed))
    target = (pts[:, :, 2].clamp(0, 2.69) / 2.7 * 20).long() + 1
    return xyz, img, target


def make():
    torch.manual_seed(0)
    net = PointNet2Multiview2Msg(21).to(dev).train()
    for m in net.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    return net, torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)


def loss_fn(logits, tgt):
    return F.cross_entropy(logits.reshape(-1, 21), tgt.reshape(-1), ignore_index=0)


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


def block_times(B, reps=20):
    net, _ = make()
    xyz, img, _ = inputs(B, 11)
    feat_pos = {pointnet_util.PointNetSetAbstraction: (1,), pointnet_util.PointNetSetAbstractionMsg: (1,),
                pointnet_util.PointNetFeaturePropagation: (2, 3)}
    captured = []

    def hook(mod, args, kwargs):
        captured.append((mod, args, kwargs))

    hs = [(name, m, m.register_forward_pre_hook(hook, with_kwargs=True)) for name, m in net.named_modules() if type(m) in feat_pos]
    names = {id(m): name for name, m, _ in hs}
    with torch.no_grad():
        net(xyz, img)
    for _, _, h in hs:
        h.remove()
    rows = []
    for mod, args, kwargs in captured:
        fp = feat_pos[type(mod)]
        args = [a.detach().requires_grad_(i in fp) if torch.is_tensor(a) and a.is_floating_point() else a for i, a in enumerate(args)]
        out = mod(*args, **kwargs)
        out = out[1] if isinstance(out, tuple) else out
        g = torch.randn_like(out)

        def fwd_bwd(new):
            def run():
                use(new)
                o = mod(*args, **kwargs)
                o = o[1] if isinstance(o, tuple) else o
                o.backward(g)
                for a in args:
                    if torch.is_tensor(a):
                        a.grad = None
            return run

        for f in (fwd_bwd(False), fwd_bwd(True)):
            f(); f()  # warm-up
        (old, new), (sd_old, sd_new) = events_ms([fwd_bwd(False), fwd_bwd(True)], reps)
        rows.append({"module": names[id(mod)], "type": type(mod).__name__, "old_ms": old, "new_ms": new, "old_std": sd_old,
                     "new_std": sd_new, "speedup": old / new})
    use(True)
    return rows


def kernel_count(new, B=4):
    from torch.profiler import ProfilerActivity, profile
    use(new)
    net, opt = make()
    xyz, img, target = inputs(B, 12)

    def step():
        opt.zero_grad(set_to_none=True)
        loss_fn(net(xyz, img), target).backward()
        opt.step()
    step(); step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kern = [n for n in names if not n.startswith("Memcpy") and not n.startswith("Memset")]
    torch_kern = [n for n in kern if "at::" in n]
    use(True)
    return {"kernels": len(kern), "torch_kernels": len(torch_kern)}


def graphed_times(B=4, reps=30):
    xyz, img, target = inputs(B, 13)
    steppers = []
    for new in (False, True):
        use(new)
        net, opt = make()
        steppers.append(GraphedTrainStep(net, opt, loss_fn, xyz, img, target))
    use(True)
    fns = [lambda s=s: s.step(xyz, img, target) for s in steppers]
    for f in fns:
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    (old, new), (sd_old, sd_new) = events_ms(fns, reps)
    losses = [float(s.step(xyz, img, target)) for s in steppers]
    return {"scenes": B, "old_ms": old, "new_ms": new, "old_std": sd_old, "new_std": sd_new, "speedup": old / new,
            "last_loss_old": losses[0], "last_loss_new": losses[1]}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "train_block_time.json"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "points_per_scene": N,
           "blocks": {str(B): block_times(B) for B in (4, 8)},
           "graphed_step": [graphed_times(4), graphed_times(4)],
           "eager_step_kernels": {"old": kernel_count(False), "new": kernel_count(True)}}
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "graphed_step": res["graphed_step"], "eager_step_kernels": res["eager_step_kernels"]}))
    for B, rows in res["blocks"].items():
        for r in rows:
            print(B, r["module"], r["type"], "%.3f -> %.3f ms" % (r["old_ms"], r["new_ms"]))


if __name__ == "__main__":
    main()
