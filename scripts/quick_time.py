"""Developer timing of the individual kernels and the whole forward (CUDA events, warm-up, L2 flush)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200"))
import numpy as np
import torch

from pn2_b200 import pointnet2_utils as pu
from pn2_b200 import scenes
from pn2_b200.models import PointNet2SemSeg
from pn2_b200.pointnet_util import fps_gather_cl, three_nn_weights_cl

dev = torch.device("cuda:0")
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
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
    return float(np.median(ts)), float(np.min(ts))


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
    N = 8192
    pts = torch.from_numpy(scenes.scannet_batch(0, B, N)).to(dev)
    xyz = pts[:, :, :3].contiguous()
    print("B=%d N=%d" % (B, N))
    for (n, m) in [(8192, 1024), (1024, 256), (256, 64), (64, 16)]:
        x = xyz[:, :n].contiguous()
        print("fps %d->%d: med %.3f ms min %.3f" % ((n, m) + timeit(lambda: fps_gather_cl(x, m))))
    from pn2_b200 import _lib as L
    for mode in (1, 2):
        L.load().pn2_debug_set_fps_mode(mode)
        print("fps 8192->1024 mode %d: med %.3f ms min %.3f" % ((mode,) + timeit(lambda: fps_gather_cl(xyz, 1024))))
        x4, x2 = xyz[:, :4096].contiguous(), xyz[:, :2048].contiguous()
        print("fps 4096->512 mode %d: med %.3f ms min %.3f" % ((mode,) + timeit(lambda: fps_gather_cl(x4, 512))))
        print("fps 2048->512 mode %d: med %.3f ms min %.3f" % ((mode,) + timeit(lambda: fps_gather_cl(x2, 512))))
    L.load().pn2_debug_set_fps_mode(0)
    idx, new_xyz = fps_gather_cl(xyz, 1024)
    print("ball_query r=.1: med %.3f min %.3f" % timeit(lambda: pu.ball_query(0.1, 32, xyz, new_xyz)))
    print("three_nn_w 8192x1024: med %.3f min %.3f" % timeit(lambda: three_nn_weights_cl(xyz, new_xyz)))
    feats = torch.randn(B, 128, 1024, device=dev)
    i3, w3 = three_nn_weights_cl(xyz, new_xyz)
    t = timeit(lambda: pu.three_interpolate(feats, i3, w3))
    byts = B * (24 * N + 4 * 128 * 1024 + 4 * 128 * N)
    print("three_interpolate C=128: med %.3f min %.3f -> %.0f GB/s" % (t + (byts / t[0] / 1e6,)))
    bq = pu.ball_query(0.1, 32, xyz, new_xyz)
    f64 = torch.randn(B, 64, N, device=dev)
    t = timeit(lambda: pu.grouping_operation(f64, bq))
    byts = B * (4 * 1024 * 32 + 4 * 64 * min(N, 1024 * 32) + 4 * 64 * 1024 * 32)
    print("group C=64: med %.3f min %.3f -> %.0f GB/s" % (t + (byts / t[0] / 1e6,)))
    model = PointNet2SemSeg(21).eval().to(dev)
    x6 = pts.permute(0, 2, 1).contiguous()
    with torch.no_grad():
        t = timeit(lambda: model(x6[:, :3], x6[:, 3:]))
    print("semseg forward: med %.3f ms min %.3f -> %.0f scenes/s" % (t + (B / t[0] * 1e3,)))
    from pn2_b200.models import GraphedForward
    g = GraphedForward(model, x6[:, :3].contiguous(), x6[:, 3:].contiguous())
    xa, xb = x6[:, :3].contiguous(), x6[:, 3:].contiguous()
    t = timeit(lambda: g.run(xa, xb))
    print("semseg forward (CUDA graph): med %.3f ms min %.3f -> %.0f scenes/s" % (t + (B / t[0] * 1e3,)))
    with torch.no_grad():
        ref = model(x6[:, :3], x6[:, 3:])
    print("graph vs eager max diff", (g.run(xa, xb) - ref).abs().max().item())
    # per-stage breakdown
    from pn2_b200.pointnet_util import to_channel_last
    with torch.no_grad():
        xyz_cl, feat_cl = to_channel_last(x6[:, :3]), to_channel_last(x6[:, 3:])
        stages = []
        l1_xyz, l1 = model.sa1.forward_cl(xyz_cl, feat_cl)
        l2_xyz, l2 = model.sa2.forward_cl(l1_xyz, l1)
        l3_xyz, l3 = model.sa3.forward_cl(l2_xyz, l2)
        l4_xyz, l4 = model.sa4.forward_cl(l3_xyz, l3)
        from pn2_b200.pointnet_util import sa_mlp_max_cl
        from pn2_b200 import _lib
        for name, mod, x, f, nx in [("sa1", model.sa1, xyz_cl, feat_cl, l1_xyz), ("sa2", model.sa2, l1_xyz, l1, l2_xyz),
                                    ("sa3", model.sa3, l2_xyz, l2, l3_xyz), ("sa4", model.sa4, l3_xyz, l3, l4_xyz)]:
            bqi = pu.ball_query(mod.radius, mod.nsample, x, nx)
            t = timeit(lambda: sa_mlp_max_cl(x, f, nx, bqi, _lib.ORDER_XYZ_FIRST, mod.folded()))
            print("  %s fused mlp: med %.3f min %.3f" % ((name,) + t))
        l3n = model.fp4.forward_cl(l3_xyz, l4_xyz, l3, l4)
        l2n = model.fp3.forward_cl(l2_xyz, l3_xyz, l2, l3n)
        l1n = model.fp2.forward_cl(l1_xyz, l2_xyz, l1, l2n)
        for name, fn in [("fp4", lambda: model.fp4.forward_cl(l3_xyz, l4_xyz, l3, l4)),
                         ("fp3", lambda: model.fp3.forward_cl(l2_xyz, l3_xyz, l2, l3n)),
                         ("fp2", lambda: model.fp2.forward_cl(l1_xyz, l2_xyz, l1, l2n)),
                         ("fp1+head", lambda: model.fp1.forward_cl(xyz_cl, l1_xyz, feat_cl, l1n, mlp=model._fp1_with_head()))]:
            print("  %s (3nn + fused mlp): med %.3f min %.3f" % ((name,) + timeit(fn)))


if __name__ == "__main__":
    main()
