"""FPS round time per kernel policy: mode 1 = one 256-thread CTA per cloud (spatial slabs per warp with skipped rounds
above 4096 points, the index-interleaved kernel up to 4096), 2 = 4-CTA cluster with DSMEM exchange.  CUDA events, L2
flushed, median of 7."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200"))
import numpy as np, torch
from pn2_b200 import _lib, scenes
from pn2_b200.pointnet_util import fps_gather_cl
dev = torch.device("cuda:0")
lib = _lib.load()
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
for (N, M) in ((8192, 1024), (4096, 1024), (2048, 512), (1024, 256)):
    xyz = torch.from_numpy(np.stack([scenes.scannet_scene(10 + b, N)[0] for b in range(B)])).to(dev)
    row = {"B": B, "N": N, "M": M}
    for mode in (1, 2):
        lib.pn2_debug_set_fps_mode(mode)
        for _ in range(2):
            fps_gather_cl(xyz, M)
        ts = []
        for _ in range(7):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fps_gather_cl(xyz, M); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ms = float(np.median(ts))
        row["mode%d_ms" % mode] = round(ms, 4)
        row["mode%d_us_per_round" % mode] = round(ms * 1e3 / (M - 1), 4)
    lib.pn2_debug_set_fps_mode(0)
    print(json.dumps(row))
