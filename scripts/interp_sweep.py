"""three_interpolate: the tiled kernels against the lane-along-channel kernel (pn2_debug_set_interp_mode), bit-equality
and HBM fraction per shape.  python scripts/interp_sweep.py"""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200"))
import numpy as np, torch
from pn2_b200 import _lib as L
if os.environ.get("PN2_LIB_PATH"):  # A/B runs against a second build of the library
    L.LIB_PATH = os.environ["PN2_LIB_PATH"]
from pn2_b200 import pointnet2_utils as pu
dev = torch.device("cuda:0")
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
_pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
PEAK = json.load(open(_pk))["hbm_gbs"] if os.path.exists(_pk) else 6650.0  # fallback: B200_PROFILING.md
lib = L.load()


def t_ms(fn, iters=9):
    for _ in range(3): fn()
    ts = []
    for _ in range(iters):
        flush.zero_(); a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
    return float(np.median(ts))


g = torch.Generator(device=dev).manual_seed(0)
SHAPES = [(32, 128, 1024, 8192)] if len(sys.argv) > 1 else [(32, 128, 1024, 8192), (64, 128, 2048, 8192), (64, 128, 4096, 16384), (16, 256, 256, 1024), (64, 128, 1024, 4096),
          (32, 256, 64, 256), (32, 128, 256, 1024), (8, 128, 1024, 8192), (2, 128, 1024, 8192),
          (3, 100, 1023, 8188), (5, 37, 700, 4100), (2, 128, 1, 512), (4, 64, 1500, 30000),
          (32, 128, 8192, 32768), (16, 64, 12000, 48000), (16, 128, 2048, 34720)]
MODES = [32, 32 | 256]  # the lane-along-channel kernel at 512 / 256 threads per CTA
for (B, C, m, n) in SHAPES:
    f = torch.randn(B, C, m, device=dev)
    idx = torch.randint(0, m, (B, n, 3), device=dev, dtype=torch.int32, generator=g)
    w = torch.rand(B, n, 3, device=dev); w = (w / w.sum(-1, keepdim=True)).contiguous()
    byts = B * (24 * n + 4 * C * m + 4 * C * n)
    lib.pn2_debug_set_interp_mode(1)
    want = pu.three_interpolate(f, idx, w)
    ms = t_ms(lambda: pu.three_interpolate(f, idx, w))
    row = {"shape": [B, C, m, n], "tiled_ms": round(ms, 4), "tiled_frac": round(byts / ms / 1e6 / PEAK, 3)}
    for mode in MODES:
        lib.pn2_debug_set_interp_mode(mode)
        got = pu.three_interpolate(f, idx, w)
        torch.cuda.synchronize()
        same = bool(torch.equal(got, want))
        ms = t_ms(lambda: pu.three_interpolate(f, idx, w))
        row["m%d" % mode] = [round(ms, 4), round(byts / ms / 1e6 / PEAK, 3), same]
    lib.pn2_debug_set_interp_mode(0)
    ms = t_ms(lambda: pu.three_interpolate(f, idx, w))
    row["auto"] = [round(ms, 4), round(byts / ms / 1e6 / PEAK, 3), bool(torch.equal(pu.three_interpolate(f, idx, w), want))]
    print(json.dumps(row), flush=True)
