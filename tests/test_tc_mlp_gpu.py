"""The tensor-core MLP kernel (csrc/row_mlp_tc.cu) against its bf16-exact reference (oracle/tc_mlp_ref.py).

launch_tc picks one of 11 kernel builds per launch (feature dtype, tiles per launch, CTAs per SM).  Small test batches
only ever reach the 8-worker builds, so every build is forced here through the developer knobs
(pn2_debug_set_tc_workers / pn2_debug_set_tc_max_ctas) and identified through pn2_debug_last_tc_launch.

Acceptance (oracle/tc_mlp_ref.agrees): (a) at most 1e-2 of the output elements differ from the reference by more than
1e-4 * max|ref|, and (b) max|diff| <= 1e-2 * max|ref| (the measurements behind the bounds are in oracle/tc_mlp_ref.py).  The reference rounds to bf16 where the kernel does, so only
fp32-versus-float64 accumulation separates them; (a) is what catches a wrong column, layout or rounding mode, which a
comparison with the fp32 modules at 2e-2 lets through.  The negative controls at the end plant such errors in the
reference and require the comparison to reject the kernel's real output.
"""
import ctypes
import math

import pytest
import torch

from oracle import tc_mlp_ref as ref
from pn2_b200 import _lib, pointnet_util, scenes
from pn2_b200.pointnet_util import FoldedMlp, fp_mlp_cl, sa_mlp_max_cl

pytestmark = pytest.mark.gpu

# forced configurations: (worker warps per tile, max CTAs per SM); "auto" = the production choice
CONFIGS = {"auto": (0, 8), "w8": (8, 8), "w8c1": (8, 1), "w4": (4, 8), "w4c3": (4, 3), "w4c2": (4, 2), "w4c1": (4, 1)}
MATRIX_CONFIGS = ["w8", "w4", "w4c3", "w4c2"]
BUILDS = ["f32_sa", "f32_fp", "f32_w8_sa", "f32_w8_fp", "bf16_sa", "bf16_fp", "bf16_wide_sa", "bf16_wide_fp",
          "bf16_x4_sa", "bf16_w8_sa", "bf16_w8_fp"]
SENTINEL = 12345.0


class Knobs:
    def __init__(self, lib):
        self.lib = lib

    def force(self, config):
        workers, ctas = CONFIGS[config]
        self.lib.pn2_debug_set_tc_workers(workers)
        self.lib.pn2_debug_set_tc_max_ctas(ctas)

    def last(self):
        """(build name, grid, threads) of the last tensor-core launch on this thread."""
        name, grid, threads = ctypes.c_char_p(), ctypes.c_int(), ctypes.c_int()
        ok = self.lib.pn2_debug_last_tc_launch(ctypes.byref(name), ctypes.byref(grid), ctypes.byref(threads))
        assert ok, "the call launched no tensor-core kernel"
        return name.value.decode(), grid.value, threads.value


@pytest.fixture
def tc(cuda):
    """bf16 precision and forced kernel builds, always restored: a failing case must not leak into later tests."""
    lib = _lib.load()
    prev = pointnet_util.set_mlp_precision("bf16")
    try:
        yield Knobs(lib)
    finally:
        lib.pn2_debug_set_tc_workers(0)
        lib.pn2_debug_set_tc_max_ctas(8)
        pointnet_util.set_mlp_precision(prev)


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def random_mlp(cin, widths, seed, dev, relu_last=True):
    g = torch.Generator().manual_seed(seed)
    layers, c = [], cin
    for i, w in enumerate(widths):
        W = torch.randn(w, c, generator=g) / math.sqrt(c)
        b = torch.randn(w, generator=g) * 0.2
        layers.append((W.to(dev), b.to(dev), relu_last or i + 1 < len(widths)))
        c = w
    mlp = FoldedMlp(layers)
    assert mlp.bf16_ok(), "widths %d -> %s do not fit the tensor-core kernel" % (cin, widths)
    return mlp


def features(t, kind):
    """kind: "f32" (16-byte aligned), "f32u" (fp32, base pointer 4 bytes off 16-byte alignment), "bf16"."""
    if t is None:
        return None
    if kind == "bf16":
        return t.to(torch.bfloat16)
    if kind == "f32u":
        buf = torch.empty(t.numel() + 1, device=t.device)
        u = buf[1:].view(t.shape)
        u.copy_(t)
        assert u.data_ptr() % 16 == 4
        return u
    return t.contiguous()


def check(got, want, label):
    frac, mx = ref.stats(got, want)
    print("%-44s frac>1e-4 %.2e  max %.2e" % (label, frac, mx))
    assert frac <= ref.FRAC_MAX and mx <= ref.MAX_REL, "%s: %.3e of the elements differ by > %g of the scale, max %.3e" % (
        label, frac, ref.FRAC_REL, mx)


def check_argmax(got, logits, label):
    """The fused arg-max output: equal to the reference's first arg-max wherever the reference's top two are not a
    near tie (within 1e-4 of the scale)."""
    scale = logits.abs().max().item()
    g = got.long()
    picked = logits.gather(-1, g.unsqueeze(-1)).squeeze(-1)
    short = logits.max(dim=-1).values - picked
    bad = (g != ref.first_argmax(logits)) & (short > ref.FRAC_REL * scale)
    print("%-44s arg-max mismatches %d of %d (near ties excluded)" % (label, int((g != ref.first_argmax(logits)).sum()), g.numel()))
    assert not bad.any(), "%s: %d rows pick a class clearly below the reference's maximum" % (label, int(bad.sum()))


# ---- SA -------------------------------------------------------------------------------------------------------------

def sa_inputs(B, N, M, K, D, seed, dev):
    g = torch.Generator().manual_seed(seed)
    xyz = torch.rand(B, N, 3, generator=g) * 3.0
    pick = torch.randint(0, N, (B, M), generator=g)
    new_xyz = torch.stack([xyz[b, pick[b]] for b in range(B)])
    # neighbours: mostly near the centre's index (a ball of a sorted-ish cloud), some anywhere
    idx = (pick[:, :, None] + torch.randint(-40, 40, (B, M, K), generator=g)).clamp(0, N - 1).to(torch.int32)
    feat = torch.randn(B, N, D, generator=g) if D else None
    return xyz.to(dev), (feat.to(dev) if feat is not None else None), new_xyz.to(dev), idx.to(dev)


def run_sa(tc, config, B, N, M, K, D, widths, order, feat_kind, out_kind, seed=0):
    dev = torch.device("cuda:0")
    xyz, feat, new_xyz, idx = sa_inputs(B, N, M, K, D, seed, dev)
    mlp = random_mlp(D + 3, widths, seed + 1, dev)
    f = features(feat, feat_kind)
    cout = widths[-1]
    tc.force(config)
    if out_kind == "slice":
        off = 7
        out = torch.full((B, M, off + cout + 5), SENTINEL, device=dev)
        sa_mlp_max_cl(xyz, f, new_xyz, idx, order, mlp, out=out, out_offset=off)
        got = out[..., off:off + cout]
    else:
        got = sa_mlp_max_cl(xyz, f, new_xyz, idx, order, mlp, out_dtype=torch.bfloat16 if out_kind == "bf16" else torch.float32)
    build = tc.last()
    torch.cuda.synchronize()
    if out_kind == "slice":
        assert (out[..., :off] == SENTINEL).all() and (out[..., off + cout:] == SENTINEL).all(), "channels outside the slice were written"
    want = ref.sa_ref(xyz, f, new_xyz, idx, order, mlp.layers, out_bf16=out_kind == "bf16")
    return got, want, build, (xyz, f, new_xyz, idx, mlp)


XF, FF = _lib.ORDER_XYZ_FIRST, _lib.ORDER_FEAT_FIRST
# id: B, N, M, K, D, widths, order, features, output
SA_MATRIX = {
    "k1_d64": (2, 500, 300, 1, 64, [64, 128], XF, "f32", "f32"),
    "k2_d13_featfirst": (2, 500, 200, 2, 13, [32, 64], FF, "f32", "f32"),
    "k8_d5_widths40_21": (1, 800, 100, 8, 5, [40, 21], XF, "f32", "f32"),
    "k32_d0_pooldup_outbf16": (2, 1000, 128, 32, 0, [32, 32, 64], XF, "f32", "bf16"),
    "k64_d3": (2, 500, 40, 64, 3, [64, 64, 128], XF, "f32", "f32"),
    "k64_d64_thin67_bf16": (2, 700, 90, 64, 64, [64, 64, 128], XF, "bf16", "bf16"),
    "k128_d128_thin131": (2, 900, 33, 128, 128, [128, 128, 256], XF, "f32", "f32"),
    "k16_d256_thin259_out512_bf16": (2, 400, 40, 16, 256, [256, 256, 512], XF, "bf16", "f32"),
    "k32_d128_hidden256": (2, 500, 40, 32, 128, [256, 256, 256], FF, "bf16", "bf16"),
    "k16_d13_six_layers": (2, 300, 70, 16, 13, [32, 64, 64, 128, 128, 64], FF, "f32", "f32"),
    "k8_m5_tile_spans_clouds_bf16": (4, 300, 5, 8, 64, [64, 64], XF, "bf16", "f32"),
    "k32_37groups_partial_tile": (1, 600, 37, 32, 3, [64, 64, 128], XF, "f32", "f32"),
    "k32_d64_misaligned_slice": (2, 600, 50, 32, 64, [64, 64, 128], FF, "f32u", "slice"),
    "k4_d64_featfirst_bf16_slice": (2, 400, 100, 4, 64, [64, 128], FF, "bf16", "slice"),
    "k64_d64_misaligned_thin67": (1, 700, 45, 64, 64, [64, 64, 128], XF, "f32u", "f32"),
}


@pytest.mark.parametrize("config", MATRIX_CONFIGS)
@pytest.mark.parametrize("case", list(SA_MATRIX))
def test_sa_matches_bf16_reference(tc, case, config):
    B, N, M, K, D, widths, order, fk, ok = SA_MATRIX[case]
    got, want, build, _ = run_sa(tc, config, B, N, M, K, D, widths, order, fk, ok, seed=len(case))
    check(got, want, "sa %s [%s -> %s]" % (case, config, build[0]))


# ---- FP -------------------------------------------------------------------------------------------------------------

def fp_inputs(B, n, m, D1, D2, seed, dev):
    g = torch.Generator().manual_seed(seed)
    feat1 = torch.randn(B, n, D1, generator=g) if D1 else None
    feat2 = torch.randn(B, m, D2, generator=g)
    idx = torch.randint(0, m, (B, n, 3), generator=g, dtype=torch.int32)
    w = torch.rand(B, n, 3, generator=g) + 0.05
    w = w / w.sum(-1, keepdim=True)
    return (feat1.to(dev) if feat1 is not None else None), feat2.to(dev), idx.to(dev), w.to(dev)


def run_fp(tc, config, B, n, m, D1, D2, widths, relu_last, f2_kind, f1_kind, out_kind, seed=0, row_order=None):
    dev = torch.device("cuda:0")
    feat1, feat2, idx, w = fp_inputs(B, n, m, D1, D2, seed, dev)
    mlp = random_mlp(D1 + D2, widths, seed + 1, dev, relu_last)
    f1, f2 = features(feat1, f1_kind), features(feat2, f2_kind)
    tc.force(config)
    dtype = {"f32": torch.float32, "bf16": torch.bfloat16, "argmax": torch.uint8}[out_kind]
    got = fp_mlp_cl(f1, f2, idx, w, mlp, n, row_order=row_order, out_dtype=dtype)
    build = tc.last()
    torch.cuda.synchronize()
    want = ref.fp_ref(f1, f2, idx, w, n, mlp.layers, out_bf16=out_kind == "bf16")
    return got, want, build, (f1, f2, idx, w, mlp)


# id: B, n, m, D1, D2, widths, ReLU on the last layer, feat2, feat1, output
FP_MATRIX = {
    "n1000_m250": (2, 1000, 250, 64, 128, [128, 128], True, "f32", "f32", "f32"),
    "n100_three_clouds_d1_3": (3, 100, 30, 3, 64, [64, 32], True, "f32", "f32", "f32"),
    "n100_three_clouds_bf16": (3, 100, 30, 16, 64, [64, 32], True, "bf16", "bf16", "bf16"),
    "m1_d1_0": (2, 300, 1, 0, 256, [256, 128], True, "f32", None, "f32"),
    "m1_bf16_skip16": (2, 300, 1, 16, 256, [128], True, "bf16", "bf16", "bf16"),
    "m2_d1_5": (2, 200, 2, 5, 40, [64], True, "f32", "f32", "f32"),
    "m3_d1_13_width21": (2, 260, 3, 13, 24, [32, 21], True, "f32", "f32", "f32"),
    "d2_1536_chunks": (1, 300, 64, 0, 1536, [256, 256], True, "f32", None, "f32"),
    "d2_1536_chunks_bf16": (1, 300, 64, 0, 1536, [256, 256], True, "bf16", None, "bf16"),
    "head5_skip6_f32": (2, 1000, 250, 6, 128, [128, 128, 128, 128, 21], False, "bf16", "f32", "f32"),
    "head5_argmax": (2, 1000, 250, 6, 128, [128, 128, 128, 128, 21], False, "bf16", "f32", "argmax"),
    "misaligned_d1_7": (2, 500, 100, 7, 128, [128, 64], True, "f32u", "f32", "f32"),
    "skip_bf16_out_bf16": (2, 700, 100, 64, 128, [128, 128], True, "bf16", "bf16", "bf16"),
    "n256_in_bf16_skip_f32": (2, 256, 64, 32, 64, [64], True, "bf16", "f32", "f32"),
}


@pytest.mark.parametrize("config", MATRIX_CONFIGS)
@pytest.mark.parametrize("case", list(FP_MATRIX))
def test_fp_matches_bf16_reference(tc, case, config):
    args = FP_MATRIX[case]
    got, want, build, _ = run_fp(tc, config, *args, seed=len(case))
    label = "fp %s [%s -> %s]" % (case, config, build[0])
    if args[-1] == "argmax":
        check_argmax(got, want, label)
    else:
        check(got, want, label)


# ---- every build, the persistent loop ---------------------------------------------------------------------------------

SA_BUILD_CASE = (2, 700, 300, 32, 64, [64, 64, 128], XF)   # cin 67: up to 4 CTAs/SM
FP_BUILD_CASE = (2, 1000, 250, 64, 128, [128, 128], True)  # up to 3 CTAs/SM with bf16 features
# build: (block, features, forced configuration)
EVERY_BUILD = {
    "f32_sa": ("sa", "f32", "w4"), "f32_fp": ("fp", "f32", "w4"),
    "f32_w8_sa": ("sa", "f32", "w8"), "f32_w8_fp": ("fp", "f32", "w8"),
    "bf16_x4_sa": ("sa", "bf16", "w4"), "bf16_sa": ("sa", "bf16", "w4c3"), "bf16_fp": ("fp", "bf16", "w4"),
    "bf16_wide_sa": ("sa", "bf16", "w4c2"), "bf16_wide_fp": ("fp", "bf16", "w4c2"),
    "bf16_w8_sa": ("sa", "bf16", "w8"), "bf16_w8_fp": ("fp", "bf16", "w8"),
}
assert sorted(EVERY_BUILD) == sorted(BUILDS)


@pytest.mark.parametrize("build", BUILDS)
def test_every_build_matches_bf16_reference(tc, build):
    block, fk, config = EVERY_BUILD[build]
    if block == "sa":
        got, want, ran, _ = run_sa(tc, config, *SA_BUILD_CASE, fk, "f32", seed=11)
    else:
        got, want, ran, _ = run_fp(tc, config, *FP_BUILD_CASE, fk, fk, "f32", seed=12)
    assert ran[0] == build, "forcing %s ran %s" % (config, ran[0])
    check(got, want, "build %s (grid %d x %d threads)" % ran)


@pytest.mark.parametrize("workers", ["w4c1", "w8c1"])
@pytest.mark.parametrize("fk", ["f32", "bf16"])
@pytest.mark.parametrize("block", ["sa", "fp"])
def test_persistent_loop_walks_three_and_four_tiles(tc, block, fk, workers):
    """One CTA per SM and ~3.3 tiles per CTA: some CTAs walk 3 tiles, others 4, so the weight ring and the mbarrier
    phases carry across an odd and an even number of tiles."""
    sms = sm_count()
    tiles = int(3.3 * sms)
    if block == "sa":
        K, B = 32, 4  # 4 groups per tile
        got, want, ran, _ = run_sa(tc, workers, B, 800, tiles, K, 64, [64, 64, 128], XF, fk, "f32", seed=21)
    else:
        B = 2
        n = (tiles * 128 - 50) // B
        got, want, ran, _ = run_fp(tc, workers, B, n, 200, 16, 64, [128, 64], True, fk, fk, "f32", seed=22)
    assert ran[1] == sms, "expected one CTA per SM, grid %d" % ran[1]
    check(got, want, "persistent %s %s [%s -> %s, %d tiles / %d CTAs]" % (block, fk, workers, ran[0], tiles, ran[1]))


# ---- bit equality ---------------------------------------------------------------------------------------------------

def test_sa_is_bit_identical_across_builds_and_feature_dtypes(tc):
    """pn2_abi.h: the worker count does not change results, and bf16 features give what the same values as fp32 give."""
    dev = torch.device("cuda:0")
    xyz, feat, new_xyz, idx = sa_inputs(2, 700, 300, 32, 64, 31, dev)
    mlp = random_mlp(67, [64, 64, 128], 32, dev)
    fb = feat.to(torch.bfloat16)
    outs = {}
    for fk, f in (("bf16", fb), ("f32", fb.float()), ("f32u", features(fb.float(), "f32u"))):
        for config in ("w8", "w8c1", "w4", "w4c3", "w4c2", "w4c1"):
            tc.force(config)
            out = sa_mlp_max_cl(xyz, f, new_xyz, idx, XF, mlp)
            outs["%s %s/%s" % (fk, config, tc.last()[0])] = out
    first_key = next(iter(outs))
    for key, out in outs.items():
        assert torch.equal(out, outs[first_key]), "%s differs from %s" % (key, first_key)
    print("sa bit-identical over:", ", ".join(outs))


@pytest.mark.parametrize("fk", ["f32", "bf16"])
def test_fp_is_bit_identical_across_builds_and_row_orders(tc, fk):
    dev = torch.device("cuda:0")
    B, n = 2, 1000
    feat1, feat2, idx, w = fp_inputs(B, n, 250, 64, 128, 41, dev)
    f1, f2 = features(feat1, fk), features(feat2, fk)
    mlp = random_mlp(192, [128, 128], 42, dev)
    g = torch.Generator().manual_seed(43)
    perm = torch.stack([torch.randperm(n, generator=g) for _ in range(B)]).to(torch.int32).to(dev)
    outs = {}
    for config in ("w8", "w8c1", "w4", "w4c2", "w4c1"):
        for po in (None, perm):
            tc.force(config)
            out = fp_mlp_cl(f1, f2, idx, w, mlp, n, row_order=po)
            outs["%s/%s%s" % (config, tc.last()[0], " row_perm" if po is not None else "")] = out
    first_key = next(iter(outs))
    check(outs[first_key], ref.fp_ref(f1, f2, idx, w, n, mlp.layers), "fp bit-identity case %s" % fk)
    for key, out in outs.items():
        assert torch.equal(out, outs[first_key]), "%s differs from %s" % (key, first_key)
    print("fp bit-identical over:", ", ".join(outs))


@pytest.mark.parametrize("later", ["w4c1", "w8c1", "w4c2"])
def test_weights_packed_under_one_cta_cap_serve_launches_under_another(tc, later):
    """FoldedMlp packs its weights once.  The weight-tile height of the packed image used to be chosen with the
    pn2_debug_set_tc_max_ctas cap applied, so a launch under another cap read the image with the wrong tile layout."""
    dev = torch.device("cuda:0")
    feat1, feat2, idx, w = fp_inputs(2, 1000, 250, 64, 128, 61, dev)
    mlp = random_mlp(192, [128, 128], 62, dev)
    tc.force("w8")
    first = fp_mlp_cl(feat1, feat2, idx, w, mlp, 1000)  # packs under the default cap
    tc.force(later)
    again = fp_mlp_cl(feat1, feat2, idx, w, mlp, 1000)
    check(again, ref.fp_ref(feat1, feat2, idx, w, 1000, mlp.layers), "fp packed under w8, launched under %s" % later)
    assert torch.equal(first, again)


# ---- every launch of the benchmark's forward -------------------------------------------------------------------------

class Recorder:
    """Wraps pointnet_util.sa_mlp_max_cl / fp_mlp_cl, keeping each launch's inputs, output and build."""

    def __init__(self, tc, monkeypatch):
        self.tc, self.launches = tc, []
        sa0, fp0 = pointnet_util.sa_mlp_max_cl, pointnet_util.fp_mlp_cl

        def sa(xyz_cl, feat_cl, new_xyz_cl, idx, order, mlp, out=None, out_offset=0, out_dtype=torch.float32):
            r = sa0(xyz_cl, feat_cl, new_xyz_cl, idx, order, mlp, out=out, out_offset=out_offset, out_dtype=out_dtype)
            build = tc.last()
            tiles = -(-idx.numel() // 128)
            args = [t.clone() if t is not None else None for t in (xyz_cl, feat_cl, new_xyz_cl, idx)]
            self.launches.append(("sa", args + [order, mlp], r[..., out_offset:out_offset + mlp.cout].clone(), build, tiles))
            return r

        def fp(feat1_cl, feat2_cl, idx, weight, mlp, n, row_order=None, out_dtype=torch.float32):
            r = fp0(feat1_cl, feat2_cl, idx, weight, mlp, n, row_order=row_order, out_dtype=out_dtype)
            build = tc.last()
            tiles = -(-feat2_cl.shape[0] * n // 128)
            args = [t.clone() if t is not None else None for t in (feat1_cl, feat2_cl, idx, weight)]
            self.launches.append(("fp", args + [n, mlp], r.clone(), build, tiles))
            return r

        monkeypatch.setattr(pointnet_util, "sa_mlp_max_cl", sa)
        monkeypatch.setattr(pointnet_util, "fp_mlp_cl", fp)

    def check_all(self, title):
        torch.cuda.synchronize()
        print("\n%s: %d tensor-core launches (%d SMs)" % (title, len(self.launches), sm_count()))
        failures = []
        for i, (kind, args, got, (build, grid, threads), tiles) in enumerate(self.launches):
            if kind == "sa":
                xyz, f, nx, idx, order, mlp = args
                want = ref.sa_ref(xyz, f, nx, idx, order, mlp.layers, out_bf16=got.dtype == torch.bfloat16)
            else:
                f1, f2, idx, w, n, mlp = args
                want = ref.fp_ref(f1, f2, idx, w, n, mlp.layers, out_bf16=got.dtype == torch.bfloat16)
            label = "%d %s %d->%s" % (i, kind, mlp.cin, [l[0].shape[0] for l in mlp.layers])
            frac, mx = ref.stats(got, want)
            print("  %-44s %-13s tiles %6d grid %4d x %3d  frac>1e-4 %.2e  max %.2e" % (label, build, tiles, grid, threads, frac, mx))
            if not (frac <= ref.FRAC_MAX and mx <= ref.MAX_REL):
                failures.append("%s: frac %.3e max %.3e" % (label, frac, mx))
            if tiles > 4 * sm_count() and "_w8" in build:
                failures.append("%s: %d tiles ran the 8-worker build %s" % (label, tiles, build))
        assert not failures, "; ".join(failures)


def test_every_launch_of_the_semseg_bench_forward(tc, monkeypatch):
    """PointNet2SemSeg(21), bf16, batch 32 x 8192 points: the shape bench.py reports."""
    from pn2_b200.models import PointNet2SemSeg
    dev = torch.device("cuda:0")
    tc.force("auto")
    torch.manual_seed(0)
    model = PointNet2SemSeg(21).eval().to(dev)
    x = torch.from_numpy(scenes.scannet_batch(0, 32, 8192)).to(dev).permute(0, 2, 1).contiguous()
    rec = Recorder(tc, monkeypatch)
    with torch.no_grad():
        model(x[:, :3].contiguous(), x[:, 3:].contiguous())
    assert len(rec.launches) == 8
    rec.check_all("PointNet2SemSeg bf16, batch 32 x 8192")


def test_every_launch_of_the_msg_multiview_forward(tc, monkeypatch):
    """PointNet2Multiview2Msg (the MSG stack of config 2), batch 8 x 8192 points, 128-channel lifted image features."""
    from pn2_b200.models import PointNet2Multiview2Msg
    dev = torch.device("cuda:0")
    tc.force("auto")
    torch.manual_seed(1)
    model = PointNet2Multiview2Msg(21).eval().to(dev)
    pts = scenes.scannet_batch(1, 8, 8192)
    xyz = torch.from_numpy(pts[:, :, :3]).to(dev).permute(0, 2, 1).contiguous()
    img = torch.randn(8, 128, 8192, device=dev)
    rec = Recorder(tc, monkeypatch)
    with torch.no_grad():
        model(xyz, img)
    assert len(rec.launches) >= 10
    rec.check_all("PointNet2Multiview2Msg bf16, batch 8 x 8192")


# ---- negative controls ------------------------------------------------------------------------------------------------

def _planted_sa(args, plant):
    xyz, f, nx, idx, mlp = args
    a = ref.sa_operand(xyz, f, nx, idx, XF, rnd=ref.bf16_rz if plant == "round_toward_zero" else ref.bf16_rn)
    if plant == "xyz_column_zeroed":
        a[..., 2] = 0.0  # z of the centred xyz
    if plant == "x_y_swapped":
        a[..., [0, 1]] = a[..., [1, 0]]
    layers = ref.weights_bf16(mlp.layers)
    if plant == "last_layer_bias_slice_dropped":
        w, b, r = layers[-1]
        b = b.clone()
        b[32:64] = 0.0
        layers[-1] = (w, b, r)
    out = ref.finish(ref.mlp_rows(a, layers).amax(dim=2))
    if plant == "last_partial_tile_zeroed":
        gpt = 128 // idx.shape[2]
        groups = idx.shape[0] * idx.shape[1]
        assert groups % gpt, "the case needs a partial last tile"
        out.view(groups, -1)[groups - groups % gpt:] = 0.0
    return out


def _planted_fp(args, plant):
    f1, f2, idx, w, mlp = args
    n = idx.shape[1]
    a = ref.fp_operand(f1, f2, idx, w, n, rnd=ref.bf16_rz if plant == "round_toward_zero" else ref.bf16_rn)
    if plant == "skip_column_zeroed":
        a[..., 3] = 0.0
    layers = ref.weights_bf16(mlp.layers)
    if plant == "last_layer_bias_slice_dropped":
        wt, b, r = layers[-1]
        b = b.clone()
        b[32:64] = 0.0
        layers[-1] = (wt, b, r)
    out = ref.finish(ref.mlp_rows(a, layers))
    if plant == "last_partial_tile_zeroed":
        rows = idx.shape[0] * n
        assert rows % 128, "the case needs a partial last tile"
        out.view(rows, -1)[rows - rows % 128:] = 0.0
    return out


@pytest.mark.parametrize("plant", ["xyz_column_zeroed", "x_y_swapped", "last_layer_bias_slice_dropped", "round_toward_zero",
                                   "last_partial_tile_zeroed"])
@pytest.mark.parametrize("config", ["w8", "w4"])
def test_sa_comparison_rejects_planted_errors(tc, plant, config):
    # 14 groups of 32 samples = 3.5 tiles: the partial last tile holds 1/7 of the output
    got, want, build, args = run_sa(tc, config, 2, 700, 7, 32, 64, [64, 64, 128], XF, "f32", "f32", seed=51)
    check(got, want, "sa control baseline [%s]" % build[0])
    frac, mx = ref.stats(got, _planted_sa(args, plant))
    print("sa control %-32s frac>1e-4 %.2e  max %.2e" % (plant, frac, mx))
    assert not ref.agrees(got, _planted_sa(args, plant))
    assert frac >= 10 * ref.FRAC_MAX, "%s rejected by less than 10x on the fraction (%.3e)" % (plant, frac)


@pytest.mark.parametrize("plant", ["skip_column_zeroed", "last_layer_bias_slice_dropped", "round_toward_zero",
                                   "last_partial_tile_zeroed"])
@pytest.mark.parametrize("config", ["w8", "w4"])
def test_fp_comparison_rejects_planted_errors(tc, plant, config):
    # 200 rows: the partial last tile holds 72 of them
    got, want, build, args = run_fp(tc, config, 1, 200, 50, 6, 128, [128, 128, 64], True, "bf16", "f32", "f32", seed=52)
    check(got, want, "fp control baseline [%s]" % build[0])
    frac, mx = ref.stats(got, _planted_fp(args, plant))
    print("fp control %-32s frac>1e-4 %.2e  max %.2e" % (plant, frac, mx))
    assert not ref.agrees(got, _planted_fp(args, plant))
    assert frac >= 10 * ref.FRAC_MAX, "%s rejected by less than 10x on the fraction (%.3e)" % (plant, frac)
