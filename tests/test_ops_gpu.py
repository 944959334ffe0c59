"""GPU parity of the nine operators: CUDA kernels (through the C ABI) vs the CPU oracle and vs the
reference's own kernels (oracle/_ref/ref_cuda.so) on the same seeded inputs.  Index outputs and pure
copies are compared bit-exactly; interpolation within 1e-5 relative (BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from oracle import ref_cuda
from pn2_b200 import pointnet2_utils as pu
from pn2_b200 import scenes

pytestmark = pytest.mark.gpu


def dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def clouds(kind, B, N, seed):
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        return rng.random((B, N, 3)).astype(np.float32)
    if kind == "dup":  # drawn with replacement from a small pool: exact duplicates, exact ties
        out = np.empty((B, N, 3), np.float32)
        for b in range(B):
            pool = rng.random((max(N // 4, 1), 3)).astype(np.float32)
            out[b] = pool[rng.integers(0, pool.shape[0], N)]
        return out
    if kind == "lattice":
        return rng.integers(0, 6, (B, N, 3)).astype(np.float32) * np.float32(0.25)
    if kind == "scannet":
        return np.stack([scenes.scannet_scene(seed * 10 + b, N)[0] for b in range(B)])
    raise ValueError(kind)


FPS_CASES = [("uniform", 3, 8192, 1024), ("scannet", 2, 8192, 1024), ("dup", 2, 8192, 512), ("lattice", 2, 4096, 300),
             ("uniform", 2, 1024, 256), ("dup", 3, 1024, 256), ("dup", 2, 256, 64), ("dup", 2, 64, 16),
             ("uniform", 2, 1000, 100), ("dup", 2, 3000, 200), ("dup", 2, 6000, 200), ("uniform", 1, 5, 5),
             ("dup", 2, 40, 50), ("uniform", 2, 33, 33), ("uniform", 1, 1, 2), ("dup", 1, 10000, 64)]


@pytest.mark.parametrize("kind,B,N,M", FPS_CASES)
def test_fps_bit_exact(cuda, kind, B, N, M):
    xyz = clouds(kind, B, N, N + M)
    got = pu.furthest_point_sample(dev(xyz, cuda), M).cpu().numpy()
    want = orc.furthest_point_sample(xyz, M)
    np.testing.assert_array_equal(got, want)
    if ref_cuda.available():
        ref = ref_cuda.furthest_point_sample(dev(xyz, cuda), M).cpu().numpy()
        np.testing.assert_array_equal(got, ref)


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("kind,B,N,M", [("scannet", 3, 8192, 1024), ("dup", 2, 8192, 700), ("lattice", 2, 4096, 300),
                                        ("dup", 2, 3000, 200), ("uniform", 2, 1025, 64), ("dup", 1, 16384, 300),
                                        ("uniform", 1, 12000, 150), ("dup", 2, 2048, 2100), ("uniform", 1, 20000, 120),
                                        ("dup", 1, 30000, 100), ("uniform", 1, 35000, 200), ("uniform", 1, 50000, 40),
                                        ("dup", 2, 5000, 5100), ("lattice", 2, 8000, 300), ("dup", 1, 6001, 300),
                                        ("uniform", 2, 4097, 64), ("dup", 2, 8192, 100), ("lattice", 2, 6000, 127)])
def test_fps_single_cta_and_cluster_kernels_agree_with_reference(cuda, mode, kind, B, N, M):
    """Both FPS policies (one 256-thread CTA per cloud / four-CTA cluster with DSMEM exchange) are bit-exact; duplicated
    points and lattices make exact distance ties frequent, so the tie order is exercised.  Under the single-CTA policy the
    last three shapes (4096 < N <= 8192, M < 128) run the index-interleaved kernel with 32 points per thread."""
    from pn2_b200 import _lib
    xyz = clouds(kind, B, N, 3 * N + M)
    _lib.load().pn2_debug_set_fps_mode(mode)
    try:
        got = pu.furthest_point_sample(dev(xyz, cuda), M).cpu().numpy()
    finally:
        _lib.load().pn2_debug_set_fps_mode(0)
    np.testing.assert_array_equal(got, orc.furthest_point_sample(xyz, M))


@pytest.mark.parametrize("mode", [1])
@pytest.mark.parametrize("kind,B,N,M", [("scannet", 4, 8192, 1024), ("dup", 2, 8192, 1024), ("lattice", 2, 8192, 1024), ("uniform", 2, 8192, 2048),
                                        ("dup", 2, 5000, 5100), ("uniform", 2, 4097, 256), ("lattice", 2, 4096, 512), ("dup", 3, 2049, 300),
                                        ("same", 2, 8192, 200), ("plane", 2, 6000, 700), ("line", 1, 8192, 400),
                                        # M < 128: the index-interleaved kernel
                                        ("scannet", 4, 8192, 127), ("dup", 2, 8192, 64), ("lattice", 2, 8192, 120), ("uniform", 2, 8192, 100),
                                        ("dup", 2, 5000, 120), ("uniform", 2, 4097, 127), ("lattice", 2, 4100, 90), ("same", 2, 8192, 100),
                                        ("plane", 2, 6000, 110), ("line", 1, 8192, 64), ("same", 1, 4097, 127)])
def test_fps_slab_kernel_bit_exact(cuda, mode, kind, B, N, M):
    """One CTA per cloud (mode 1 = the single-CTA policy) against the oracle: for 4096 < N <= 8192 the kernel with spatial
    slabs per warp and skipped rounds, or the index-interleaved kernel it replaced when M < 128 picks make the slab set-up
    not pay.  Duplicates / lattices (frequent exact ties, explicit tie keys), degenerate clouds (all points equal: zero
    extent; points on a plane / a line), padded slabs."""
    from pn2_b200 import _lib
    if kind == "same":
        xyz = np.tile(np.float32([[0.25, -1.5, 3.0]]), (B, N, 1))
    elif kind == "plane":
        xyz = clouds("uniform", B, N, 11 * N + M)
        xyz[:, :, 2] = np.float32(0.5)
    elif kind == "line":
        xyz = clouds("dup", B, N, 13 * N + M)
        xyz[:, :, 1:] = np.float32(-2.0)
    else:
        xyz = clouds(kind, B, N, 9 * N + M)
    _lib.load().pn2_debug_set_fps_mode(mode)
    try:
        got = pu.furthest_point_sample(dev(xyz, cuda), M).cpu().numpy()
    finally:
        _lib.load().pn2_debug_set_fps_mode(0)
    np.testing.assert_array_equal(got, orc.furthest_point_sample(xyz, M))


@pytest.mark.parametrize("kind,B,N,M", [("dup", 1, 49153, 60), ("lattice", 1, 60000, 48), ("dup", 2, 65536, 40), ("uniform", 1, 57000, 64),
                                        ("dup", 1, 70000, 40), ("dup", 2, 131072, 24), ("lattice", 1, 100000, 32), ("uniform", 1, 65537, 48)])
def test_fps_large_clouds_bit_exact(cuda, kind, B, N, M):
    """The 8-CTA cluster kernel (49152 < N <= 65536, tie key extended by the thread's half) and fps_global_kernel
    (N > 65536, running minima in caller scratch), with duplicated / lattice points so that exact ties are frequent."""
    xyz = clouds(kind, B, N, 7 * N + M)
    got = pu.furthest_point_sample(dev(xyz, cuda), M).cpu().numpy()
    np.testing.assert_array_equal(got, orc.furthest_point_sample(xyz, M))
    if ref_cuda.available():
        np.testing.assert_array_equal(got, ref_cuda.furthest_point_sample(dev(xyz, cuda), M).cpu().numpy())


def test_fps_properties_full_size(cuda):
    # BASELINE config size, properties that need no oracle: first index 0, unique picks while distinct
    # points remain, and the running minimum distance of the picks is non-increasing.
    xyz = clouds("uniform", 8, 8192, 5)
    idx = pu.furthest_point_sample(dev(xyz, cuda), 1024).cpu().numpy()
    assert (idx[:, 0] == 0).all() and idx.min() >= 0 and idx.max() < 8192
    for b in range(8):
        assert len(set(idx[b].tolist())) == 1024
        p = xyz[b][idx[b]].astype(np.float64)
        dmin = np.full(8192, np.inf)
        prev = np.inf
        for j in range(1, 1024):
            dmin = np.minimum(dmin, ((xyz[b].astype(np.float64) - p[j - 1]) ** 2).sum(1))
            cur = dmin[idx[b, j]]
            assert cur <= prev * (1 + 1e-6) and abs(cur - dmin.max()) <= 1e-6 * max(dmin.max(), 1e-12)
            prev = cur


def test_fps_m_zero_and_gather_fused(cuda):
    from pn2_b200.pointnet_util import fps_gather_cl
    xyz = clouds("scannet", 2, 2048, 9)
    x = dev(xyz, cuda)
    idx, new_xyz = fps_gather_cl(x, 128)
    np.testing.assert_array_equal(idx.cpu().numpy(), orc.furthest_point_sample(xyz, 128))
    np.testing.assert_array_equal(new_xyz.cpu().numpy(), np.take_along_axis(xyz, idx.cpu().numpy()[..., None].astype(np.int64), 1))
    assert pu.furthest_point_sample(x, 0).shape == (2, 0)


BQ_CASES = [("scannet", 2, 8192, 1024, 0.1, 32), ("scannet", 2, 8192, 1024, 0.2, 32), ("uniform", 2, 1024, 256, 0.2, 32),
            ("dup", 2, 256, 64, 0.4, 32), ("uniform", 2, 64, 16, 0.8, 32), ("uniform", 2, 5000, 300, 0.05, 16),
            ("lattice", 1, 3000, 100, 0.25, 64), ("uniform", 1, 100, 33, 0.3, 7), ("uniform", 1, 2500, 40, 10.0, 128)]


@pytest.mark.parametrize("kind,B,N,M,r,K", BQ_CASES)
def test_ball_query_bit_exact(cuda, kind, B, N, M, r, K):
    xyz = clouds(kind, B, N, N + M + K)
    new_xyz = xyz[:, orc.furthest_point_sample(xyz, M)[0]].copy() if kind != "lattice" else xyz[:, :M].copy()
    new_xyz[:, -1] += 100.0  # one query with an empty ball
    got = pu.ball_query(r, K, dev(xyz, cuda), dev(new_xyz, cuda)).cpu().numpy()
    want = orc.ball_query(r, K, xyz, new_xyz)
    np.testing.assert_array_equal(got, want)
    assert (got[:, -1] == 0).all()
    if ref_cuda.available():
        ref = ref_cuda.ball_query(r, K, dev(xyz, cuda), dev(new_xyz, cuda)).cpu().numpy()
        np.testing.assert_array_equal(got, ref)


NN_CASES = [("scannet", 2, 8192, 1024), ("uniform", 2, 1024, 256), ("lattice", 2, 500, 64), ("uniform", 2, 64, 16),
            ("uniform", 1, 300, 5000), ("uniform", 1, 10, 2), ("dup", 2, 700, 100)]


@pytest.mark.parametrize("kind,B,n,m", NN_CASES)
def test_three_nn_bit_exact(cuda, kind, B, n, m):
    unknown = clouds(kind, B, n, n + m)
    known = clouds(kind, B, m, n + m + 1) if kind != "scannet" else unknown[:, :m].copy()
    d, idx = pu.three_nn(dev(unknown, cuda), dev(known, cuda))
    wd, widx = orc.three_nn(unknown, known)
    np.testing.assert_array_equal(idx.cpu().numpy(), widx)
    np.testing.assert_array_equal(d.cpu().numpy(), wd)
    if ref_cuda.available():
        rd, ridx = ref_cuda.three_nn(dev(unknown, cuda), dev(known, cuda))
        np.testing.assert_array_equal(idx.cpu().numpy(), ridx.cpu().numpy())
        np.testing.assert_array_equal(d.cpu().numpy(), rd.cpu().numpy())


def test_three_nn_weights_fused(cuda):
    from pn2_b200.pointnet_util import three_nn_weights_cl
    unknown, known = clouds("scannet", 2, 4096, 3), clouds("scannet", 2, 512, 3)[:, :512]
    known[:, 0] = unknown[:, 0]  # a zero distance exercises the 1e-10 clamp
    idx, w = three_nn_weights_cl(dev(unknown, cuda), dev(known, cuda))
    d, widx = orc.three_nn(unknown, known)
    np.testing.assert_array_equal(idx.cpu().numpy(), widx)
    np.testing.assert_allclose(w.cpu().numpy(), orc.fp_weights(d), rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("B,C,N,M", [(2, 3, 8192, 1024), (2, 64, 1024, 256), (1, 131, 777, 333), (2, 1, 50, 70)])
def test_gather_bit_exact_and_grad(cuda, B, C, N, M):
    rng = np.random.default_rng(C * N)
    f = rng.standard_normal((B, C, N)).astype(np.float32)
    idx = rng.integers(0, N, (B, M)).astype(np.int32)
    ft = dev(f, cuda).requires_grad_(True)
    out = pu.gather_operation(ft, dev(idx, cuda))
    np.testing.assert_array_equal(out.detach().cpu().numpy(), orc.gather_operation(f, idx))
    go = rng.standard_normal((B, C, M)).astype(np.float32)
    out.backward(dev(go, cuda))
    np.testing.assert_allclose(ft.grad.cpu().numpy(), orc.gather_operation_grad(go, idx, N), rtol=1e-5, atol=1e-5)
    if ref_cuda.available():
        np.testing.assert_array_equal(out.detach().cpu().numpy(), ref_cuda.gather_operation(dev(f, cuda), dev(idx, cuda)).cpu().numpy())


@pytest.mark.parametrize("B,C,N,P,S", [(2, 3, 8192, 1024, 32), (2, 64, 1024, 256, 32), (1, 259, 64, 16, 32), (2, 5, 100, 7, 3)])
def test_group_bit_exact_and_grad(cuda, B, C, N, P, S):
    rng = np.random.default_rng(C * N + S)
    f = rng.standard_normal((B, C, N)).astype(np.float32)
    idx = rng.integers(0, N, (B, P, S)).astype(np.int32)
    ft = dev(f, cuda).requires_grad_(True)
    out = pu.grouping_operation(ft, dev(idx, cuda))
    np.testing.assert_array_equal(out.detach().cpu().numpy(), orc.grouping_operation(f, idx))
    go = rng.standard_normal((B, C, P, S)).astype(np.float32)
    out.backward(dev(go, cuda))
    np.testing.assert_allclose(ft.grad.cpu().numpy(), orc.grouping_operation_grad(go, idx, N), rtol=1e-4, atol=1e-4)
    if ref_cuda.available():
        np.testing.assert_array_equal(out.detach().cpu().numpy(), ref_cuda.grouping_operation(dev(f, cuda), dev(idx, cuda)).cpu().numpy())


# the staged-row kernel of group_points where few rows fit in shared memory (long source rows): one staged row per
# 1024-thread CTA with the index vectors of the next iteration in flight (N = 32768), two rows and an index list that is
# not a multiple of four (scalar loop), four rows per 512-thread CTA
@pytest.mark.parametrize("B,C,N,P,S", [(2, 16, 32768, 2048, 32), (1, 33, 20000, 1667, 25), (2, 17, 12000, 3000, 8)])
def test_group_long_rows_bit_exact(cuda, B, C, N, P, S):
    rng = np.random.default_rng(C * N + S)
    f = rng.standard_normal((B, C, N)).astype(np.float32)
    idx = rng.integers(0, N, (B, P, S)).astype(np.int32)
    idx[:, 0, :] = N - 1  # last element of every row
    out = pu.grouping_operation(dev(f, cuda), dev(idx, cuda))
    np.testing.assert_array_equal(out.cpu().numpy(), orc.grouping_operation(f, idx))


@pytest.mark.parametrize("B,C,m,n", [(2, 128, 1024, 8192), (2, 256, 64, 256), (1, 7, 50, 33), (2, 512, 16, 64),
                                     (1, 70, 8192, 32768), (1, 66, 15000, 30002), (2, 33, 6000, 12001),  # large coarse sets
                                     (1, 70, 4096, 16384), (2, 40, 2048, 8192)])  # tiled kernel, one / two CTAs per SM (index prefetch)
def test_three_interpolate_and_grad(cuda, B, C, m, n):
    rng = np.random.default_rng(C + m + n)
    f = rng.standard_normal((B, C, m)).astype(np.float32)
    idx = rng.integers(0, m, (B, n, 3)).astype(np.int32)
    w = rng.random((B, n, 3)).astype(np.float32)
    w /= w.sum(-1, keepdims=True)
    ft = dev(f, cuda).requires_grad_(True)
    out = pu.three_interpolate(ft, dev(idx, cuda), dev(w, cuda))
    want = orc.three_interpolate(f, idx, w)
    # tolerance from BASELINE.json: interpolated outputs within 1e-5 relative (fp32); the kernel uses the
    # reference's own rounding sequence, so in practice the match is exact
    np.testing.assert_allclose(out.detach().cpu().numpy(), want, rtol=1e-5, atol=1e-6)
    np.testing.assert_array_equal(out.detach().cpu().numpy(), want)
    go = rng.standard_normal((B, C, n)).astype(np.float32)
    out.backward(dev(go, cuda))
    np.testing.assert_allclose(ft.grad.cpu().numpy(), orc.three_interpolate_grad(go, idx, w, m), rtol=1e-4, atol=1e-4)
    if ref_cuda.available():
        ref = ref_cuda.three_interpolate(dev(f, cuda), dev(idx, cuda), dev(w, cuda)).cpu().numpy()
        np.testing.assert_array_equal(out.detach().cpu().numpy(), ref)


# every kernel choice of pn2_three_interpolate (pn2_debug_set_interp_mode: tiled kernels, the lane-along-channel kernel in its
# 512- and 256-thread forms, automatic) against the oracle and the reference's kernel, bit for bit; shapes cover a partial
# last channel tile (100, 37 channels), a partial last granule (n = 8200), a coarse set that is not a multiple of 4
# (scalar stage), a single coarse point and two (cloud, tile) pairs inside one CTA's range
@pytest.mark.parametrize("B,C,m,n", [(4, 128, 1024, 8192), (3, 100, 1023, 8200), (5, 37, 700, 4104), (2, 128, 1, 512),
                                     (16, 64, 256, 1024), (40, 32, 64, 256), (2, 96, 1500, 30000)])
def test_three_interpolate_kernel_choices(cuda, B, C, m, n):
    from pn2_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(B + C + m + n)
    f = rng.standard_normal((B, C, m)).astype(np.float32)
    idx = rng.integers(0, m, (B, n, 3)).astype(np.int32)
    w = rng.random((B, n, 3)).astype(np.float32)
    w /= w.sum(-1, keepdims=True)
    want = orc.three_interpolate(f, idx, w)
    ft, it, wt = dev(f, cuda), dev(idx, cuda), dev(w, cuda)
    try:
        for mode in (1, 32, 32 | 256, 0):
            lib.pn2_debug_set_interp_mode(mode)
            got = pu.three_interpolate(ft, it, wt).cpu().numpy()
            np.testing.assert_array_equal(got, want, err_msg="mode %d" % mode)
    finally:
        lib.pn2_debug_set_interp_mode(0)
    if ref_cuda.available():
        np.testing.assert_array_equal(ref_cuda.three_interpolate(ft, it, wt).cpu().numpy(), want)


def test_aliases_and_query_and_group(cuda):
    xyz = clouds("scannet", 2, 2048, 21)
    x = dev(xyz, cuda)
    idx = pu.farthest_point_sample(x, 64)
    np.testing.assert_array_equal(idx.cpu().numpy(), orc.furthest_point_sample(xyz, 64))
    new_xyz = pu.index_points(x, idx)
    np.testing.assert_array_equal(new_xyz.cpu().numpy(), np.take_along_axis(xyz, idx.cpu().numpy()[..., None].astype(np.int64), 1))
    bq = pu.query_ball_point(0.2, 16, x, new_xyz)
    np.testing.assert_array_equal(bq.cpu().numpy(), orc.ball_query(0.2, 16, xyz, new_xyz.cpu().numpy()))
    grouped = pu.index_points(x, bq)
    assert grouped.shape == (2, 64, 16, 3)
    sq = pu.square_distance(new_xyz[:, :4], x[:, :100]).cpu().numpy()
    for b in range(2):
        for i in range(4):
            for k in range(0, 100, 17):
                a, c = new_xyz[b, i].cpu().numpy(), xyz[b, k]
                dx, dy, dz = np.float32(a[0] - c[0]), np.float32(a[1] - c[1]), np.float32(a[2] - c[2])
                t = np.float32(np.float64(dy) * dy)
                t = np.float32(np.float64(dx) * dx + t)
                assert sq[b, i, k] == np.float32(np.float64(dz) * dz + t)
    feats = dev(np.random.default_rng(0).standard_normal((2, 5, 2048)).astype(np.float32), cuda)
    qg = pu.QueryAndGroup(0.2, 16)(x, new_xyz, feats)
    assert qg.shape == (2, 8, 64, 16)
    want_xyz = orc.grouping_operation(xyz.transpose(0, 2, 1), bq.cpu().numpy()) - new_xyz.cpu().numpy().transpose(0, 2, 1)[..., None]
    np.testing.assert_array_equal(qg[:, :3].cpu().numpy(), want_xyz)
    ga = pu.GroupAll()(x, None, feats)
    assert ga.shape == (2, 8, 1, 2048)


# ---- uniform-grid neighbour search: bit-identical to the brute-force kernels (and hence to the reference) ------------

GRID_BQ = [("uniform", 1, 32768, 256, 0.03, 32, 1.01), ("uniform", 1, 16384, 512, 0.04, 32, 1.01), ("scannet", 2, 8192, 1024, 0.1, 32, 1.01), ("scannet", 2, 8192, 1024, 0.2, 32, 1.01), ("dup", 2, 4096, 300, 0.1, 16, 1.5),
           ("lattice", 1, 3000, 100, 0.25, 64, 1.01), ("uniform", 1, 2500, 40, 10.0, 128, 1.01), ("uniform", 2, 5000, 300, 0.05, 16, 1.01),
           ("dup", 2, 1024, 256, 0.3, 32, 1.01), ("uniform", 1, 700, 64, 0.3, 200, 0.3), ("scannet", 1, 8192, 512, 0.8, 32, 1.01),
           # beyond the single-CTA sort: counting sort by cell (order inside a cell unspecified, results identical)
           ("uniform", 2, 34720, 300, 0.03, 32, 1.01), ("dup", 1, 40000, 200, 0.05, 16, 1.01), ("uniform", 1, 70000, 128, 0.02, 32, 1.5)]


@pytest.mark.parametrize("kind,B,N,M,r,K,cellf", GRID_BQ)
def test_grid_ball_query_bit_exact(cuda, kind, B, N, M, r, K, cellf):
    from pn2_b200.pointnet_util import SpatialGrid
    xyz = clouds(kind, B, N, 7 * N + M)
    new_xyz = xyz[:, orc.furthest_point_sample(xyz, M)[0]].copy()
    new_xyz[:, -1] += 100.0   # far outside the grid: empty ball
    new_xyz[:, -2] -= 0.03    # off-grid-point query
    grid = SpatialGrid(dev(xyz, cuda), cellf * r)
    got = grid.ball_query(r, K, dev(new_xyz, cuda)).cpu().numpy()
    np.testing.assert_array_equal(got, orc.ball_query(r, K, xyz, new_xyz))
    order = grid.order.cpu().numpy()
    for b in range(B):
        assert sorted(order[b].tolist()) == list(range(N))  # a permutation


GRID_NN = [("scannet", 2, 8192, 1024, 0.1), ("scannet", 2, 8192, 1024, 0.0), ("uniform", 2, 3000, 600, 0.0), ("lattice", 2, 900, 500, 0.3),
           ("dup", 2, 2000, 700, 0.05), ("uniform", 1, 500, 2, 0.0), ("uniform", 1, 400, 5000, 0.02), ("scannet", 1, 4096, 64, 0.0),
           ("uniform", 1, 1500, 40000, 0.0)]  # a known set beyond the single-CTA sort


@pytest.mark.parametrize("kind,B,n,m,cell", GRID_NN)
def test_grid_three_nn_bit_exact(cuda, kind, B, n, m, cell):
    from pn2_b200.pointnet_util import SpatialGrid
    unknown = clouds(kind, B, n, 11 * n + m)
    known = clouds(kind, B, m, 11 * n + m + 1) if kind != "scannet" else unknown[:, :m].copy()
    unknown[:, 0] += 50.0  # a query far outside the known set's bounding box
    grid = SpatialGrid(dev(known, cuda), cell)
    idx, d2 = grid.three_nn(dev(unknown, cuda), want_dist2=True, want_weight=False)
    wd2, widx = orc.three_nn_dist2(unknown, known)
    np.testing.assert_array_equal(idx.cpu().numpy(), widx)
    np.testing.assert_array_equal(d2.cpu().numpy(), wd2)
    order = SpatialGrid(dev(unknown, cuda), 0.0).order
    idx2, w = grid.three_nn(dev(unknown, cuda), query_order=order)
    np.testing.assert_array_equal(idx2.cpu().numpy(), widx)
    np.testing.assert_allclose(w.cpu().numpy(), orc.fp_weights(np.sqrt(wd2)), rtol=1e-5, atol=1e-7)
