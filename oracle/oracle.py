"""numpy front end of the CPU oracle (oracle/pn2_oracle.c).

TEST INFRASTRUCTURE ONLY -- see the header of pn2_oracle.c.  The product package
never imports this module; tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs do.

Parity status: the reference has no golden vectors for this path; the oracle is
pinned against the reference's own kernels (oracle/_ref/ref_cuda.so) run on a
B200 -- tests/test_ops_gpu.py live, tests/golden/ref_cuda_r1.npz offline -- and, for
the lifting and the frustum count, against the reference's own utils/projection.py
run on the host (tests/golden/projection_r2.npz); see tests/test_golden.py.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

_f = ctypes.POINTER(ctypes.c_float)
_i = ctypes.POINTER(ctypes.c_int32)


def lib():
    global _LIB
    if _LIB is None:
        import importlib.util
        spec = importlib.util.spec_from_file_location("_oracle_build", os.path.join(_HERE, "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        path = mod.build_oracle()  # rebuilds only when pn2_oracle.c or its flags changed
        _LIB = ctypes.CDLL(path)
        _LIB.orc_project_point.restype = ctypes.c_int32
        _LIB.orc_opt_n_threads.restype = ctypes.c_int
        _LIB.orc_num_threads.restype = ctypes.c_int
    return _LIB


def _fp(a):
    assert a.dtype == np.float32 and a.flags.c_contiguous
    return a.ctypes.data_as(_f)


def _ip(a):
    assert a.dtype == np.int32 and a.flags.c_contiguous
    return a.ctypes.data_as(_i)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def num_threads():
    return int(lib().orc_num_threads())


def opt_n_threads(n):
    return int(lib().orc_opt_n_threads(int(n)))


def furthest_point_sample(xyz, npoint):
    """xyz (B,N,3) f32 -> idx (B,npoint) i32.  model/pointnet2_utils.py:10-36"""
    xyz = _f32(xyz)
    B, N, _ = xyz.shape
    idx = np.zeros((B, npoint), dtype=np.int32)
    lib().orc_fps(B, N, npoint, _fp(xyz), _ip(idx))
    return idx


def gather_operation(features, idx):
    """features (B,C,N), idx (B,M) -> (B,C,M).  model/pointnet2_utils.py:39-73"""
    features, idx = _f32(features), _i32(idx)
    B, C, N = features.shape
    M = idx.shape[1]
    out = np.empty((B, C, M), dtype=np.float32)
    lib().orc_gather(B, C, N, M, _fp(features), _ip(idx), _fp(out))
    return out


def gather_operation_grad(grad_out, idx, N):
    grad_out, idx = _f32(grad_out), _i32(idx)
    B, C, M = grad_out.shape
    g = np.zeros((B, C, N), dtype=np.float32)
    lib().orc_gather_grad(B, C, N, M, _fp(grad_out), _ip(idx), _fp(g))
    return g


def ball_query(radius, nsample, xyz, new_xyz):
    """xyz (B,N,3), new_xyz (B,M,3) -> idx (B,M,nsample).  model/pointnet2_utils.py:198-226"""
    xyz, new_xyz = _f32(xyz), _f32(new_xyz)
    B, N, _ = xyz.shape
    M = new_xyz.shape[1]
    idx = np.zeros((B, M, nsample), dtype=np.int32)
    lib().orc_ball_query(B, N, M, ctypes.c_float(radius), nsample, _fp(new_xyz), _fp(xyz), _ip(idx))
    return idx


def grouping_operation(features, idx):
    """features (B,C,N), idx (B,P,S) -> (B,C,P,S).  model/pointnet2_utils.py:154-195"""
    features, idx = _f32(features), _i32(idx)
    B, C, N = features.shape
    _, P, S = idx.shape
    out = np.empty((B, C, P, S), dtype=np.float32)
    lib().orc_group(B, C, N, P, S, _fp(features), _ip(idx), _fp(out))
    return out


def grouping_operation_grad(grad_out, idx, N):
    grad_out, idx = _f32(grad_out), _i32(idx)
    B, C, P, S = grad_out.shape
    g = np.zeros((B, C, N), dtype=np.float32)
    lib().orc_group_grad(B, C, N, P, S, _fp(grad_out), _ip(idx), _fp(g))
    return g


def three_nn_dist2(unknown, known):
    unknown, known = _f32(unknown), _f32(known)
    B, n, _ = unknown.shape
    m = known.shape[1]
    d2 = np.empty((B, n, 3), dtype=np.float32)
    idx = np.empty((B, n, 3), dtype=np.int32)
    lib().orc_three_nn(B, n, m, _fp(unknown), _fp(known), _fp(d2), _ip(idx))
    return d2, idx


def three_nn(unknown, known):
    """-> (dist (B,n,3) = sqrt of the kernel's squared distances, idx).  model/pointnet2_utils.py:76-104"""
    d2, idx = three_nn_dist2(unknown, known)
    return np.sqrt(d2), idx


def three_interpolate(features, idx, weight):
    """features (B,C,m), idx/weight (B,n,3) -> (B,C,n).  model/pointnet2_utils.py:107-151"""
    features, idx, weight = _f32(features), _i32(idx), _f32(weight)
    B, C, m = features.shape
    n = idx.shape[1]
    out = np.empty((B, C, n), dtype=np.float32)
    lib().orc_three_interpolate(B, C, m, n, _fp(features), _ip(idx), _fp(weight), _fp(out))
    return out


def three_interpolate_grad(grad_out, idx, weight, m):
    grad_out, idx, weight = _f32(grad_out), _i32(idx), _f32(weight)
    B, C, n = grad_out.shape
    g = np.zeros((B, C, m), dtype=np.float32)
    lib().orc_three_interpolate_grad(B, C, n, m, _fp(grad_out), _ip(idx), _fp(weight), _fp(g))
    return g


def fp_weights(dist):
    """model/pointnet_util.py:206-208: clamp 1e-10, reciprocal of the (un-squared) distance, normalise."""
    d = np.array(dist, dtype=np.float32, copy=True)
    d[d < np.float32(1e-10)] = np.float32(1e-10)
    w = (np.float32(1.0) / d).astype(np.float32)
    s = ((w[..., 0] + w[..., 1]) + w[..., 2]).astype(np.float32)
    return (w / s[..., None]).astype(np.float32)


def lift_views(points, feats, depth, w2c, corner2, corner4, normals, intr, dmin, dmax, acc, reduce="max"):
    """Batched multi-view lifting; see orc_lift_views.  Returns (out (B,C,N), pix (B,V,N))."""
    points, feats, depth = _f32(points), _f32(feats), _f32(depth)
    w2c, corner2, corner4, normals, intr = _f32(w2c), _f32(corner2), _f32(corner4), _f32(normals), _f32(intr)
    B, N, _ = points.shape
    _, V, C, H, W = feats.shape
    out = np.empty((B, C, N), dtype=np.float32)
    pix = np.empty((B, V, N), dtype=np.int32)
    lib().orc_lift_views(B, N, V, C, H, W, _fp(points), _fp(feats), _fp(depth), _fp(w2c), _fp(corner2), _fp(corner4),
                         _fp(normals), _fp(intr), ctypes.c_float(dmin), ctypes.c_float(dmax), ctypes.c_float(acc),
                         1 if reduce == "first" else 0, _fp(out), _ip(pix))
    return out, pix


def frustum_count(points, corners, normals, return_mask=False):
    """points (N,3), corners (P,8,3), normals (P,6,3) fp32 -> counts (P,) int64 [, mask (P,N) bool]: the loader's fp64
    frustum membership test, data_utils/ScanNetDataLoader.py:91-97 -> utils/projection.py:132-164."""
    points, corners, normals = _f32(points), _f32(corners), _f32(normals)
    N, P = points.shape[0], corners.shape[0]
    counts = np.zeros(P, dtype=np.int64)
    mask = np.zeros((P, N), dtype=np.uint8) if return_mask else None
    lib().orc_frustum_count(N, P, _fp(points), _fp(corners), _fp(normals), counts.ctypes.data_as(ctypes.c_void_p),
                            mask.ctypes.data_as(ctypes.c_void_p) if return_mask else None)
    return (counts, mask.astype(bool)) if return_mask else counts


def mlp_layer(x, w, b, relu=True):
    """x (rows,cin), w (cout,cin), b (cout) -> (rows,cout)"""
    x, w, b = _f32(x), _f32(w), _f32(b)
    rows, cin = x.shape
    cout = w.shape[0]
    y = np.empty((rows, cout), dtype=np.float32)
    lib().orc_mlp_layer(rows, cin, cout, _fp(x), _fp(w), _fp(b), 1 if relu else 0, _fp(y))
    return y
