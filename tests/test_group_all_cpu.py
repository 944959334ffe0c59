"""The group_all entry points (pn2_sa_all_mlp_max, the PN2_ROWS_ALL row source, pn2_train_bn_relu_max_all,
pn2_train_max_bwd_all) refuse bad input with a message before any CUDA call, so this runs without a GPU; empty batches
are no-ops."""
import ctypes

from pn2_b200 import _lib

FAKE = 1 << 20  # a non-null address; validation fails before anything is dereferenced


def _mlp(widths, c0, relu_last=True):
    d = _lib.Pn2Mlp()
    d.num_layers = len(widths)
    c = c0
    for i, w in enumerate(widths):
        d.cin[i], d.cout[i], d.relu[i] = c, w, int(relu_last or i < len(widths) - 1)
        d.weight[i] = d.bias[i] = FAKE
        c = w
    return d


def _sa_all(b, n, d, mlp, xyz=FAKE, feat=FAKE, out=FAKE, stride=None, offset=0):
    lib = _lib.load()
    cl = mlp.cout[mlp.num_layers - 1] if mlp is not None else 0
    stride = cl + offset if stride is None else stride
    return lib.pn2_sa_all_mlp_max(b, n, d, xyz, feat, None if mlp is None else ctypes.byref(mlp), out, stride, offset, None)


def test_sa_all_mlp_max_validates_without_gpu():
    err = _lib.load().pn2_last_error
    m = _mlp([32, 64], 8)
    assert _sa_all(2, 0, 5, m) == 1 and b"bad dims" in err()
    assert _sa_all(-1, 16, 5, m) == 1 and b"bad dims" in err()
    assert _sa_all(2, 16, -1, m) == 1 and b"bad dims" in err()
    assert _sa_all(2, 16, 5, None) == 1 and b"null mlp" in err()
    assert _sa_all(2, 16, 6, m) == 1 and b"expects cin" in err()                 # 3 + d must feed layer 0
    assert _sa_all(2, 16, 5, m, stride=63) == 1 and b"out_stride" in err()
    assert _sa_all(2, 16, 5, m, stride=64, offset=1) == 1 and b"out_stride" in err()
    assert _sa_all(2, 16, 5, m, offset=-1, stride=64) == 1 and b"out_stride" in err()
    assert _sa_all(2, 16, 5, m, xyz=None) == 1 and b"null pointer" in err()
    assert _sa_all(2, 16, 5, m, feat=None) == 1 and b"null pointer" in err()     # d > 0 needs features
    assert _sa_all(2, 16, 5, m, out=None) == 1 and b"null pointer" in err()
    assert _sa_all(2, 16, 5, _mlp([32, 64], 8, relu_last=False)) == 2 and b"ReLU" in err()   # PN2_ERR_UNSUPPORTED
    assert _sa_all(0, 16, 5, m, xyz=None, feat=None, out=None) == 0              # no clouds: no-op


def test_sa_all_support_query_is_the_row_tile_query():
    lib = _lib.load()
    cls = _mlp([256, 512, 1024], 259)   # the classification head's group_all layer
    assert lib.pn2_mlp_fp32_supported(ctypes.byref(cls), 259, 0) == 1
    assert lib.pn2_mlp_fp32_supported(ctypes.byref(_mlp([4096, 64], 8)), 8, 0) == 0   # beyond shared memory


def _all(**over):
    d = dict(kind=_lib.ROWS_ALL, b=2, n=100, d=5, xyz=FAKE, feat=FAKE)
    d.update(over)
    return _lib.Pn2Rows(**d)


def _fwd(rows, cin, desc):
    return _lib.load().pn2_train_linear_fwd_rows(rows, cin, 16, ctypes.byref(desc), FAKE, FAKE, FAKE, FAKE, None)


def _bwd(rows, cin, desc, g_in=None, g_skip=None):
    return _lib.load().pn2_train_linear_bwd_rows(rows, cin, 16, ctypes.byref(desc), *([FAKE] * 8), g_in, g_skip, FAKE, None)


def test_all_row_source_validates_without_gpu():
    err = _lib.load().pn2_last_error
    R = 200
    assert _fwd(R, 8, _all(kind=4)) == 1 and b"unknown row source kind" in err()
    assert _fwd(R, 8, _all(n=0)) == 1 and b"bad group_all source" in err()
    assert _fwd(R, 8, _all(d=-1)) == 1 and b"bad group_all source" in err()
    assert _fwd(R + 1, 8, _all()) == 1 and b"do not match" in err()
    assert _fwd(R, 9, _all()) == 1 and b"do not match" in err()
    assert _fwd(R, 8, _all(xyz=None)) == 1 and b"null pointer" in err()
    assert _fwd(R, 8, _all(feat=None)) == 1 and b"null pointer" in err()          # d > 0 needs features
    assert _fwd(R, 3, _all(d=0)) == 1 and b"null pointer" in err()                # d == 0 takes none
    assert _fwd(0, 8, _all()) == 0                                                 # no rows: no-op
    assert _bwd(R, 8, _all(), g_skip=FAKE) == 1 and b"g_skip" in err()
    assert _bwd(R, 3, _all(d=0, feat=None), g_in=FAKE) == 1 and b"no input gradient" in err()
    assert _bwd(R, 8, _all(xyz=None)) == 1 and b"null pointer" in err()
    assert _bwd(R + 1, 8, _all()) == 1 and b"do not match" in err()


def test_pooling_over_all_rows_validates_without_gpu():
    lib = _lib.load()
    err = lib.pn2_last_error
    mx, bw = lib.pn2_train_bn_relu_max_all, lib.pn2_train_max_bwd_all
    assert mx(4, 0, 8, FAKE, FAKE, FAKE, FAKE, 8, 0, FAKE, None) == 1 and b"bad dims" in err()       # k < 1
    assert mx(4, 1 << 31, 8, FAKE, FAKE, FAKE, FAKE, 8, 0, FAKE, None) == 1 and b"bad dims" in err()
    assert mx(-1, 16, 8, FAKE, FAKE, FAKE, FAKE, 8, 0, FAKE, None) == 1 and b"bad dims" in err()
    assert mx(4, 16, 0, FAKE, FAKE, FAKE, FAKE, 8, 0, FAKE, None) == 1 and b"bad dims" in err()
    assert mx(4, 16, 8, FAKE, FAKE, FAKE, FAKE, 8, 1, FAKE, None) == 1 and b"out_stride" in err()
    assert mx(4, 16, 8, FAKE, FAKE, FAKE, FAKE, 8, 0, None, None) == 1 and b"null pointer" in err()
    assert mx(4, 16, 8, None, FAKE, FAKE, FAKE, 8, 0, FAKE, None) == 1 and b"null pointer" in err()
    assert mx(0, 16, 8, None, None, None, None, 8, 0, None, None) == 0
    assert bw(4, 0, 8, FAKE, 8, 0, FAKE, FAKE, None) == 1 and b"bad dims" in err()
    assert bw(4, 16, 8, FAKE, 7, 0, FAKE, FAKE, None) == 1 and b"gp_stride" in err()
    assert bw(4, 16, 8, FAKE, 8, 0, None, FAKE, None) == 1 and b"null pointer" in err()
    assert bw(4, 16, 8, FAKE, 8, 0, FAKE, None, None) == 1 and b"null pointer" in err()
    assert bw(0, 16, 8, None, 8, 0, None, None, None) == 0
