"""The entry points of the training-mode SA / FP blocks refuse bad dimensions and null pointers with a message before any
CUDA call (so this runs without a GPU); empty batches are no-ops."""
import ctypes

from pn2_b200 import _lib

FAKE = 1 << 20  # a non-null address; validation fails before anything is dereferenced


def _grouped(**over):
    d = dict(kind=_lib.ROWS_GROUPED, order=_lib.ORDER_XYZ_FIRST, b=2, n=64, m=8, k=16, d=5,
             xyz=FAKE, new_xyz=FAKE, feat=FAKE, idx=FAKE)
    d.update(over)
    return _lib.Pn2Rows(**d)


def _interp(**over):
    d = dict(kind=_lib.ROWS_INTERP, b=2, n=64, m=8, d=6, d_skip=3, feat=FAKE, skip=FAKE, idx=FAKE, weight=FAKE)
    d.update(over)
    return _lib.Pn2Rows(**d)


def _fwd(rows, cin, desc, ptrs=FAKE):
    lib = _lib.load()
    return lib.pn2_train_linear_fwd_rows(rows, cin, 16, desc if desc is None else ctypes.byref(desc), ptrs, ptrs, ptrs, ptrs, None)


def _bwd(rows, cin, desc, g_in=None, g_skip=None):
    lib = _lib.load()
    return lib.pn2_train_linear_bwd_rows(rows, cin, 16, ctypes.byref(desc), *([FAKE] * 8), g_in, g_skip, FAKE, None)


def test_row_source_entries_validate_without_gpu():
    err = _lib.load().pn2_last_error
    R = 2 * 8 * 16
    assert _fwd(R, 8, None) == 1 and b"null row source" in err()
    assert _fwd(R, 8, _grouped(kind=7)) == 1 and b"unknown row source kind" in err()
    assert _fwd(R, 8, _grouped(order=2)) == 1 and b"bad grouped source" in err()
    assert _fwd(R, 8, _grouped(k=0)) == 1 and b"bad grouped source" in err()
    assert _fwd(R + 1, 8, _grouped()) == 1 and b"do not match" in err()
    assert _fwd(R, 9, _grouped()) == 1 and b"do not match" in err()
    assert _fwd(R, 8, _grouped(xyz=None)) == 1 and b"null pointer" in err()
    assert _fwd(R, 8, _grouped(feat=None)) == 1 and b"null pointer" in err()       # d > 0 needs features
    assert _fwd(R, 3, _grouped(d=0)) == 1 and b"null pointer" in err()            # d == 0 takes none
    assert _fwd(R, 8, _grouped(), ptrs=None) == 1 and b"null pointer" in err()
    assert _fwd(-1, 8, _grouped()) == 1 and b"bad dims" in err()
    assert _fwd(0, 8, None) == 0                                                    # no rows: no-op
    assert _fwd(128, 9, _interp(idx=None)) == 1 and b"null pointer" in err()       # m > 1 needs the 3-NN
    assert _fwd(128, 9, _interp(skip=None)) == 1 and b"null pointer" in err()
    assert _fwd(128, 10, _interp()) == 1 and b"do not match" in err()
    assert _fwd(128, 9, _interp(d=0, d_skip=9)) == 1 and b"bad interpolated source" in err()
    assert _bwd(R, 8, _grouped(), g_skip=FAKE) == 1 and b"g_skip" in err()
    assert _bwd(128, 6, _interp(d_skip=0, skip=None), g_skip=FAKE) == 1 and b"g_skip" in err()   # no skip columns
    assert _bwd(R, 8, _grouped(idx=None)) == 1 and b"null pointer" in err()
    assert _bwd(R + 16, 8, _grouped()) == 1 and b"do not match" in err()
    assert _bwd(128, 9, _interp(weight=None)) == 1 and b"null pointer" in err()


def test_pooling_and_scatter_entries_validate_without_gpu():
    lib = _lib.load()
    err = lib.pn2_last_error
    assert lib.pn2_train_bn_relu_max(4, 257, 8, FAKE, FAKE, FAKE, FAKE, 8, 0, FAKE, None) == 1 and b"k <= 256" in err()
    assert lib.pn2_train_bn_relu_max(4, 16, 0, FAKE, FAKE, FAKE, FAKE, 8, 0, FAKE, None) == 1 and b"bad dims" in err()
    assert lib.pn2_train_bn_relu_max(4, 16, 8, FAKE, FAKE, FAKE, FAKE, 8, 1, FAKE, None) == 1 and b"out_stride" in err()
    assert lib.pn2_train_bn_relu_max(4, 16, 8, FAKE, FAKE, FAKE, FAKE, 8, 0, None, None) == 1 and b"null pointer" in err()
    assert lib.pn2_train_bn_relu_max(0, 16, 8, None, None, None, None, 8, 0, None, None) == 0
    assert lib.pn2_train_max_bwd(4, 0, 8, FAKE, 8, 0, FAKE, FAKE, None) == 1 and b"bad dims" in err()
    assert lib.pn2_train_max_bwd(4, 16, 8, FAKE, 7, 0, FAKE, FAKE, None) == 1 and b"gp_stride" in err()
    assert lib.pn2_train_max_bwd(4, 16, 8, FAKE, 8, 0, None, FAKE, None) == 1 and b"null pointer" in err()
    assert lib.pn2_train_max_bwd(0, 16, 8, None, 8, 0, None, None, None) == 0
    sc = lib.pn2_scatter_rows_det_cl
    assert sc(1, 4, 8, 10, 3, FAKE, 4, 0, FAKE, FAKE, FAKE, FAKE, None) == 1 and b"multiple of div" in err()
    assert sc(1, 4, 8, 9, 2, FAKE, 4, 0, FAKE, FAKE, FAKE, FAKE, None) == 1 and b"bad dims" in err()
    assert sc(1, 4, 8, 9, 3, FAKE, 6, 3, FAKE, FAKE, FAKE, FAKE, None) == 1 and b"row_stride" in err()
    assert sc(1, 4, 8, 9, 3, None, 4, 0, FAKE, FAKE, FAKE, FAKE, None) == 1 and b"null pointer" in err()
    assert sc(1, 4, 8, 9, 3, FAKE, 4, 0, FAKE, FAKE, FAKE, None, None) == 1 and b"null pointer" in err()
    assert sc(0, 4, 8, 9, 3, None, 4, 0, None, None, None, None, None) == 0
    assert sc(2, 0, 8, 9, 3, None, 0, 0, None, None, None, None, None) == 0   # no feature channels: nothing to write
