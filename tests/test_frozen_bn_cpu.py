"""The running-statistics BatchNorm entries (pn2_train_bn_running, pn2_train_bn_running_bwd_coeffs) and the statistics-free
training forward (stats == NULL) refuse bad input with a message before any CUDA call, so this runs without a GPU;
empty row sets are no-ops."""
import ctypes

from pn2_b200 import _lib

FAKE = 1 << 20  # a non-null address; validation fails before anything is dereferenced


def test_running_statistics_entries_validate_without_gpu():
    lib = _lib.load()
    err = lib.pn2_last_error
    run, bwd = lib.pn2_train_bn_running, lib.pn2_train_bn_running_bwd_coeffs
    ok = [FAKE] * 4
    assert run(0, *ok, 1e-5, FAKE, FAKE, FAKE, None) == 1 and b"bad dims" in err()
    assert run(-3, *ok, 1e-5, FAKE, FAKE, FAKE, None) == 1 and b"bad dims" in err()
    assert run(8, *ok, -1.0, FAKE, FAKE, FAKE, None) == 1 and b"eps" in err()
    for i in range(4):  # running_mean, running_var, gamma, beta
        args = list(ok)
        args[i] = None
        assert run(8, *args, 1e-5, FAKE, FAKE, FAKE, None) == 1 and b"null pointer" in err()
    for i in range(3):  # scale, shift, mean_rstd
        outs = [FAKE] * 3
        outs[i] = None
        assert run(8, *ok, 1e-5, *outs, None) == 1 and b"null pointer" in err()
    assert bwd(0, *([FAKE] * 7), None) == 1 and b"bad dims" in err()
    for i in range(7):  # sums, mean_rstd, scale, coef, dgamma, dbeta, dbias
        args = [FAKE] * 7
        args[i] = None
        assert bwd(8, *args, None) == 1 and b"null pointer" in err()


def test_statistics_free_forward_validates_without_gpu():
    """stats == NULL is accepted (nothing is launched for zero rows); every other pointer is still required, and the
    act_in pair must be both NULL or both set."""
    lib = _lib.load()
    err = lib.pn2_last_error
    fwd = lib.pn2_train_linear_fwd
    assert fwd(0, 8, 16, FAKE, None, None, FAKE, FAKE, FAKE, None, None) == 0
    assert fwd(-1, 8, 16, FAKE, None, None, FAKE, FAKE, FAKE, None, None) == 1 and b"bad dims" in err()
    assert fwd(64, 0, 16, FAKE, None, None, FAKE, FAKE, FAKE, None, None) == 1 and b"bad dims" in err()
    assert fwd(64, 8, 16, FAKE, FAKE, None, FAKE, FAKE, FAKE, None, None) == 1 and b"null pointer" in err()   # mismatched pair
    assert fwd(64, 8, 16, FAKE, None, FAKE, FAKE, FAKE, FAKE, None, None) == 1 and b"null pointer" in err()
    for i in (0, 3, 4, 5):  # x, w, bias, z
        args = [FAKE, None, None, FAKE, FAKE, FAKE]
        args[i] = None
        assert fwd(64, 8, 16, *args, None, None) == 1 and b"null pointer" in err()
    assert fwd(64, 8, 16, FAKE + 4, None, None, FAKE, FAKE, FAKE, None, None) == 1 and b"alignment" in err()

    rows = _lib.Pn2Rows(kind=_lib.ROWS_GROUPED, order=_lib.ORDER_XYZ_FIRST, b=2, n=64, m=8, k=16, d=5, xyz=FAKE, new_xyz=FAKE,
                        feat=FAKE, idx=FAKE)
    fwd_rows = lib.pn2_train_linear_fwd_rows
    R = 2 * 8 * 16
    assert fwd_rows(0, 8, 16, None, FAKE, FAKE, FAKE, None, None) == 0
    assert fwd_rows(R, 8, 16, None, FAKE, FAKE, FAKE, None, None) == 1 and b"null row source" in err()
    assert fwd_rows(R + 1, 8, 16, ctypes.byref(rows), FAKE, FAKE, FAKE, None, None) == 1 and b"do not match" in err()
    for i in range(3):  # w, bias, z
        args = [FAKE] * 3
        args[i] = None
        assert fwd_rows(R, 8, 16, ctypes.byref(rows), *args, None, None) == 1 and b"null pointer" in err()
    allrows = _lib.Pn2Rows(kind=_lib.ROWS_ALL, b=2, n=100, d=5, xyz=FAKE, feat=None)
    assert fwd_rows(200, 8, 16, ctypes.byref(allrows), FAKE, FAKE, FAKE, None, None) == 1 and b"null pointer" in err()
