"""Every training-mode MLP entry point of csrc/train_mlp.cu called on its own through _lib.call and compared with its
float64 restatement in oracle/train_mlp_ref.py, at the shapes where the kernels branch: ragged widths and row counts,
each output-tile width, the grid-stride loop, NULL outputs, misaligned pointers, ties in the poolings, and BatchNorm
statistics of channels whose mean is far larger than their spread.

Outputs are pre-filled with NaN (or a sentinel), so every element must be written and nothing outside the output's
columns may be touched.  GEMM outputs are held to an element-wise bound C 2^-24 sqrt(K) (|A| |B|); everything
elementwise to the float64 value rounded once (one ulp where the reference double-rounds an fma)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import train_mlp_ref as ref
from pn2_b200 import _lib
from pn2_b200._lib import ptr

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
# GEMM bound constant.  A k-sequential fp32 fma chain has a worst-case error of K u sum |a b|, but its roundings are
# independent, so the error grows like sqrt(K) u sum |a b| with a constant below 1; the operand's own fp32 formation
# (act_in's fma, the three-term interpolation, dz = ca dy + cb + cc z with two fmas) adds at most 2 u sum |a b|, which
# sqrt(K) >= 1 covers.  4 leaves room for both without hiding a wrong element (an off-by-one row or column is O(1)).
C_GEMM = 4.0
C_SUM = 4.0        # the same for the BatchNorm reductions, with R rows in place of K
# the per-channel coefficient kernels round float64 expressions whose last bits depend on the operation order
ULP_COEF = 2


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _nan(shape, dev):
    return torch.full(shape if isinstance(shape, tuple) else (shape,), float("nan"), dtype=torch.float32, device=dev)


def _st():
    return _lib.stream_ptr()


class _Pin:
    """Device pointers of numpy arrays copied to the GPU, the copies kept alive by the test: a temporary freed as soon as
    its pointer is taken could be handed to the next argument by the caching allocator before the kernel runs."""

    def __init__(self, dev):
        self.dev, self.held = dev, []

    def __call__(self, a):
        if a is None:
            return None
        t = _t(a, self.dev)
        self.held.append(t)
        return ptr(t)


def _gemm_close(got, want, mag, K, what):
    """|got - want| <= C 2^-24 sqrt(K) mag element-wise, mag = |A| |B| (+ |bias|)."""
    got = got.detach().cpu().numpy().astype(np.float64)
    assert np.isfinite(got).all(), "%s: unwritten (NaN) elements" % what
    bound = C_GEMM * U * np.sqrt(K) * mag + 1e-30
    ratio = float((np.abs(got - want) / bound).max())
    print("%s: worst error / bound = %.3f" % (what, ratio))
    assert ratio <= 1.0, "%s: error %.3f x the bound C 2^-24 sqrt(K) |A||B|" % (what, ratio)


def _ulp_close(got, want, what, ulps=1):
    got = got.detach().cpu().numpy() if torch.is_tensor(got) else np.asarray(got)
    want = np.asarray(want, dtype=np.float32)
    assert got.shape == want.shape, what
    tol = ulps * np.spacing(np.abs(want))
    assert (np.abs(got.astype(np.float64) - want.astype(np.float64)) <= tol).all(), "%s: more than %d ulp" % (what, ulps)


def _var_check(stats, z, what):
    """stats = (sum z, sum z^2) of the kernel's own z: the variance they give within 1e-5 relative, sum z within the
    reduction bound.  A constant channel's variance must come out 0 to the square of its fp32 rounding."""
    s = stats.cpu().numpy()
    z = z.cpu().numpy().astype(np.float64)
    R = z.shape[0]
    s1, var = z.sum(0), z.var(0)
    assert (np.abs(s[0] - s1) <= C_SUM * U * np.sqrt(R) * np.abs(z).sum(0) + 1e-300).all(), "%s: sum z" % what
    got = s[1] / R - (s[0] / R) ** 2
    mean2 = (s1 / R) ** 2
    tol = np.where(var > 0, 1e-5 * var, 0.0) + 1e-12 * mean2
    rel = np.abs(got - var) / np.maximum(var, 1e-300)
    print("%s: worst variance relative error %.3e" % (what, float(rel[var > 0].max()) if (var > 0).any() else 0.0))
    assert (np.abs(got - var) <= tol).all(), "%s: variance from stats off by %s relative" % (what, rel.max())


def _linear_fwd(dev, x, w, b, scale=None, shift=None, stats=True):
    R, cin = x.shape
    cout = w.shape[0]
    z = _nan((R, cout), dev)
    st = torch.zeros((2, cout), dtype=torch.float64, device=dev) if stats else None
    _lib.call("pn2_train_linear_fwd", R, cin, cout, ptr(x), ptr(scale), ptr(shift), ptr(w), ptr(b), ptr(z), ptr(st), _st())
    return z, st


@pytest.mark.parametrize("stats", [True, False])
@pytest.mark.parametrize("R,cin,cout,act", [(1, 3, 5, False), (129, 7, 33, True), (4109, 131, 64, False), (777, 515, 130, True),
                                            (300, 1536, 512, False), (50000, 16, 24, False)])
def test_linear_fwd(dev, R, cin, cout, act, stats):
    rng = np.random.default_rng(R + cin)
    x = rng.normal(size=(R, cin)).astype(np.float32)
    w = (rng.normal(size=(cout, cin)) / np.sqrt(cin)).astype(np.float32)
    b = rng.normal(size=cout).astype(np.float32)
    sc = rng.uniform(0.5, 1.5, cin).astype(np.float32) if act else None
    sh = rng.normal(0, 0.3, cin).astype(np.float32) if act else None
    z, st = _linear_fwd(dev, _t(x, dev), _t(w, dev), _t(b, dev), None if sc is None else _t(sc, dev), None if sh is None else _t(sh, dev), stats)
    want, _, a = ref.linear_fwd(x, w, b, sc, sh)
    _gemm_close(z, want, np.abs(a).astype(np.float64) @ np.abs(w).T.astype(np.float64) + np.abs(b), cin + 1, "z (%d,%d,%d)" % (R, cin, cout))
    if stats:
        _var_check(st, z, "stats (%d,%d,%d)" % (R, cin, cout))


@pytest.mark.parametrize("cout", [8, 40, 100])   # one output tile width each: NT 32, 64, 128
def test_linear_fwd_statistics_of_conditioned_channels(dev, cout):
    """Channels with mean / std = 30, 100, 1000 (bias offsets on unit-variance z) and one constant channel (zero weight
    row): the variance from stats must hold 1e-5 relative, as it does for centred channels."""
    R, cin = 16384, 16
    rng = np.random.default_rng(cout)
    x = rng.normal(size=(R, cin)).astype(np.float32)
    w = rng.normal(size=(cout, cin))
    w = (w / np.linalg.norm(w, axis=1, keepdims=True)).astype(np.float32)
    w[cout // 2] = 0.0
    b = np.array([(30.0, 100.0, 1000.0, -100.0)[j % 4] for j in range(cout)], dtype=np.float32)
    b[cout // 2] = 0.37
    z, st = _linear_fwd(dev, _t(x, dev), _t(w, dev), _t(b, dev))
    _var_check(st, z, "conditioned stats cout=%d" % cout)


@pytest.mark.parametrize("rows,c", [(5, 1), (5, 31), (4096, 33), (3000, 300), (16384, 31)])
def test_bn_bwd_reduce(dev, rows, c):
    """sum dy and sum dy z against float64; S2 - mean S1 within C 2^-24 sqrt(R) sum |dy| |z - mean| at mean / std up to
    1e4 (every channel is conditioned: z = ratio + N(0, 1))."""
    P = _Pin(dev)
    rng = np.random.default_rng(rows * 7 + c)
    ratio = np.array([(0.0, 30.0, 1e3, 1e4, -1e2)[j % 5] for j in range(c)])
    z = (ratio + rng.normal(size=(rows, c))).astype(np.float32)
    g = rng.normal(size=(rows, c)).astype(np.float32)
    z64 = z.astype(np.float64)
    mean = z64.mean(0)
    rstd = 1.0 / np.sqrt(z64.var(0) + 1e-5)
    gamma = rng.uniform(0.5, 1.5, c)
    beta = rng.normal(0, 0.2, c)
    scale, shift = (gamma * rstd).astype(np.float32), (beta - mean * gamma * rstd).astype(np.float32)
    sums = torch.zeros((2, c), dtype=torch.float64, device=dev)
    _lib.call("pn2_train_bn_bwd_reduce", rows, c, P(g), P(z), P(scale), P(shift),
              ptr(sums), _st())
    S1, S2 = sums.cpu().numpy()
    dy = np.where(ref.relu_open(z, scale, shift), g.astype(np.float64), 0.0)
    w1, w2 = ref.bwd_reduce(g, z, scale, shift)
    assert (np.abs(S1 - w1) <= C_SUM * U * np.sqrt(rows) * np.abs(dy).sum(0) + 1e-300).all(), "S1"
    want = (dy * (z64 - mean)).sum(0)
    bound = C_SUM * U * np.sqrt(rows) * (np.abs(dy) * np.abs(z64 - mean)).sum(0) + 1e-300
    err = np.abs((S2 - mean * S1) - want)
    print("bn_bwd_reduce rows=%d c=%d: worst (S2 - mean S1) error / bound = %.3f" % (rows, c, float((err / bound).max())))
    assert (err <= bound).all(), "S2 - mean S1 off by %s x the bound (ratios %s)" % ((err / bound).max(), ratio[np.argmax(err / bound)])


@pytest.mark.parametrize("rows,running", [(1, True), (2, True), (2, False), (1000, True)])
def test_bn_finalize(dev, rows, running):
    P = _Pin(dev)
    c = 37
    rng = np.random.default_rng(rows)
    z = (rng.normal(size=(rows, c)) + 3.0).astype(np.float64)
    z[:, 5] = 2.5                                                           # constant channel
    stats = np.stack([z.sum(0), (z * z).sum(0)])
    stats[1, 6] = stats[0, 6] ** 2 / rows * (1 - 1e-9)                      # E[z^2] < mean^2: the variance clamp
    gamma, beta = rng.uniform(0.5, 1.5, c).astype(np.float32), rng.normal(size=c).astype(np.float32)
    rm, rv = rng.normal(size=c).astype(np.float32), rng.uniform(0.5, 2, c).astype(np.float32)
    scale, shift = _nan(c, dev), _nan(c, dev)
    mr = torch.full((2, c), float("nan"), dtype=torch.float64, device=dev)
    trm, trv = (_t(rm, dev), _t(rv, dev)) if running else (None, None)
    _lib.call("pn2_train_bn_finalize", rows, c, P(stats), P(gamma), P(beta), 1e-5, 0.1, ptr(scale),
              ptr(shift), ptr(mr), ptr(trm), ptr(trv), _st())
    wsc, wsh, wmr, wrm, wrv = ref.finalize(rows, stats, gamma, beta, 1e-5, 0.1, rm if running else None, rv if running else None)
    _ulp_close(scale, wsc, "scale", ULP_COEF)
    _ulp_close(shift, wsh, "shift", ULP_COEF)
    got = mr.cpu().numpy()
    np.testing.assert_allclose(got[0], wmr[0], rtol=1e-15)
    # var = E[z^2] - mean^2 in float64 cancels; its last bits depend on fma contraction, and rstd moves by
    # d var / (2 (var + eps)): allow a few float64 ulps of E[z^2] through that derivative
    var = np.maximum(stats[1] / rows - wmr[0] ** 2, 0.0)
    np.testing.assert_array_less(np.abs(got[1] - wmr[1]), wmr[1] * (1e-15 + 4 * 2.0 ** -52 * (stats[1] / rows) / (2 * (var + 1e-5))))
    assert mr[1, 6].item() == pytest.approx(1 / np.sqrt(1e-5), rel=1e-14)
    if running:
        _ulp_close(trm, wrm, "running_mean", ULP_COEF)
        _ulp_close(trv, wrv, "running_var", ULP_COEF)


def test_bn_coefficient_kernels(dev):
    P = _Pin(dev)
    c, rows = 45, 777
    rng = np.random.default_rng(3)
    sums = np.stack([rng.normal(size=c) * 10, rng.normal(size=c) * 100])
    mr = np.stack([rng.normal(size=c), rng.uniform(0.5, 2, c)])
    gamma, beta = rng.uniform(0.5, 1.5, c).astype(np.float32), rng.normal(size=c).astype(np.float32)
    coef, dg, db = _nan((3, c), dev), _nan(c, dev), _nan(c, dev)
    _lib.call("pn2_train_bn_bwd_coeffs", rows, c, P(sums), P(mr), P(gamma), ptr(coef), ptr(dg), ptr(db), _st())
    wc, wdg, wdb = ref.bwd_coeffs(rows, sums, mr, gamma)
    _ulp_close(coef, wc, "coef", ULP_COEF)
    _ulp_close(dg, wdg, "dgamma", ULP_COEF)
    _ulp_close(db, wdb, "dbeta", ULP_COEF)
    rm, rv = rng.normal(size=c).astype(np.float32), rng.uniform(0.5, 2, c).astype(np.float32)
    sc, sh = _nan(c, dev), _nan(c, dev)
    mr2 = torch.full((2, c), float("nan"), dtype=torch.float64, device=dev)
    _lib.call("pn2_train_bn_running", c, P(rm), P(rv), P(gamma), P(beta), 1e-3, ptr(sc), ptr(sh),
              ptr(mr2), _st())
    wsc, wsh, wmr = ref.running(rm, rv, gamma, beta, 1e-3)
    _ulp_close(sc, wsc, "running scale", ULP_COEF)
    _ulp_close(sh, wsh, "running shift", ULP_COEF)
    np.testing.assert_allclose(mr2.cpu().numpy(), wmr, rtol=1e-14)
    coef2, dg2, db2, dbias = _nan((3, c), dev), _nan(c, dev), _nan(c, dev), _nan(c, dev)
    _lib.call("pn2_train_bn_running_bwd_coeffs", c, P(sums), ptr(mr2), ptr(sc), ptr(coef2), ptr(dg2), ptr(db2), ptr(dbias), _st())
    wc2, wdg2, wdb2, wdbias = ref.running_bwd_coeffs(sums, wmr, wsc)
    _ulp_close(coef2, wc2, "running coef", ULP_COEF)
    _ulp_close(dg2, wdg2, "running dgamma", ULP_COEF)
    _ulp_close(db2, wdb2, "running dbeta", ULP_COEF)
    _ulp_close(dbias, wdbias, "running dbias", ULP_COEF)


@pytest.mark.parametrize("c,offset", [(64, 0), (33, 0), (64, 1)])
def test_bn_relu(dev, c, offset):
    P = _Pin(dev)
    rows = 1000
    rng = np.random.default_rng(c + offset)
    z = rng.normal(size=(rows, c)).astype(np.float32)
    sc, sh = rng.uniform(-1, 1.5, c).astype(np.float32), rng.normal(size=c).astype(np.float32)
    buf = _nan((rows * c + offset,), dev)
    out = buf[offset:]                            # offset 1: a pointer 4 bytes off 16-byte alignment -> the scalar kernel
    zb = torch.zeros(rows * c + offset, device=dev)
    zb[offset:] = _t(z.reshape(-1), dev)
    _lib.call("pn2_train_bn_relu", rows, c, ptr(zb[offset:]), P(sc), P(sh), ptr(out), _st())
    _ulp_close(out.view(rows, c), ref.bn_act(z, sc, sh), "bn_relu")
    if offset:
        assert torch.isnan(buf[0]), "bn_relu wrote in front of its output"


def _pool_inputs(rng, groups, k, c):
    z = rng.normal(size=(groups * k, c)).astype(np.float32)
    zg = z.reshape(groups, k, c)
    if k > 1:
        zg[0, k - 1] = zg[0].max(0) + 1.0              # the maximum on the last row (arg k - 1)
        if groups > 1:
            zg[1, k // 2] = zg[1, k - 1] = zg[1].max(0) + 0.5   # exact ties at a non-zero value: the first row wins
    sc = np.abs(rng.normal(size=c)).astype(np.float32) + 0.5
    sh = rng.normal(size=c).astype(np.float32)
    sh[c // 2] = -1e6                                  # an all-zero channel: arg 0
    return z, sc, sh


@pytest.mark.parametrize("k", [1, 3, 255, 256])
@pytest.mark.parametrize("c", [1, 33])
def test_bn_relu_max_and_max_bwd(dev, k, c):
    P = _Pin(dev)
    groups, stride, off = 37, c + 7, 5
    rng = np.random.default_rng(k * 100 + c)
    z, sc, sh = _pool_inputs(rng, groups, k, c)
    out = _nan((groups, stride), dev)
    arg = torch.full((groups, c), 0xAB, dtype=torch.uint8, device=dev)
    _lib.call("pn2_train_bn_relu_max", groups, k, c, P(z), P(sc), P(sh), ptr(out), stride, off, ptr(arg), _st())
    want, warg = ref.max_pool(ref.bn_act(z, sc, sh), groups, k)
    _ulp_close(out[:, off:off + c], want, "pooled")
    assert torch.isnan(out[:, :off]).all() and torch.isnan(out[:, off + c:]).all(), "wrote outside out_offset"
    assert np.array_equal(arg.cpu().numpy(), warg), "arg"
    gp = rng.normal(size=(groups, stride)).astype(np.float32)
    g = _nan((groups * k, c), dev)
    _lib.call("pn2_train_max_bwd", groups, k, c, P(gp), stride, off, ptr(arg), ptr(g), _st())
    assert np.array_equal(g.cpu().numpy(), ref.max_bwd(gp[:, off:off + c], warg, k)), "max_bwd"


@pytest.mark.parametrize("k", [1, 127, 128, 129, 200000])
def test_bn_relu_max_all_and_max_bwd_all(dev, k):
    P = _Pin(dev)
    groups, c, stride, off = 2, 33, 40, 3
    rng = np.random.default_rng(k)
    z, sc, sh = _pool_inputs(rng, groups, k, c)
    if k > 128:   # equal maxima in two row ranges of at least 128 rows: rows 3 and k - 1 of group 0
        zg = z.reshape(groups, k, c)
        zg[0, 3] = zg[0, k - 1]
    out = _nan((groups, stride), dev)
    arg = torch.full((groups, c), -7, dtype=torch.int32, device=dev)
    _lib.call("pn2_train_bn_relu_max_all", groups, k, c, P(z), P(sc), P(sh), ptr(out), stride, off,
              ptr(arg), _st())
    want, warg = ref.max_pool(ref.bn_act(z, sc, sh), groups, k)
    _ulp_close(out[:, off:off + c], want, "pooled")
    assert torch.isnan(out[:, :off]).all() and torch.isnan(out[:, off + c:]).all(), "wrote outside out_offset"
    assert np.array_equal(arg.cpu().numpy(), warg), "arg"
    assert (warg[:, c // 2] == 0).all() and (k <= 128 or (warg[0] == 3).sum() >= c - 1)
    gp = rng.normal(size=(groups, stride)).astype(np.float32)
    g = _nan((groups * k, c), dev)
    _lib.call("pn2_train_max_bwd_all", groups, k, c, P(gp), stride, off, ptr(arg), ptr(g), _st())
    assert np.array_equal(g.cpu().numpy(), ref.max_bwd(gp[:, off:off + c], warg, k)), "max_bwd_all"


def test_pooling_over_no_groups_writes_nothing(dev):
    out = _nan((1, 8), dev)
    arg = torch.full((1, 8), -7, dtype=torch.int32, device=dev)
    _lib.call("pn2_train_bn_relu_max_all", 0, 16, 8, ptr(out), ptr(out), ptr(out), ptr(out), 8, 0, ptr(arg), _st())
    _lib.call("pn2_train_max_bwd_all", 0, 16, 8, ptr(out), 8, 0, ptr(arg), ptr(out), _st())
    torch.cuda.synchronize()
    assert torch.isnan(out).all() and (arg == -7).all()


def _bwd_inputs(rng, R, cout):
    g = rng.normal(size=(R, cout)).astype(np.float32)
    z = rng.normal(size=(R, cout)).astype(np.float32)
    sc = rng.uniform(0.5, 1.5, cout).astype(np.float32)
    sh = rng.normal(0, 0.3, cout).astype(np.float32)
    coef = np.stack([rng.uniform(0.5, 1.5, cout), rng.normal(size=cout) * 0.1, rng.normal(size=cout) * 0.1]).astype(np.float32)
    dzv = ref.dz(g, z, sc, sh, coef)
    dy = np.where(ref.relu_open(z, sc, sh), g, 0).astype(np.float64)
    dmag = np.abs(coef[0] * dy) + np.abs(coef[1]) + np.abs(coef[2] * z.astype(np.float64))  # the operand's fp32 terms
    return (g, z, sc, sh, coef), dzv, dmag


def _check_bwd(got_in, got_w, a, w, dzv, dmag, what, g_cols=None):
    """g_in = dz W (K = cout) on the columns g_cols of the operand; dW = dz^T a (K = rows)."""
    want_in, want_w = ref.linear_bwd(a, w, dzv)
    mag_in = dmag @ np.abs(w).astype(np.float64)
    if got_in is not None:
        cols = slice(None) if g_cols is None else g_cols
        _gemm_close(got_in, want_in[:, cols], mag_in[:, cols], w.shape[0], "g_in %s" % what)
    _gemm_close(got_w, want_w, dmag.T @ np.abs(a).astype(np.float64), a.shape[0], "dW %s" % what)


@pytest.mark.parametrize("R,cin,cout,act,need_in", [(100, 20, 30, False, True), (5000, 60, 50, True, True), (3000, 130, 120, False, True),
                                                    (20000, 16, 200, True, True), (700, 131, 64, False, False), (129, 3, 5, False, True)])
def test_linear_bwd(dev, R, cin, cout, act, need_in):
    P = _Pin(dev)
    rng = np.random.default_rng(R + cin + cout)
    x = rng.normal(size=(R, cin)).astype(np.float32)
    w = (rng.normal(size=(cout, cin)) / np.sqrt(cin)).astype(np.float32)
    isc = rng.uniform(0.5, 1.5, cin).astype(np.float32) if act else None
    ish = rng.normal(0, 0.3, cin).astype(np.float32) if act else None
    (g, z, sc, sh, coef), dzv, dmag = _bwd_inputs(rng, R, cout)
    g_in = _nan((R, cin), dev) if need_in else None
    dW = torch.zeros((cout, cin), device=dev)
    tc = _t(coef, dev)
    _lib.call("pn2_train_linear_bwd", R, cin, cout, P(x), P(isc),
              P(ish), P(np.ascontiguousarray(w.T)), P(g), P(z),
              P(sc), P(sh), ptr(tc[0]), ptr(tc[1]), ptr(tc[2]), ptr(g_in), ptr(dW), _st())
    a = x if isc is None else ref.bn_act(x, isc, ish)
    _check_bwd(g_in, dW, a, w, dzv, dmag, "(%d,%d,%d)" % (R, cin, cout))


def _rows_fwd_bwd(dev, desc, rows, a, cout, rng, g_in_shape=None, g_skip_shape=None, g_cols=None, skip_cols=None):
    """forward through the row source against ref.linear_fwd on its materialised rows `a`, then the backward."""
    P = _Pin(dev)
    cin = a.shape[1]
    w = (rng.normal(size=(cout, cin)) / np.sqrt(cin)).astype(np.float32)
    b = rng.normal(size=cout).astype(np.float32)
    z = _nan((rows, cout), dev)
    st = torch.zeros((2, cout), dtype=torch.float64, device=dev)
    tw = _t(w, dev)
    _lib.call("pn2_train_linear_fwd_rows", rows, cin, cout, ctypes.byref(desc), ptr(tw), P(b), ptr(z), ptr(st), _st())
    want, _, _ = ref.linear_fwd(a, w, b)
    _gemm_close(z, want, np.abs(a).astype(np.float64) @ np.abs(w).T.astype(np.float64) + np.abs(b), cin + 1, "z rows")
    _var_check(st, z, "rows stats")
    (g, zz, sc, sh, coef), dzv, dmag = _bwd_inputs(rng, rows, cout)
    g_in = _nan(g_in_shape, dev) if g_in_shape else None
    g_skip = _nan(g_skip_shape, dev) if g_skip_shape else None
    dW = torch.zeros((cout, cin), device=dev)
    tc = _t(coef, dev)
    _lib.call("pn2_train_linear_bwd_rows", rows, cin, cout, ctypes.byref(desc), P(np.ascontiguousarray(w.T)), P(g),
              P(zz), P(sc), P(sh), ptr(tc[0]), ptr(tc[1]), ptr(tc[2]), ptr(g_in), ptr(g_skip), ptr(dW), _st())
    _check_bwd(None if g_in is None else g_in.reshape(rows, -1), dW, a, w, dzv, dmag, "rows", g_cols)
    if g_skip is not None:
        want_in, _ = ref.linear_bwd(a, w, dzv)
        mag = dmag @ np.abs(w).astype(np.float64)
        _gemm_close(g_skip.reshape(rows, -1), want_in[:, skip_cols], mag[:, skip_cols], cout, "g_skip rows")


@pytest.mark.parametrize("k", [1, 32, 128])
@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("d", [0, 6, 13, 32])
def test_grouped_rows(dev, d, order, k):
    B, N, m, cout = 2, 300, 24, 40
    rng = np.random.default_rng(d * 1000 + order * 100 + k)
    xyz = (rng.normal(size=(B, N, 3)) * 2 + 5).astype(np.float32)
    new_xyz = (xyz[:, :m] + rng.normal(size=(B, m, 3)) * 0.1).astype(np.float32)
    feat = rng.normal(size=(B, N, d)).astype(np.float32) if d else None
    idx = rng.integers(0, N, size=(B, m, k)).astype(np.int32)
    idx[:, -1, -1] = N - 1
    rows = B * m * k
    desc = _lib.Pn2Rows(kind=_lib.ROWS_GROUPED, order=order, b=B, n=N, m=m, k=k, d=d)
    keep = [_t(xyz, dev), _t(new_xyz, dev), None if feat is None else _t(feat, dev), _t(idx, dev)]
    desc.xyz, desc.new_xyz, desc.feat, desc.idx = ptr(keep[0]), ptr(keep[1]), ptr(keep[2]), ptr(keep[3])
    a = ref.grouped_rows(xyz, new_xyz, feat, idx, order)
    _rows_fwd_bwd(dev, desc, rows, a, cout, rng, g_in_shape=(rows, 3 + d))


@pytest.mark.parametrize("g_in,g_skip", [(True, True), (True, False), (False, True), (False, False)])
@pytest.mark.parametrize("d", [33, 64])
@pytest.mark.parametrize("d_skip,m", [(0, 50), (5, 50), (8, 50), (5, 1)])
def test_interpolated_rows(dev, d_skip, m, d, g_in, g_skip):
    if g_skip and d_skip == 0:
        pytest.skip("no skip columns: g_skip is refused (tested without a GPU)")
    B, n, cout = 2, 700, 48
    rng = np.random.default_rng(d_skip * 100 + m + d)
    feat = rng.normal(size=(B, m, d)).astype(np.float32)
    skip = rng.normal(size=(B, n, d_skip)).astype(np.float32) if d_skip else None
    idx = rng.integers(0, m, size=(B, n, 3)).astype(np.int32)
    idx[0, 0] = m - 1
    w = rng.uniform(0, 1, size=(B, n, 3)).astype(np.float32)
    w = (w / w.sum(-1, keepdims=True)).astype(np.float32)
    rows = B * n
    keep = [_t(feat, dev), None if skip is None else _t(skip, dev), _t(idx, dev), _t(w, dev)]
    desc = _lib.Pn2Rows(kind=_lib.ROWS_INTERP, b=B, n=n, m=m, d=d, d_skip=d_skip, feat=ptr(keep[0]), skip=ptr(keep[1]),
                        idx=ptr(keep[2]) if m > 1 else None, weight=ptr(keep[3]) if m > 1 else None)
    a = ref.interp_rows(skip, feat, idx if m > 1 else None, w if m > 1 else None, n)
    _rows_fwd_bwd(dev, desc, rows, a, cout, rng, g_in_shape=(rows, d) if g_in else None, g_skip_shape=(rows, d_skip) if g_skip else None,
                  g_cols=slice(d_skip, None), skip_cols=slice(0, d_skip))


@pytest.mark.parametrize("d,N", [(0, 1000), (5, 1000), (64, 1000), (5, 1)])
def test_all_rows(dev, d, N):
    B, cout = 3, 70
    rng = np.random.default_rng(d + N)
    xyz = (rng.normal(size=(B, N, 3)) + 4).astype(np.float32)
    feat = rng.normal(size=(B, N, d)).astype(np.float32) if d else None
    keep = [_t(xyz, dev), None if feat is None else _t(feat, dev)]
    desc = _lib.Pn2Rows(kind=_lib.ROWS_ALL, b=B, n=N, d=d, xyz=ptr(keep[0]), feat=ptr(keep[1]))
    a = ref.all_rows(xyz, feat)
    _rows_fwd_bwd(dev, desc, B * N, a, cout, rng, g_in_shape=(B * N, d) if d else None, g_cols=slice(3, None))

