"""Float64 restatement of every training-mode MLP entry point of include/pn2_abi.h (csrc/train_mlp.cu), one function per
entry point (TEST INFRASTRUCTURE ONLY).

Each function takes the fp32 arrays the kernel receives and returns what the contract says it computes, in float64
unless the contract stores fp32 (then the fp32 value the kernel must store).  Per-element fp32 operations the kernels
perform with one rounding (the act_in / BatchNorm + ReLU fma) are formed exactly in float64 and rounded once to fp32;
that differs from a true fp32 fma by at most one ulp, in the rare case where the float64 sum is itself rounded.
Row sources reuse the C oracle's grouping and three_interpolate (the reference kernels' operation order)."""
import numpy as np

from . import oracle as orc

f32, f64 = np.float32, np.float64


def bn_act(z, scale, shift):
    """relu(fma(z, scale, shift)) per channel of the last axis, fp32 (pn2_train_bn_relu and the act_in operand)."""
    return np.maximum((z.astype(f64) * scale.astype(f64) + shift.astype(f64)).astype(f32), f32(0))


def linear_fwd(x, w, b, in_scale=None, in_shift=None):
    """pn2_train_linear_fwd: z = act_in(x) W^T + b (float64) and stats = (sum z, sum z^2).  -> (z, stats, operand a)"""
    a = x if in_scale is None else bn_act(x, in_scale, in_shift)
    z = a.astype(f64) @ w.astype(f64).T + b.astype(f64)
    return z, np.stack([z.sum(0), (z * z).sum(0)]), a


def grouped_rows(xyz, new_xyz, feat, idx, order):
    """PN2_ROWS_GROUPED: row (b*m + s)*k + j = [xyz[p] - new_xyz[s] | feat[p]] (order PN2_ORDER_XYZ_FIRST = 0) or
    [feat[p] | xyz[p] - new_xyz[s]] (PN2_ORDER_FEAT_FIRST = 1), p = idx[b, s, j]; the centring is one fp32 subtraction."""
    B, S, K = idx.shape
    gx = orc.grouping_operation(xyz.transpose(0, 2, 1), idx).transpose(0, 2, 3, 1)        # (B, S, K, 3)
    cx = (gx - new_xyz[:, :, None, :]).astype(f32)
    parts = [cx]
    if feat is not None and feat.shape[2] > 0:
        gf = orc.grouping_operation(feat.transpose(0, 2, 1), idx).transpose(0, 2, 3, 1)
        parts = [cx, gf] if order == 0 else [gf, cx]
    return np.ascontiguousarray(np.concatenate(parts, -1).reshape(B * S * K, -1), dtype=f32)


def interp_rows(skip, feat, idx, weight, n):
    """PN2_ROWS_INTERP: row b*n + i = [skip[i] | three_interpolate(feat, idx[i], weight[i])]; m == 1 repeats the one
    coarse row (idx / weight unused)."""
    B, m, d = feat.shape
    if m == 1:
        it = np.repeat(feat, n, axis=1)
    else:
        it = orc.three_interpolate(feat.transpose(0, 2, 1), idx, weight).transpose(0, 2, 1)
    parts = [it] if skip is None else [skip, it]
    return np.ascontiguousarray(np.concatenate(parts, -1).reshape(B * n, -1), dtype=f32)


def all_rows(xyz, feat):
    """PN2_ROWS_ALL: row b*n + i = [xyz[i] | feat[i]], not centred."""
    B, N, _ = xyz.shape
    parts = [xyz] if feat is None else [xyz, feat]
    return np.ascontiguousarray(np.concatenate(parts, -1).reshape(B * N, -1), dtype=f32)


def finalize(rows, stats, gamma, beta, eps, momentum, running_mean=None, running_var=None):
    """pn2_train_bn_finalize -> (scale, shift, mean_rstd, running_mean', running_var'): biased variance (clamped at 0)
    for the normalisation, torch's momentum update with the UNBIASED variance for the running estimate."""
    R = float(rows)
    mean = stats[0] / R
    var = np.maximum(stats[1] / R - mean * mean, 0.0)
    rstd = 1.0 / np.sqrt(var + eps)
    g = gamma.astype(f64)
    scale, shift = (g * rstd).astype(f32), (beta.astype(f64) - mean * g * rstd).astype(f32)
    rm = rv = None
    if running_mean is not None:
        unbiased = var.astype(f32).astype(f64) * (R / (R - 1.0 if R > 1.0 else 1.0))
        rm = ((1.0 - momentum) * running_mean.astype(f64) + momentum * mean.astype(f32).astype(f64)).astype(f32)
        rv = ((1.0 - momentum) * running_var.astype(f64) + momentum * unbiased).astype(f32)
    return scale, shift, np.stack([mean, rstd]), rm, rv


def running(running_mean, running_var, gamma, beta, eps):
    """pn2_train_bn_running -> (scale, shift, mean_rstd) of a BatchNorm that normalises with its running statistics."""
    rm = running_mean.astype(f64)
    rstd = 1.0 / np.sqrt(running_var.astype(f64) + eps)
    g = gamma.astype(f64)
    return (g * rstd).astype(f32), (beta.astype(f64) - rm * g * rstd).astype(f32), np.stack([rm, rstd])


def relu_open(z, scale, shift):
    """The backward's ReLU mask [fma(z, scale, shift) > 0] (the same fp32 value as the forward's)."""
    return (z.astype(f64) * scale.astype(f64) + shift.astype(f64)).astype(f32) > 0


def bwd_reduce(g, z, scale, shift):
    """pn2_train_bn_bwd_reduce: sums = (sum dy, sum dy z), dy = g [scale z + shift > 0]."""
    dy = np.where(relu_open(z, scale, shift), g.astype(f64), 0.0)
    return np.stack([dy.sum(0), (dy * z.astype(f64)).sum(0)])


def bwd_coeffs(rows, sums, mean_rstd, gamma):
    """pn2_train_bn_bwd_coeffs -> (coef (3, c) = ca | cb | cc, dgamma, dbeta), fp32 as stored."""
    S1, S2 = sums
    mean, rstd = mean_rstd
    g = gamma.astype(f64)
    t = S2 - mean * S1
    ca = g * rstd
    cc = -g * rstd ** 3 * t / float(rows)
    cb = -ca * S1 / float(rows) - cc * mean
    return np.stack([ca, cb, cc]).astype(f32), (rstd * t).astype(f32), S1.astype(f32)


def running_bwd_coeffs(sums, mean_rstd, scale):
    """pn2_train_bn_running_bwd_coeffs -> (coef = scale | 0 | 0, dgamma, dbeta, dbias = scale S1)."""
    S1, S2 = sums
    rm, rstd = mean_rstd
    coef = np.stack([scale, np.zeros_like(scale), np.zeros_like(scale)]).astype(f32)
    return coef, (rstd * (S2 - rm * S1)).astype(f32), S1.astype(f32), (scale.astype(f64) * S1).astype(f32)


def dz(g, z, scale, shift, coef):
    """The backward GEMMs' operand dz = ca dy + cb + cc z (float64 from the fp32 coefficients)."""
    ca, cb, cc = (c.astype(f64) for c in coef)
    dy = np.where(relu_open(z, scale, shift), g.astype(f64), 0.0)
    return ca * dy + cb + cc * z.astype(f64)


def linear_bwd(a, w, dzv):
    """pn2_train_linear_bwd / _rows: g_in = dz W (rows, cin) and dW = dz^T a (cout, cin), float64; `a` is the forward's
    operand (act_in(x) or the row source's rows)."""
    return dzv @ w.astype(f64), dzv.T @ a.astype(f64)


def max_pool(a, groups, k):
    """pn2_train_bn_relu_max / _max_all on the activations a (groups * k, c): the maximum over each group's k rows and
    the first row that reaches it (torch.max(dim) semantics)."""
    g = a.reshape(groups, k, -1)
    return g.max(1), g.argmax(1)


def max_bwd(gp, arg, k):
    """pn2_train_max_bwd / _all: the pooled gradient gp (groups, c) on the winning row, 0 elsewhere -> (groups * k, c)."""
    groups, c = gp.shape
    out = np.zeros((groups, k, c), dtype=f32)
    np.put_along_axis(out, arg[:, None, :].astype(np.int64), gp[:, None, :], axis=1)
    return out.reshape(groups * k, c)
