"""oracle/train_mlp_ref.py, the float64 restatement of the training-mode MLP entry points, pinned to torch float64
autograd (chained, it must be Conv1d -> BatchNorm1d -> ReLU with every gradient and the running statistics) and to the
CPU grouping / interpolation; and the entry points' refusals, which happen before any CUDA call."""
import copy
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import oracle as orc
from oracle import train_mlp_ref as ref
from pn2_b200 import _lib, train_mlp

FAKE = 1 << 20  # a non-null, 16-byte aligned address; validation fails before anything is dereferenced


def _stack(widths, seed, momentum):
    torch.manual_seed(seed)
    convs, bns = nn.ModuleList(), nn.ModuleList()
    for cin, cout in zip(widths[:-1], widths[1:]):
        convs.append(nn.Conv1d(cin, cout, 1))
        bn = nn.BatchNorm1d(cout, momentum=momentum)
        with torch.no_grad():
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.normal_(0, 0.2)
            bn.running_mean.normal_(0, 0.1)
            bn.running_var.uniform_(0.5, 1.5)
        bns.append(bn)
    return convs, bns


def _np(t):
    return t.detach().numpy().astype(np.float32)


def _close(got, want, rel, what):
    want = np.asarray(want, dtype=np.float64)
    err = float(np.abs(np.asarray(got, dtype=np.float64) - want).max())
    scale = max(float(np.abs(want).max()), 1e-30)
    assert err <= rel * scale, "%s: max err %.3e vs %.1e * %.3e" % (what, err, rel, scale)


def _chain(x, convs, bns, probe):
    """The references chained as pn2_b200/train_mlp.py chains the entry points -> (out, g_x, per-layer grads, running)."""
    tensors, meta = train_mlp._layer_tensors(convs, bns)   # torch's mode rule, momentum, num_batches_tracked
    R = x.shape[0]
    a, zs, saved = x, [], []
    for l, (eps, momentum, batch) in enumerate(meta):
        W, b, gamma, beta, rm, rv = [None if t is None else _np(t) for t in tensors[6 * l:6 * l + 6]]
        prev = saved[-1] if saved else None
        z, stats, op = ref.linear_fwd(x if l == 0 else zs[-1].astype(np.float32), W.reshape(W.shape[0], -1), b,
                                      None if prev is None else prev[0], None if prev is None else prev[1])
        if batch:
            scale, shift, mr, rm2, rv2 = ref.finalize(R, stats, gamma, beta, eps, momentum, rm, rv)
        else:
            (scale, shift, mr), rm2, rv2 = ref.running(rm, rv, gamma, beta, eps), None, None
        zs.append(z)
        saved.append((scale, shift, mr, op, W.reshape(W.shape[0], -1), gamma, batch, rm2, rv2))
    out = ref.bn_act(zs[-1].astype(np.float32), saved[-1][0], saved[-1][1])
    g, grads = probe, [None] * len(saved)
    for l in range(len(saved) - 1, -1, -1):
        scale, shift, mr, op, W, gamma, batch, _, _ = saved[l]
        z = zs[l].astype(np.float32)
        sums = ref.bwd_reduce(g, z, scale, shift)
        if batch:
            coef, dgamma, dbeta = ref.bwd_coeffs(R, sums, mr, gamma)
            dbias = np.zeros_like(dbeta)
        else:
            coef, dgamma, dbeta, dbias = ref.running_bwd_coeffs(sums, mr, scale)
        g_in, dW = ref.linear_bwd(op, W, ref.dz(g, z, scale, shift, coef))
        grads[l] = (dW, dbias, dgamma, dbeta)
        g = g_in.astype(np.float32)
    return out, g, grads, [(s[7], s[8]) for s in saved]


@pytest.mark.parametrize("widths,momentum,frozen", [([7, 16, 33], 0.1, ()), ([5, 12, 9], None, ()), ([6, 8, 10], 0.1, (0,)),
                                                    ([4, 11, 6], 0.1, (0, 1))])
def test_chained_references_are_conv_batchnorm_relu_under_autograd(widths, momentum, frozen):
    R = 300
    convs, bns = _stack(widths, 7 + len(frozen), momentum)
    for l in frozen:
        bns[l].eval()                                     # normalises with its running statistics, which stay
    if momentum is None:
        for bn in bns:
            bn.num_batches_tracked.fill_(3)               # cumulative average: momentum 1 / 4 on this call
    t_convs, t_bns = copy.deepcopy(convs).double(), copy.deepcopy(bns).double()
    g = torch.Generator().manual_seed(1)
    x = (torch.randn(R, widths[0], generator=g) * 2 + 1).float()
    probe = torch.randn(R, widths[-1], generator=g).float()

    xt = x.double().t().unsqueeze(0).requires_grad_(True)
    y = xt
    for conv, bn in zip(t_convs, t_bns):
        y = F.relu(bn(conv(y)))
    (y.squeeze(0).t() * probe.double()).sum().backward()

    out, g_x, grads, run = _chain(x.numpy(), convs, bns, probe.numpy())
    _close(out, y.squeeze(0).t().detach().numpy(), 1e-5, "output")
    _close(g_x, xt.grad.squeeze(0).t().numpy(), 1e-5, "input gradient")
    for l, (c, bn, (dW, dbias, dgamma, dbeta)) in enumerate(zip(t_convs, t_bns, grads)):
        _close(dW, c.weight.grad.squeeze(-1).numpy(), 1e-5, "dW%d" % l)
        if l in frozen:
            _close(dbias, c.bias.grad.numpy(), 1e-5, "dbias%d" % l)
        else:       # zero in front of a batch-statistics BatchNorm; torch's is rounding noise
            assert np.abs(c.bias.grad.numpy()).max() <= 1e-9 * max(1.0, np.abs(dW).max()) and not dbias.any()
        _close(dgamma, bn.weight.grad.numpy(), 1e-5, "dgamma%d" % l)
        _close(dbeta, bn.bias.grad.numpy(), 1e-5, "dbeta%d" % l)
        rm, rv = run[l]
        if l in frozen:
            assert rm is None and int(bns[l].num_batches_tracked) == int(bn.num_batches_tracked)
        else:
            _close(rm, bn.running_mean.numpy(), 1e-6, "running_mean%d" % l)
            _close(rv, bn.running_var.numpy(), 1e-6, "running_var%d" % l)
            assert int(bns[l].num_batches_tracked) == int(bn.num_batches_tracked)


def test_finalize_clamps_the_variance_and_keeps_one_row():
    stats = np.array([[3.0, 2.0], [4.5, 1.0]])                 # channel 0: var = 4.5 / 1 - 9 < 0 -> 0
    scale, shift, mr, rm, rv = ref.finalize(1, stats, np.ones(2, np.float32), np.zeros(2, np.float32), 1e-5, 0.1,
                                            np.zeros(2, np.float32), np.ones(2, np.float32))
    assert mr[1, 0] == 1.0 / np.sqrt(1e-5) and mr[0, 0] == 3.0
    assert rv[0] == np.float32(0.9)                            # rows = 1: the unbiased variance divides by 1, clamped 0


@pytest.mark.parametrize("order,d", [(0, 0), (0, 6), (1, 13), (1, 32)])
def test_grouped_rows_are_sample_and_group(order, d):
    rng = np.random.default_rng(d)
    B, N, S, K = 2, 50, 7, 5
    xyz = rng.normal(size=(B, N, 3)).astype(np.float32) * 3 + 10
    new_xyz = xyz[:, :S] + np.float32(0.1)
    feat = rng.normal(size=(B, N, d)).astype(np.float32) if d else None
    idx = rng.integers(0, N, size=(B, S, K)).astype(np.int32)
    idx[0, 0, 0] = N - 1
    gx = np.stack([xyz[b][idx[b]] for b in range(B)]) - new_xyz[:, :, None, :]
    want = gx if d == 0 else np.concatenate([gx, np.stack([feat[b][idx[b]] for b in range(B)])][::1 if order == 0 else -1], -1)
    assert np.array_equal(ref.grouped_rows(xyz, new_xyz, feat, idx, order), want.reshape(B * S * K, -1))


@pytest.mark.parametrize("d_skip,m", [(0, 9), (5, 9), (8, 1)])
def test_interpolated_rows_are_three_nn_interpolation(d_skip, m):
    rng = np.random.default_rng(m + d_skip)
    B, n, d = 2, 40, 33
    x1 = rng.normal(size=(B, n, 3)).astype(np.float32)
    x2 = rng.normal(size=(B, m, 3)).astype(np.float32)
    feat = rng.normal(size=(B, m, d)).astype(np.float32)
    skip = rng.normal(size=(B, n, d_skip)).astype(np.float32) if d_skip else None
    if m > 1:
        dist, idx = orc.three_nn(x1, x2)
        w = orc.fp_weights(dist)
        gathered = np.stack([feat[b][idx[b]] for b in range(B)])                # (B, n, 3, d)
        interp = (gathered.astype(np.float64) * w[..., None]).sum(2)
    else:
        idx = w = None
        interp = np.repeat(feat, n, 1).astype(np.float64)
    got = ref.interp_rows(skip, feat, idx, w, n)
    want = interp if skip is None else np.concatenate([skip, interp], -1)
    np.testing.assert_allclose(got, want.reshape(B * n, -1), rtol=0, atol=4e-7 * max(1.0, np.abs(want).max()))


def test_all_rows_are_uncentred_xyz_and_features():
    xyz = np.arange(12, dtype=np.float32).reshape(1, 4, 3)
    feat = -np.arange(8, dtype=np.float32).reshape(1, 4, 2)
    assert np.array_equal(ref.all_rows(xyz, feat), np.concatenate([xyz, feat], -1)[0])
    assert np.array_equal(ref.all_rows(xyz[:, :1], None), xyz[0, :1])


def test_max_pool_takes_the_first_maximum_and_its_backward_puts_the_gradient_there():
    a = np.array([[0, 2], [3, 2], [3, 0], [0, 0], [0, 0], [1, 0]], np.float32)   # 2 groups of k = 3
    out, arg = ref.max_pool(a, 2, 3)
    assert out.tolist() == [[3, 2], [1, 0]] and arg.tolist() == [[1, 0], [2, 0]]
    g = ref.max_bwd(np.array([[5, 6], [7, 8]], np.float32), arg, 3)
    assert g.tolist() == [[0, 6], [5, 0], [0, 0], [0, 8], [0, 0], [7, 0]]


def test_training_entry_points_refuse_bad_input_without_gpu():
    lib = _lib.load()
    err = lib.pn2_last_error
    # misaligned pointers (16-byte loads)
    assert lib.pn2_train_linear_fwd(10, 8, 8, FAKE + 4, None, None, FAKE, FAKE, FAKE, None, None) == 1 and b"alignment" in err()
    assert lib.pn2_train_linear_fwd(10, 8, 8, FAKE, FAKE, None, FAKE, FAKE, FAKE, None, None) == 1 and b"null pointer" in err()
    assert lib.pn2_train_linear_fwd(10, 0, 8, FAKE, None, None, FAKE, FAKE, FAKE, None, None) == 1 and b"bad dims" in err()
    assert lib.pn2_train_linear_fwd(0, 8, 8, None, None, None, None, None, None, None, None) == 0
    bwd = lib.pn2_train_linear_bwd
    assert bwd(10, 8, 8, FAKE, None, None, FAKE, FAKE + 4, *([FAKE] * 8), None) == 1 and b"16-byte alignment" in err()
    assert bwd(10, 8, 8, FAKE, None, None, FAKE, FAKE, FAKE, FAKE + 4, *([FAKE] * 5), FAKE, None) == 1 and b"per-channel" in err()
    # k > 256 and out_stride < out_offset + c
    mx = lib.pn2_train_bn_relu_max
    assert mx(4, 257, 8, FAKE, FAKE, FAKE, FAKE, 8, 0, FAKE, None) == 1 and b"k <= 256" in err()
    assert mx(4, 16, 8, FAKE, FAKE, FAKE, FAKE, 9, 2, FAKE, None) == 1 and b"out_stride" in err()
    assert lib.pn2_train_max_bwd(4, 257, 8, FAKE, 8, 0, FAKE, FAKE, None) == 1 and b"k <= 256" in err()
    assert lib.pn2_train_max_bwd(4, 16, 8, FAKE, 8, 1, FAKE, FAKE, None) == 1 and b"gp_stride" in err()
    # g_skip without skip columns: a grouped source, and an interpolated one with d_skip == 0
    grouped = _lib.Pn2Rows(kind=_lib.ROWS_GROUPED, order=0, b=1, n=10, m=2, k=4, d=5, xyz=FAKE, new_xyz=FAKE, feat=FAKE, idx=FAKE)
    interp = _lib.Pn2Rows(kind=_lib.ROWS_INTERP, b=1, n=8, m=3, d=6, d_skip=0, feat=FAKE, idx=FAKE, weight=FAKE)
    br = lib.pn2_train_linear_bwd_rows
    assert br(8, 8, 16, ctypes.byref(grouped), *([FAKE] * 8), None, FAKE, FAKE, None) == 1 and b"g_skip" in err()
    assert br(8, 6, 16, ctypes.byref(interp), *([FAKE] * 8), None, FAKE, FAKE, None) == 1 and b"g_skip" in err()
    assert br(8, 6, 16, ctypes.byref(interp), FAKE + 4, *([FAKE] * 7), None, None, FAKE, None) == 1 and b"alignment" in err()
    # finalize: rows >= 1, running statistics both or neither
    fin = lib.pn2_train_bn_finalize
    assert fin(0, 4, FAKE, FAKE, FAKE, 1e-5, 0.1, FAKE, FAKE, FAKE, None, None, None) == 1 and b"bad dims" in err()
    assert fin(4, 4, FAKE, FAKE, FAKE, 1e-5, 0.1, FAKE, FAKE, FAKE, FAKE, None, None) == 1 and b"null pointer" in err()
    assert lib.pn2_train_bn_relu(4, 0, FAKE, FAKE, FAKE, FAKE, None) == 1 and b"bad dims" in err()
    assert lib.pn2_train_bn_bwd_reduce(4, 8, FAKE, None, FAKE, FAKE, FAKE, None) == 1 and b"null pointer" in err()
