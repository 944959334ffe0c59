"""Training-mode shared MLP: n x (1x1 conv -> BatchNorm -> ReLU) as ONE autograd Function over channel-last row matrices,
on the kernels of csrc/train_mlp.cu.

The reference runs this chain as torch.nn.Conv2d / Conv1d + BatchNorm + F.relu per layer (model/pointnet_util.py:105-107,
162-165, 218-220): cuDNN fprop / dgrad / wgrad plus separate BatchNorm and ReLU passes in both directions.  Here every
layer is one forward launch (the previous layer's normalisation and ReLU are applied while the operand is loaded, the
batch statistics are reduced in the same pass) and three backward launches (BatchNorm reductions, input gradient, weight
gradient); only the pre-BatchNorm activations are kept for the backward.  Semantics are torch's, per layer: a BatchNorm
normalises with the batch statistics iff bn.training or it has no running statistics (biased variance for the
normalisation, unbiased for the running estimate, eps / momentum of the module, running statistics and
num_batches_tracked updated in place when bn.training and bn.track_running_stats); otherwise with its running statistics,
which it leaves untouched -- a frozen BatchNorm (`m.eval()` inside a training network) and an eval() network under
autograd.  Such a layer's forward reduces no statistics, its backward is dz = gamma rstd dy, and its conv bias gets the
gradient sum dz.  One stack may mix the two modes.
"""
import torch
from torch.autograd import Function

from . import _lib
from ._lib import ptr


def _stream(t):
    return _lib.stream_ptr(t.device)


def _forward_layers(R, meta, tensors, dev, st, first):
    """The per-layer forward of a stack of L = len(tensors) // 6 layers over R rows; `first(cin, cout, W, b, z, stats)`
    issues layer 0's forward (its operand is the caller's; stats None: no statistics), layers 1.. read the previous z
    through act_in.  -> (zs, scales, shifts, mrs), per layer."""
    L = len(tensors) // 6
    zs, scales, shifts, mrs = [], [], [], []
    for l in range(L):
        W, b, gamma, beta, rmean, rvar = tensors[6 * l:6 * l + 6]
        eps, momentum, batch = meta[l]
        cout, cin = W.shape
        Wc, bc = W.detach().contiguous(), b.detach().contiguous()
        gc, bec = gamma.detach().contiguous(), beta.detach().contiguous()
        z = torch.empty((R, cout), dtype=torch.float32, device=dev)
        stats = torch.zeros((2, cout), dtype=torch.float64, device=dev) if batch else None
        if l == 0:
            first(cin, cout, Wc, bc, z, stats)
        else:
            _lib.call("pn2_train_linear_fwd", R, cin, cout, ptr(zs[-1]), ptr(scales[-1]), ptr(shifts[-1]), ptr(Wc), ptr(bc), ptr(z),
                      ptr(stats), st)
        scale = torch.empty(cout, dtype=torch.float32, device=dev)
        shift = torch.empty(cout, dtype=torch.float32, device=dev)
        mr = torch.empty((2, cout), dtype=torch.float64, device=dev)
        if batch:
            _lib.call("pn2_train_bn_finalize", R, cout, ptr(stats), ptr(gc), ptr(bec), float(eps), float(momentum), ptr(scale),
                      ptr(shift), ptr(mr), ptr(rmean), ptr(rvar), st)
        else:
            _lib.call("pn2_train_bn_running", cout, ptr(rmean), ptr(rvar), ptr(gc), ptr(bec), float(eps), ptr(scale), ptr(shift),
                      ptr(mr), st)
        zs.append(z); scales.append(scale); shifts.append(shift); mrs.append(mr)
    return zs, scales, shifts, mrs


def _backward_layers(R, g, zs, scales, shifts, mrs, params, batch, dev, st, first):
    """The per-layer backward from g = dL/da_L (R, C_L) down to layer 0; `first(cin, cout, Wt, g, z, scale, shift, coef, dW)`
    issues layer 0's backward and returns its input gradient(s); batch[l]: layer l used batch statistics.
    -> (that return value, parameter gradients)."""
    L = len(zs)
    grads = [None] * (6 * L)
    out = None
    for l in range(L - 1, -1, -1):
        W, b, gamma, beta = params[4 * l:4 * l + 4]
        cout, cin = W.shape
        z, scale, shift, mr = zs[l], scales[l], shifts[l], mrs[l]
        sums = torch.zeros((2, cout), dtype=torch.float64, device=dev)
        _lib.call("pn2_train_bn_bwd_reduce", R, cout, ptr(g), ptr(z), ptr(scale), ptr(shift), ptr(sums), st)
        coef = torch.empty((3, cout), dtype=torch.float32, device=dev)
        dgamma = torch.empty(cout, dtype=torch.float32, device=dev)
        dbeta = torch.empty(cout, dtype=torch.float32, device=dev)
        if batch[l]:
            _lib.call("pn2_train_bn_bwd_coeffs", R, cout, ptr(sums), ptr(mr), ptr(gamma.detach().contiguous()), ptr(coef), ptr(dgamma),
                      ptr(dbeta), st)
            dbias = torch.zeros_like(b)  # a bias in front of a batch-statistics BatchNorm has zero gradient
        else:
            dbias = torch.empty(cout, dtype=torch.float32, device=dev)
            _lib.call("pn2_train_bn_running_bwd_coeffs", cout, ptr(sums), ptr(mr), ptr(scale), ptr(coef), ptr(dgamma), ptr(dbeta),
                      ptr(dbias), st)
        dW = torch.zeros((cout, cin), dtype=torch.float32, device=dev)
        Wt = torch.empty((cin, cout), dtype=torch.float32, device=dev)
        _lib.call("pn2_transpose", 1, cout, cin, ptr(W.detach().contiguous()), ptr(Wt), st)  # W^T: an exact copy, one launch
        if l == 0:
            out = first(cin, cout, Wt, g, z, scale, shift, coef, dW)
        else:
            g_in = torch.empty((R, cin), dtype=torch.float32, device=dev)
            _lib.call("pn2_train_linear_bwd", R, cin, cout, ptr(zs[l - 1]), ptr(scales[l - 1]), ptr(shifts[l - 1]), ptr(Wt), ptr(g),
                      ptr(z), ptr(scale), ptr(shift), ptr(coef[0]), ptr(coef[1]), ptr(coef[2]), ptr(g_in), ptr(dW), st)
            g = g_in
        grads[6 * l] = dW.view_as(W)
        grads[6 * l + 1] = dbias.view_as(b)
        grads[6 * l + 2] = dgamma
        grads[6 * l + 3] = dbeta
    return out, grads


def _saved_layers(saved, L):
    zs, scales, shifts, mrs = saved[:L], saved[L:2 * L], saved[2 * L:3 * L], saved[3 * L:4 * L]
    return zs, scales, shifts, mrs, saved[4 * L:]


def _params(tensors, L):
    params = []
    for l in range(L):
        params += list(tensors[6 * l:6 * l + 4])
    return params


class _FusedMlpTrain(Function):
    @staticmethod
    def forward(ctx, x0, meta, *tensors):
        """x0 (R, C0) fp32 rows; meta = [(eps, momentum, batch statistics?), ...] per layer; tensors = (W (cout, cin), b,
        gamma, beta, running_mean or None, running_var or None) per layer -> a_L (R, C_L).  A batch-statistics layer updates
        the running statistics it is given in place (momentum, unbiased variance), like torch.nn.BatchNorm in training
        mode; a running-statistics layer only reads them."""
        L = len(tensors) // 6
        R = x0.shape[0]
        dev = x0.device
        x0 = _lib.check_f32(x0, "x0")
        st = _stream(x0)
        with torch.cuda.device(dev):
            def first(cin, cout, W, b, z, stats):
                _lib.call("pn2_train_linear_fwd", R, cin, cout, ptr(x0), None, None, ptr(W), ptr(b), ptr(z), ptr(stats), st)

            zs, scales, shifts, mrs = _forward_layers(R, meta, tensors, dev, st, first)
            a = torch.empty_like(zs[-1])
            _lib.call("pn2_train_bn_relu", R, a.shape[1], ptr(zs[-1]), ptr(scales[-1]), ptr(shifts[-1]), ptr(a), st)
        ctx.L, ctx.batch = L, [m[2] for m in meta]
        ctx.save_for_backward(x0, *zs, *scales, *shifts, *mrs, *_params(tensors, L))
        return a

    @staticmethod
    def backward(ctx, g_a):
        saved = ctx.saved_tensors
        x0 = saved[0]
        zs, scales, shifts, mrs, params = _saved_layers(saved[1:], ctx.L)
        R = x0.shape[0]
        dev = x0.device
        st = _stream(x0)
        need_x0 = ctx.needs_input_grad[0]
        with torch.cuda.device(dev):
            def first(cin, cout, Wt, g, z, scale, shift, coef, dW):
                g_in = torch.empty((R, cin), dtype=torch.float32, device=dev) if need_x0 else None
                _lib.call("pn2_train_linear_bwd", R, cin, cout, ptr(x0), None, None, ptr(Wt), ptr(g), ptr(z), ptr(scale), ptr(shift),
                          ptr(coef[0]), ptr(coef[1]), ptr(coef[2]), ptr(g_in), ptr(dW), st)
                return g_in

            g_x0, grads = _backward_layers(R, g_a.contiguous(), zs, scales, shifts, mrs, params, ctx.batch, dev, st, first)
        return (g_x0, None, *grads)


def _rows_desc(kind, **fields):
    d = _lib.Pn2Rows()
    d.kind = kind
    for k, v in fields.items():
        setattr(d, k, v)
    return d


def _pooled_grad_view(g):
    """(tensor, row stride) of a (B, S, C) gradient: itself when its (b, s) rows are C contiguous floats at a fixed
    stride (e.g. a slice of the gradient of a channel concatenation), else a contiguous copy (a broadcast gradient such
    as that of a sum has stride 0)."""
    B, S, C = g.shape
    if not (g.stride(2) == 1 and g.stride(1) >= C and g.stride(0) == S * g.stride(1)):
        g = g.contiguous()
    return g, g.stride(1)


class _SaScaleTrain(Function):
    """One SA scale in training mode: grouping + centring + concat read by the first layer's load, the conv -> BatchNorm
    -> ReLU chain, and the max over nsample fused into the last layer.  Channel-last throughout."""

    @staticmethod
    def forward(ctx, xyz, new_xyz, idx, feat, order, meta, *tensors):
        """xyz (B, N, 3), new_xyz (B, S, 3), idx (B, S, K) int32, feat (B, N, D) or None, order PN2_ORDER_* ->
        (B, S, C_L).  The max's winning sample (first maximum) is kept as uint8 per (b, s, c)."""
        L = len(tensors) // 6
        B, N, _ = xyz.shape
        S, K = idx.shape[1], idx.shape[2]
        D = 0 if feat is None else feat.shape[2]
        R = B * S * K
        dev = xyz.device
        st = _stream(xyz)
        desc = _rows_desc(_lib.ROWS_GROUPED, order=order, b=B, n=N, m=S, k=K, d=D, xyz=ptr(xyz), new_xyz=ptr(new_xyz),
                          feat=ptr(feat), idx=ptr(idx))
        with torch.cuda.device(dev):
            def first(cin, cout, W, b, z, stats):
                _lib.call("pn2_train_linear_fwd_rows", R, cin, cout, desc, ptr(W), ptr(b), ptr(z), ptr(stats), st)

            zs, scales, shifts, mrs = _forward_layers(R, meta, tensors, dev, st, first)
            C = zs[-1].shape[1]
            out = torch.empty((B, S, C), dtype=torch.float32, device=dev)
            arg = torch.empty((B, S, C), dtype=torch.uint8, device=dev)
            _lib.call("pn2_train_bn_relu_max", B * S, K, C, ptr(zs[-1]), ptr(scales[-1]), ptr(shifts[-1]), ptr(out), C, 0, ptr(arg), st)
        ctx.L, ctx.order, ctx.has_feat, ctx.batch = L, order, feat is not None, [m[2] for m in meta]
        ctx.save_for_backward(xyz, new_xyz, idx, feat, arg, *zs, *scales, *shifts, *mrs, *_params(tensors, L))
        return out

    @staticmethod
    def backward(ctx, g_out):
        saved = ctx.saved_tensors
        xyz, new_xyz, idx, feat, arg = saved[:5]
        zs, scales, shifts, mrs, params = _saved_layers(saved[5:], ctx.L)
        B, N, _ = xyz.shape
        S, K = idx.shape[1], idx.shape[2]
        D = 0 if feat is None else feat.shape[2]
        R = B * S * K
        C = zs[-1].shape[1]
        dev = xyz.device
        st = _stream(xyz)
        need_feat = D > 0 and ctx.needs_input_grad[3]
        desc = _rows_desc(_lib.ROWS_GROUPED, order=ctx.order, b=B, n=N, m=S, k=K, d=D, xyz=ptr(xyz), new_xyz=ptr(new_xyz),
                          feat=ptr(feat), idx=ptr(idx))
        with torch.cuda.device(dev):
            gp, gp_stride = _pooled_grad_view(g_out)
            g = torch.empty((R, C), dtype=torch.float32, device=dev)
            _lib.call("pn2_train_max_bwd", B * S, K, C, ptr(gp), gp_stride, 0, ptr(arg), ptr(g), st)

            def first(cin, cout, Wt, g, z, scale, shift, coef, dW):
                g_in = torch.empty((R, cin), dtype=torch.float32, device=dev) if need_feat else None
                _lib.call("pn2_train_linear_bwd_rows", R, cin, cout, desc, ptr(Wt), ptr(g), ptr(z), ptr(scale), ptr(shift),
                          ptr(coef[0]), ptr(coef[1]), ptr(coef[2]), ptr(g_in), None, ptr(dW), st)
                return g_in

            g_in, grads = _backward_layers(R, g, zs, scales, shifts, mrs, params, ctx.batch, dev, st, first)
            g_feat = None
            if need_feat:
                # grouping backward without atomics: every point sums the feature columns of its rows in row order
                seg_start = torch.empty(B * N + 1, dtype=torch.int32, device=dev)
                pos = torch.empty(R, dtype=torch.int32, device=dev)
                _lib.call("pn2_inverse_index", B, N, S * K, ptr(idx), ptr(seg_start), ptr(pos), st)
                g_feat = torch.empty((B, N, D), dtype=torch.float32, device=dev)
                col = 3 if ctx.order == _lib.ORDER_XYZ_FIRST else 0
                _lib.call("pn2_scatter_rows_det_cl", B, D, N, S * K, 1, ptr(g_in), 3 + D, col, ptr(seg_start), ptr(pos), None,
                          ptr(g_feat), st)
        return (None, None, None, g_feat, None, None, *grads)


class _FpBlockTrain(Function):
    """One FP block in training mode: 3-NN interpolation and the skip concat read by the first layer's load, then the
    conv -> BatchNorm -> ReLU chain.  Channel-last throughout."""

    @staticmethod
    def forward(ctx, feat1, feat2, idx, weight, n, meta, *tensors):
        """feat1 (B, n, D1) or None, feat2 (B, m, D2), idx / weight (B, n, 3) (None when m == 1: the coarse row is repeated)
        -> (B, n, C_L)."""
        L = len(tensors) // 6
        B, m, D2 = feat2.shape
        D1 = 0 if feat1 is None else feat1.shape[2]
        R = B * n
        dev = feat2.device
        st = _stream(feat2)
        desc = _rows_desc(_lib.ROWS_INTERP, b=B, n=n, m=m, d=D2, d_skip=D1, feat=ptr(feat2), skip=ptr(feat1), idx=ptr(idx),
                          weight=ptr(weight))
        with torch.cuda.device(dev):
            def first(cin, cout, W, b, z, stats):
                _lib.call("pn2_train_linear_fwd_rows", R, cin, cout, desc, ptr(W), ptr(b), ptr(z), ptr(stats), st)

            zs, scales, shifts, mrs = _forward_layers(R, meta, tensors, dev, st, first)
            C = zs[-1].shape[1]
            a = torch.empty((B, n, C), dtype=torch.float32, device=dev)
            _lib.call("pn2_train_bn_relu", R, C, ptr(zs[-1]), ptr(scales[-1]), ptr(shifts[-1]), ptr(a), st)
        ctx.L, ctx.n, ctx.batch = L, n, [m[2] for m in meta]
        ctx.save_for_backward(feat1, feat2, idx, weight, *zs, *scales, *shifts, *mrs, *_params(tensors, L))
        return a

    @staticmethod
    def backward(ctx, g_a):
        saved = ctx.saved_tensors
        feat1, feat2, idx, weight = saved[:4]
        zs, scales, shifts, mrs, params = _saved_layers(saved[4:], ctx.L)
        B, m, D2 = feat2.shape
        n = ctx.n
        D1 = 0 if feat1 is None else feat1.shape[2]
        R = B * n
        dev = feat2.device
        st = _stream(feat2)
        need1, need2 = D1 > 0 and ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        desc = _rows_desc(_lib.ROWS_INTERP, b=B, n=n, m=m, d=D2, d_skip=D1, feat=ptr(feat2), skip=ptr(feat1), idx=ptr(idx),
                          weight=ptr(weight))
        with torch.cuda.device(dev):
            def first(cin, cout, Wt, g, z, scale, shift, coef, dW):
                g1 = torch.empty((B, n, D1), dtype=torch.float32, device=dev) if need1 else None  # row i is point i: no scatter
                g_in = torch.empty((R, D2), dtype=torch.float32, device=dev) if need2 else None
                _lib.call("pn2_train_linear_bwd_rows", R, cin, cout, desc, ptr(Wt), ptr(g), ptr(z), ptr(scale), ptr(shift),
                          ptr(coef[0]), ptr(coef[1]), ptr(coef[2]), ptr(g_in), ptr(g1), ptr(dW), st)
                return g1, g_in

            (g1, g_in), grads = _backward_layers(R, g_a.contiguous(), zs, scales, shifts, mrs, params, ctx.batch, dev, st, first)
            g2 = None
            if need2:
                g2 = torch.empty((B, m, D2), dtype=torch.float32, device=dev)
                if idx is None:
                    # m == 1: the one coarse row was repeated n times; every row refers to point 0
                    idx_rep = torch.zeros((B, n), dtype=torch.int32, device=dev)
                    seg_start = torch.empty(B + 1, dtype=torch.int32, device=dev)
                    pos = torch.empty(B * n, dtype=torch.int32, device=dev)
                    _lib.call("pn2_inverse_index", B, 1, n, ptr(idx_rep), ptr(seg_start), ptr(pos), st)
                    _lib.call("pn2_scatter_rows_det_cl", B, D2, 1, n, 1, ptr(g_in), D2, 0, ptr(seg_start), ptr(pos), None, ptr(g2), st)
                else:
                    # three_interpolate backward without atomics: every coarse point sums w * g over its rows in order
                    seg_start = torch.empty(B * m + 1, dtype=torch.int32, device=dev)
                    pos = torch.empty(B * n * 3, dtype=torch.int32, device=dev)
                    _lib.call("pn2_inverse_index", B, m, 3 * n, ptr(idx), ptr(seg_start), ptr(pos), st)
                    _lib.call("pn2_scatter_rows_det_cl", B, D2, m, 3 * n, 3, ptr(g_in), D2, 0, ptr(seg_start), ptr(pos), ptr(weight),
                              ptr(g2), st)
        return (g1, g2, None, None, None, None, *grads)


class _SaAllTrain(Function):
    """The group_all SA layer in training mode: the [xyz | feat] rows read by the first layer's load, the conv ->
    BatchNorm -> ReLU chain, and the max over all N points of each cloud fused into the last layer."""

    @staticmethod
    def forward(ctx, xyz, feat, meta, *tensors):
        """xyz (B, N, 3), feat (B, N, D) or None -> (B, 1, C_L).  The max's winning point (first maximum) is kept as int32
        per (b, c)."""
        L = len(tensors) // 6
        B, N, _ = xyz.shape
        D = 0 if feat is None else feat.shape[2]
        R = B * N
        dev = xyz.device
        st = _stream(xyz)
        desc = _rows_desc(_lib.ROWS_ALL, b=B, n=N, d=D, xyz=ptr(xyz), feat=ptr(feat))
        with torch.cuda.device(dev):
            def first(cin, cout, W, b, z, stats):
                _lib.call("pn2_train_linear_fwd_rows", R, cin, cout, desc, ptr(W), ptr(b), ptr(z), ptr(stats), st)

            zs, scales, shifts, mrs = _forward_layers(R, meta, tensors, dev, st, first)
            C = zs[-1].shape[1]
            out = torch.empty((B, 1, C), dtype=torch.float32, device=dev)
            arg = torch.empty((B, C), dtype=torch.int32, device=dev)
            _lib.call("pn2_train_bn_relu_max_all", B, N, C, ptr(zs[-1]), ptr(scales[-1]), ptr(shifts[-1]), ptr(out), C, 0, ptr(arg), st)
        ctx.L, ctx.batch = L, [m[2] for m in meta]
        ctx.save_for_backward(xyz, feat, arg, *zs, *scales, *shifts, *mrs, *_params(tensors, L))
        return out

    @staticmethod
    def backward(ctx, g_out):
        saved = ctx.saved_tensors
        xyz, feat, arg = saved[:3]
        zs, scales, shifts, mrs, params = _saved_layers(saved[3:], ctx.L)
        B, N, _ = xyz.shape
        D = 0 if feat is None else feat.shape[2]
        R = B * N
        C = zs[-1].shape[1]
        dev = xyz.device
        st = _stream(xyz)
        need_feat = D > 0 and ctx.needs_input_grad[1]
        desc = _rows_desc(_lib.ROWS_ALL, b=B, n=N, d=D, xyz=ptr(xyz), feat=ptr(feat))
        with torch.cuda.device(dev):
            gp = g_out[:, 0]  # (B, C): read in place when its rows are C contiguous floats (not for a broadcast gradient)
            if not (gp.stride(1) == 1 and gp.stride(0) >= C):
                gp = gp.contiguous()
            g = torch.empty((R, C), dtype=torch.float32, device=dev)
            _lib.call("pn2_train_max_bwd_all", B, N, C, ptr(gp), gp.stride(0), 0, ptr(arg), ptr(g), st)

            def first(cin, cout, Wt, g, z, scale, shift, coef, dW):
                g_feat = torch.empty((B, N, D), dtype=torch.float32, device=dev) if need_feat else None  # row = point: no scatter
                _lib.call("pn2_train_linear_bwd_rows", R, cin, cout, desc, ptr(Wt), ptr(g), ptr(z), ptr(scale), ptr(shift),
                          ptr(coef[0]), ptr(coef[1]), ptr(coef[2]), ptr(g_feat), None, ptr(dW), st)
                return g_feat

            g_feat, grads = _backward_layers(R, g, zs, scales, shifts, mrs, params, ctx.batch, dev, st, first)
        return (None, g_feat, None, *grads)


def _layer_tensors(convs, bns):
    """(tensors, meta) of a conv / BatchNorm stack for the Functions above, each BatchNorm in its own mode by torch's rule:
    batch statistics iff bn.training or it has no running statistics; the running statistics (and num_batches_tracked)
    are updated iff bn.training and bn.track_running_stats, and are read instead of the batch's otherwise."""
    tensors, meta = [], []
    for conv, bn in zip(convs, bns):
        batch = bn.training or bn.running_mean is None
        update = bn.training and bn.track_running_stats and bn.running_mean is not None
        if update:
            bn.num_batches_tracked += 1
        momentum = bn.momentum if bn.momentum is not None else (1.0 / float(bn.num_batches_tracked) if update else 0.0)
        running = update or not batch
        tensors += [conv.weight.reshape(conv.out_channels, conv.in_channels), conv.bias, bn.weight, bn.bias,
                    bn.running_mean if running else None, bn.running_var if running else None]
        meta.append((float(bn.eps), float(momentum), batch))
    return tensors, meta


def fused_mlp_train(x0, convs, bns):
    """x0 (R, C0) rows -> (R, C_L) = the conv -> BatchNorm -> ReLU chain under autograd, every BatchNorm in its own mode
    (batch or running statistics, running statistics and num_batches_tracked updated) exactly like torch.nn.BatchNorm."""
    tensors, meta = _layer_tensors(convs, bns)
    return _FusedMlpTrain.apply(x0, meta, *tensors)


def sa_scale_train(xyz, new_xyz, idx, feat, order, convs, bns):
    """One SA scale in training mode, channel-last: xyz (B, N, 3), new_xyz (B, S, 3), idx (B, S, K) int32 (K <= 256),
    feat (B, N, D) or None, order _lib.ORDER_XYZ_FIRST (SSG) / ORDER_FEAT_FIRST (MSG) -> (B, S, C_L) = the max over the K
    grouped rows of the conv -> BatchNorm -> ReLU chain.  Same values, gradients and running statistics as
    sample_and_group + fused_mlp_train + max(dim=2); xyz and new_xyz get no gradient."""
    xyz, new_xyz, idx = _lib.check_f32(xyz, "xyz"), _lib.check_f32(new_xyz, "new_xyz"), _lib.check_i32(idx, "idx")
    feat = _lib.check_f32(feat, "feat")
    tensors, meta = _layer_tensors(convs, bns)
    return _SaScaleTrain.apply(xyz, new_xyz, idx, feat, int(order), meta, *tensors)


def sa_all_train(xyz, feat, convs, bns):
    """The group_all SA layer in training mode, channel-last: xyz (B, N, 3), feat (B, N, D) or None -> (B, 1, C_L) = the
    max over all N rows [xyz | feat] of each cloud of the conv -> BatchNorm -> ReLU chain.  Same values, gradients
    and running statistics as sample_and_group_all + fused_mlp_train + max(dim=2); xyz gets no gradient."""
    xyz, feat = _lib.check_f32(xyz, "xyz"), _lib.check_f32(feat, "feat")
    tensors, meta = _layer_tensors(convs, bns)
    return _SaAllTrain.apply(xyz, feat, meta, *tensors)


def fp_block_train(feat1, feat2, idx, weight, convs, bns, n):
    """One FP block in training mode, channel-last: feat1 (B, n, D1) or None (skip features, first), feat2 (B, m, D2),
    idx / weight (B, n, 3) of the 3-NN (None when m == 1) -> (B, n, C_L)."""
    feat1, feat2 = _lib.check_f32(feat1, "feat1"), _lib.check_f32(feat2, "feat2")
    idx, weight = _lib.check_i32(idx, "idx"), _lib.check_f32(weight, "weight")
    tensors, meta = _layer_tensors(convs, bns)
    return _FpBlockTrain.apply(feat1, feat2, idx, weight, int(n), meta, *tensors)


def fusable_training(x0, convs, bns):
    """The fused training chain serves CUDA fp32 stacks of 1x1 convolutions with bias, each followed by an affine BatchNorm."""
    if not (x0.is_cuda and x0.dtype == torch.float32):
        return False
    for conv, bn in zip(convs, bns):
        if conv.bias is None or bn is None or not bn.affine or conv.weight.dtype != torch.float32 or not conv.weight.is_cuda:
            return False
        if tuple(conv.kernel_size) != (1,) * len(conv.kernel_size):
            return False
    return True
