"""Geometry modules: the call surface of the reference's model/pointnet_util.py.

    sample_and_group (:20-47)          sample_and_group_all (:50-67)
    PointNetSetAbstraction (:70-111)   PointNetSetAbstractionMsg (:114-171)
    PointNetFeaturePropagation (:174-221)

Constructor arguments, forward signatures, tensor layouts (channel-first (B, C, N) in and out) and
state_dict keys (mlp_convs.i / mlp_bns.i / conv_blocks.i.j / bn_blocks.i.j) are the reference's, so
checkpoints and calling code carry over unchanged.

Two execution paths per module:
  * inference (module.eval() and no gradient needed): ONE fused kernel per SA scale / FP block --
    grouping, centring, concat, every 1x1 conv with its eval BatchNorm folded in, ReLU and the max
    over nsample never leave shared memory (csrc/row_mlp.cu).  Activations are channel-last inside;
    `forward_cl` exposes that layout so a whole network can stay in it (pn2_b200/models.py).
  * training, and eval() under autograd: one autograd Function per SA scale / FP block (pn2_b200/train_mlp.py):
    the first layer reads the grouped / interpolated rows where they lie, the last one pools, the backward scatters the
    input gradients without atomics.  Every BatchNorm follows its own mode as in torch -- batch statistics iff
    bn.training or it has no running statistics, else its running statistics, left untouched -- so frozen-BatchNorm
    fine-tuning (`net.train()`, then `m.eval()` on every BatchNorm) and eval-mode gradients run here too.  With
    deterministic algorithms, set_fused_training(False) or coordinates that need a gradient, the reference's own
    composition of operators -- our kernels for the geometry, torch.nn for conv/BN (coordinates that need a gradient
    still take the fused training chain over the materialised rows).  Both with identical semantics.
The group_all SA layer (one group of all N points per cloud, xyz not centred) takes the same two paths: in eval one
fp32 kernel that pools whole clouds (under both set_mlp_precision settings), in training one autograd Function.
"""
import ctypes
import os
import threading
from time import time

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, pointnet2_utils, train_mlp
from ._lib import Pn2Mlp, ptr

_FUSED_TRAINING = True


def set_fused_training(enabled):
    """Training-mode shared MLPs on the kernels of csrc/train_mlp.cu (default) or as torch.nn conv / BatchNorm / ReLU
    modules under autograd (the reference's composition).  Returns the previous setting."""
    global _FUSED_TRAINING
    prev, _FUSED_TRAINING = _FUSED_TRAINING, bool(enabled)
    return prev


def _train_fused(module, x0, convs, bns, *inputs):
    """The fused training chain serves training mode and eval mode under autograd (the calls _fusable declines because
    of autograd; each BatchNorm then normalises as torch would, see train_mlp._layer_tensors).  `inputs`: further
    tensors of the call besides x0 that may require grad."""
    # the weight gradients are accumulated with fp32 atomics (order unspecified, like the reference's backward kernels):
    # bit-reproducible training (pointnet2_utils.set_deterministic / torch.use_deterministic_algorithms) keeps torch's modules
    if not _FUSED_TRAINING or pointnet2_utils._deterministic():
        return False
    if not (module.training or _autograd(module, x0, *inputs)):
        return False
    return train_mlp.fusable_training(x0, convs, bns)


def _train_blocks(module, convs, bns, xyzs, feats, nsample=None):
    """Training-mode block Functions (train_mlp.sa_scale_train / fp_block_train): wherever the fused training chain runs,
    for fp32 CUDA inputs, coordinates that need no gradient and at most 256 samples per ball (the pooled arg-max is uint8)."""
    if not _train_fused(module, xyzs[0], convs, bns, *feats):
        return False
    if any(t.requires_grad for t in xyzs):
        return False
    if not all(t is None or (t.is_cuda and t.dtype == torch.float32) for t in list(xyzs) + list(feats)):
        return False
    return nsample is None or nsample <= 256


def _cl_view(x):
    """(B, C, N) -> (B, N, C) under autograd: the permuted view itself when x is a permuted channel-last tensor (what every
    block after the first receives), else a contiguous copy."""
    t = x.permute(0, 2, 1)
    return t if t.is_contiguous() else t.contiguous()


def _cl_xyz(xyz):
    """Coordinates (B, 3, N) that need no gradient -> contiguous (B, N, 3), without a copy when they already lie so."""
    t = xyz.permute(0, 2, 1)
    return t if t.is_contiguous() else to_channel_last(xyz)


def _sampled(xyz_cl, xyz, npoint, fps_idx):
    """new_xyz (B, npoint, 3) of the furthest point sampling, or of the caller's `fps_idx`."""
    if fps_idx is None:
        return fps_gather_cl(xyz_cl, npoint)[1]
    return pointnet2_utils.gather_operation(xyz.contiguous(), fps_idx).permute(0, 2, 1).contiguous()


def _three_nn_weights_torch(xyz1_t, xyz2_t):
    """three_nn + the reference's weight formula (model/pointnet_util.py:205-208) as torch operators: xyz1 (B, n, 3),
    xyz2 (B, m, 3) -> idx, weight (B, n, 3).  pn2_three_nn_weights computes the same formula in one kernel but differs
    from it in the last bit of some weights, so training keeps these."""
    B, N, _ = xyz1_t.shape
    dist, idx = pointnet2_utils.three_nn(xyz1_t, xyz2_t)
    dist = torch.where(dist < 1e-10, torch.full_like(dist, 1e-10), dist)
    weight = 1.0 / dist
    weight = weight / torch.sum(weight, dim=-1).view(B, N, 1)
    return idx, weight


def timeit(tag, t):
    print("{}: {}s".format(tag, time() - t))
    return time()


def pc_normalize(pc):
    centroid = np.mean(pc, axis=0)
    pc = pc - centroid
    m = np.max(np.sqrt(np.sum(pc ** 2, axis=1)))
    return pc / m


# ---------------------------------------------------------------------------------------------------
# fused-path helpers
# ---------------------------------------------------------------------------------------------------

def fold_conv_bn(conv, bn):
    """(W, b) of y = BN_eval(conv(x)) as one affine map.  conv: 1x1 Conv1d/Conv2d; bn may be None."""
    w = conv.weight.detach().reshape(conv.out_channels, conv.in_channels).to(torch.float32)
    b = conv.bias.detach().to(torch.float32) if conv.bias is not None else torch.zeros(
        conv.out_channels, device=w.device, dtype=torch.float32)
    if bn is not None:
        scale = bn.weight.detach() * torch.rsqrt(bn.running_var.detach() + bn.eps) if bn.affine else torch.rsqrt(
            bn.running_var.detach() + bn.eps)
        shift = bn.bias.detach() if bn.affine else 0.0
        w = w * scale[:, None]
        b = (b - bn.running_mean.detach()) * scale + shift
    return w.contiguous(), b.contiguous()


class FoldedMlp:
    """A stack of folded (W, b, relu) layers resident on the device, plus the pn2_mlp descriptor."""

    def __init__(self, layers):
        self.layers = [(w.contiguous(), b.contiguous(), bool(r)) for (w, b, r) in layers]
        if not 1 <= len(self.layers) <= _lib.PN2_MAX_LAYERS:
            raise _lib.Pn2Error("a fused MLP holds 1..%d layers (got %d)" % (_lib.PN2_MAX_LAYERS, len(self.layers)))
        d = Pn2Mlp()
        d.num_layers = len(self.layers)
        for i, (w, b, r) in enumerate(self.layers):
            d.cin[i], d.cout[i], d.relu[i] = w.shape[1], w.shape[0], int(r)
            d.weight[i], d.bias[i] = w.data_ptr(), b.data_ptr()
        self.desc = d
        self.cin = self.layers[0][0].shape[1]
        self.cout = self.layers[-1][0].shape[0]
        self._packed = {}
        self._bf16_ok = None

    def extended(self, more):
        return FoldedMlp(self.layers + list(more))

    def bf16_ok(self):
        """True when the widths fit the tensor-core kernel's shared memory / TMEM budget."""
        if self._bf16_ok is None:
            self._bf16_ok = bool(_lib.load().pn2_mlp_bf16_supported(ctypes.byref(self.desc)))
        return self._bf16_ok

    def packed(self, rotate):
        """bf16 pre-swizzled UMMA weight tiles (pn2_mlp_pack_bf16), cached per first-layer column rotation."""
        buf = self._packed.get(rotate)
        if buf is None:
            dev = self.layers[0][0].device
            size = int(_lib.load().pn2_mlp_pack_bf16_size(ctypes.byref(self.desc)))
            buf = torch.empty(size, dtype=torch.uint8, device=dev)
            with torch.cuda.device(dev):
                _lib.call("pn2_mlp_pack_bf16", ctypes.byref(self.desc), int(rotate), ptr(buf), _lib.stream_ptr(dev))
            self._packed[rotate] = buf
        return buf


_PRECISION = os.environ.get("PN2_MLP_PRECISION", "fp32")  # "fp32" | "bf16"; see set_mlp_precision
if _PRECISION not in ("bf16", "fp32"):
    raise ValueError("PN2_MLP_PRECISION must be 'bf16' or 'fp32'")


def set_mlp_precision(precision):
    """Arithmetic of the fused shared-MLP kernels: "fp32" (FFMA; within 1e-5 relative of the reference -- the default,
    so a reference checkpoint loaded into these drop-in modules reproduces the reference's logits) or "bf16" (tcgen05
    tensor cores, fp32 accumulate; outputs within 2e-2 relative of fp32; what bench.py and the throughput paths of
    pn2_b200/models.py select explicitly).  Returns the previous value.  Blocks whose widths do not fit the tensor-core
    kernel always run in fp32."""
    global _PRECISION
    if precision not in ("bf16", "fp32"):
        raise ValueError("precision must be 'bf16' or 'fp32'")
    prev, _PRECISION = _PRECISION, precision
    return prev


def get_mlp_precision():
    return _PRECISION


def _fold_key(convs, bns):
    """Identity + version of exactly the tensors a fold reads (weights, biases, BatchNorm affine and running statistics)."""
    key = []
    for conv, bn in zip(convs, bns):
        ts = [conv.weight, conv.bias]
        if bn is not None:
            ts += [bn.weight, bn.bias, bn.running_mean, bn.running_var]
        for t in ts:
            key.append(None if t is None else (t.data_ptr(), t._version, t.device.index))
    return tuple(key)


class _FoldCache:
    """Folded weights of one conv/BN stack, re-folded only when a tensor it reads changed (version counters).

    One entry per device, guarded by a lock: torch.nn.DataParallel replicas shallow-copy the module's __dict__, so every
    per-device replica thread sees this same object.  Replicas themselves are never cached -- their parameters are fresh
    broadcast copies whose (pointer, version) pairs the caching allocator recycles, which would make a stale hit possible
    -- they fold on every call (a handful of tiny launches).  `module.train()` drops the entries.  The cache is dropped,
    not copied, by pickling / deepcopy (the descriptor holds raw device pointers)."""

    def __init__(self):
        self._lock = threading.Lock()
        self._entries = {}

    def clear(self):
        with self._lock:
            self._entries.clear()

    def get(self, owner, convs, bns, relus):
        def fold():
            return FoldedMlp([fold_conv_bn(c, b) + (r,) for c, b, r in zip(convs, bns, relus)])

        if getattr(owner, "_is_replica", False):
            return fold()
        dev = convs[0].weight.device
        key = _fold_key(convs, bns)
        with self._lock:
            hit = self._entries.get(dev)
            if hit is not None and hit[0] == key:
                return hit[1]
        value = fold()
        with self._lock:
            self._entries[dev] = (key, value)
        return value

    def __getstate__(self):
        return {}

    def __setstate__(self, state):
        self.__init__()

    def __deepcopy__(self, memo):
        return _FoldCache()


def _all_f32(*tensors):
    return all(t is None or t.dtype == torch.float32 for t in tensors)


def _autograd(module, *tensors):
    """Grad mode is on and one of `tensors` or a parameter of `module` requires grad: the call builds an autograd graph."""
    return torch.is_grad_enabled() and (any(t is not None and t.requires_grad for t in tensors)
                                        or any(p.requires_grad for p in module.parameters()))


def _fusable(module, *tensors):
    """The fused kernels serve eval-mode, no-autograd calls on CUDA fp32 tensors with fp32 parameters; everything else
    (training, autograd, half / double models or inputs) takes the training path (_train_fused) or the reference's
    operator composition, where torch raises the same dtype errors the reference would."""
    if module.training or _autograd(module, *tensors):
        return False
    if not all(t is None or t.is_cuda for t in tensors) or not _all_f32(*tensors):
        return False
    return all(p.dtype == torch.float32 and p.is_cuda for p in module.parameters())


def _fp32_supported(mlp, c0, nsample):
    return bool(_lib.load().pn2_mlp_fp32_supported(ctypes.byref(mlp.desc), int(c0), int(nsample)))


def to_channel_last(x):
    """(B, C, N) -> contiguous (B, N, C)"""
    if x is None:
        return None
    B, C, N = x.shape
    x = _lib.check_f32(x, "channel-first tensor")
    out = torch.empty((B, N, C), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.call("pn2_transpose", B, C, N, ptr(x), ptr(out), _lib.stream_ptr(x.device))
    return out


def to_channel_first(x):
    """(B, N, C) -> contiguous (B, C, N)"""
    B, N, C = x.shape
    x = _lib.check_f32(x, "channel-last tensor")
    out = torch.empty((B, C, N), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.call("pn2_transpose", B, N, C, ptr(x), ptr(out), _lib.stream_ptr(x.device))
    return out


FPS_POLICIES = {"auto": 0, "throughput": 1, "latency": 2}


class fps_policy:
    """Context manager over pn2_set_fps_policy (include/pn2_abi.h): "auto", "throughput" (one CTA per cloud: leaves the
    SMs to the other batches in flight) or "latency" (4-CTA cluster per cloud).  The policy is read when the sampling
    kernel is launched or captured; results are identical."""

    def __init__(self, policy):
        self.policy = FPS_POLICIES[policy]

    def __enter__(self):
        self.prev = _lib.load().pn2_set_fps_policy(self.policy)
        return self

    def __exit__(self, *exc):
        _lib.load().pn2_set_fps_policy(self.prev)
        return False


def fps_gather_cl(xyz_cl, npoint):
    """xyz (B, N, 3) -> (idx (B, npoint) int32, new_xyz (B, npoint, 3)); the sampler writes the picked
    coordinates itself, replacing gather_operation + two layout copies (model/pointnet_util.py:34-35)."""
    xyz_cl = _lib.check_f32(xyz_cl, "xyz")
    B, N, _ = xyz_cl.shape
    idx = torch.empty((B, npoint), dtype=torch.int32, device=xyz_cl.device)
    new_xyz = torch.empty((B, npoint, 3), dtype=torch.float32, device=xyz_cl.device)
    temp = torch.empty((B, N), dtype=torch.float32, device=xyz_cl.device) if N > 49152 else None  # beyond the on-chip kernels
    with torch.cuda.device(xyz_cl.device):
        _lib.call("pn2_fps_gather", B, N, npoint, ptr(xyz_cl), ptr(temp), ptr(idx), ptr(new_xyz),
                  _lib.stream_ptr(xyz_cl.device))
    return idx, new_xyz


class SpatialGrid:
    """A cloud batch sorted by uniform-grid cell (csrc/grid.cu): exact ball queries / 3-NN without the brute-force
    scan, and a spatially coherent point order.  xyz (B, N, 3) with N <= grid_max_points(); cell <= 0 = automatic."""

    def __init__(self, xyz_cl, cell):
        xyz_cl = _lib.check_f32(xyz_cl, "xyz")
        B, N, _ = xyz_cl.shape
        dev = xyz_cl.device
        self.xyz, self.B, self.N = xyz_cl, B, N
        self.sorted = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        self.cell_start = torch.empty((B, grid_table_stride()), dtype=torch.int32, device=dev)
        self.order = torch.empty((B, N), dtype=torch.int32, device=dev)
        self.meta = torch.empty((B, 8), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.call("pn2_grid_build", B, N, ptr(xyz_cl), float(cell), ptr(self.sorted), ptr(self.cell_start), ptr(self.order),
                      ptr(self.meta), _lib.stream_ptr(dev))

    def tensors(self):
        return [self.sorted, self.cell_start, self.order, self.meta]

    def ball_query(self, radius, nsample, new_xyz_cl):
        """Bit-identical to pointnet2_utils.ball_query(radius, nsample, xyz, new_xyz); build with cell >= 1.01 * radius."""
        new_xyz_cl = _lib.check_f32(new_xyz_cl, "new_xyz")
        M = new_xyz_cl.shape[1]
        idx = torch.empty((self.B, M, nsample), dtype=torch.int32, device=self.xyz.device)
        with torch.cuda.device(self.xyz.device):
            _lib.call("pn2_ball_query_grid", self.B, self.N, M, float(radius), nsample, ptr(new_xyz_cl), ptr(self.xyz),
                      ptr(self.sorted), ptr(self.cell_start), ptr(self.meta), ptr(idx), _lib.stream_ptr(self.xyz.device))
        return idx

    def three_nn(self, unknown_cl, query_order=None, want_dist2=False, want_weight=True):
        """3-NN of `unknown` (B, n, 3) in this (known) cloud -> (idx, weight) [or (idx, dist2)]; bit-identical to the
        brute-force kernels."""
        unknown_cl, query_order = _lib.check_f32(unknown_cl, "unknown"), _lib.check_i32(query_order, "query_order")
        n = unknown_cl.shape[1]
        dev = self.xyz.device
        idx = torch.empty((self.B, n, 3), dtype=torch.int32, device=dev)
        d2 = torch.empty((self.B, n, 3), dtype=torch.float32, device=dev) if want_dist2 else None
        w = torch.empty((self.B, n, 3), dtype=torch.float32, device=dev) if want_weight else None
        with torch.cuda.device(dev):
            _lib.call("pn2_three_nn_grid", self.B, n, self.N, ptr(unknown_cl), ptr(self.xyz), ptr(self.sorted),
                      ptr(self.cell_start), ptr(self.meta), ptr(query_order), ptr(d2), ptr(idx), ptr(w), _lib.stream_ptr(dev))
        return (idx, d2) if want_dist2 and not want_weight else (idx, w)


_GRID_LIMITS = {}


def grid_max_points():
    if "n" not in _GRID_LIMITS:
        _GRID_LIMITS["n"] = int(_lib.load().pn2_grid_max_points())
    return _GRID_LIMITS["n"]


def grid_table_stride():
    if "s" not in _GRID_LIMITS:
        _GRID_LIMITS["s"] = int(_lib.load().pn2_grid_table_stride())
    return _GRID_LIMITS["s"]


def _bf16_flags(block0, skip, out):
    f = 0
    if block0 is not None and block0.dtype == torch.bfloat16:
        f |= _lib.FLAG_IN_BF16
    if skip is not None and skip.dtype == torch.bfloat16:
        f |= _lib.FLAG_SKIP_BF16
    if out.dtype == torch.bfloat16:
        f |= _lib.FLAG_OUT_BF16
    if out.dtype == torch.uint8:
        f |= _lib.FLAG_OUT_ARGMAX
    return f


def sa_mlp_max_cl(xyz_cl, feat_cl, new_xyz_cl, idx, order, mlp, out=None, out_offset=0, out_dtype=torch.float32):
    """Fused grouping + MLP + max.  Returns (B, M, cout) (or writes a channel slice of `out`).  bf16 feature / output
    tensors are accepted by the tensor-core path only (activations travelling between tensor-core blocks)."""
    xyz_cl, new_xyz_cl, idx = _lib.check_f32(xyz_cl, "xyz"), _lib.check_f32(new_xyz_cl, "new_xyz"), _lib.check_i32(idx, "idx")
    feat_cl = _lib.check_f32(feat_cl, "features", allow_bf16=True)
    B, N, _ = xyz_cl.shape
    M, K = idx.shape[1], idx.shape[2]
    D = 0 if feat_cl is None else feat_cl.shape[2]
    if out is None:
        out = torch.empty((B, M, mlp.cout), dtype=out_dtype, device=xyz_cl.device)
    with torch.cuda.device(xyz_cl.device):
        if _PRECISION == "bf16" and mlp.bf16_ok():
            rotate = (3 % mlp.cin) if order == _lib.ORDER_XYZ_FIRST else 0
            _lib.call("pn2_sa_mlp_max_bf16", B, N, M, K, D, ptr(xyz_cl), ptr(feat_cl), ptr(new_xyz_cl), ptr(idx),
                      mlp.desc, ptr(mlp.packed(rotate)), ptr(out), out.shape[2], out_offset, _bf16_flags(feat_cl, None, out),
                      _lib.stream_ptr(xyz_cl.device))
        elif (feat_cl is not None and feat_cl.dtype != torch.float32) or out.dtype != torch.float32:
            raise _lib.Pn2Error("bf16 activations need the tensor-core path (set_mlp_precision('bf16') and widths it supports)")
        else:
            _lib.call("pn2_sa_mlp_max", B, N, M, K, D, ptr(xyz_cl), ptr(feat_cl), ptr(new_xyz_cl), ptr(idx), order,
                      mlp.desc, ptr(out), out.shape[2], out_offset, _lib.stream_ptr(xyz_cl.device))
    return out


def sa_all_mlp_max_cl(xyz_cl, feat_cl, mlp, out=None, out_offset=0):
    """Fused group_all SA layer: rows [xyz | feat] of every point, MLP, max over all N points of each cloud.
    xyz (B, N, 3), feat (B, N, D) or None -> (B, 1, cout) (or writes a channel slice of `out`).  Always the fp32 kernel:
    the last layer must have a ReLU (every folded SA stack has one)."""
    xyz_cl, feat_cl = _lib.check_f32(xyz_cl, "xyz"), _lib.check_f32(feat_cl, "features")
    B, N, _ = xyz_cl.shape
    D = 0 if feat_cl is None else feat_cl.shape[2]
    if out is None:
        out = torch.empty((B, 1, mlp.cout), dtype=torch.float32, device=xyz_cl.device)
    with torch.cuda.device(xyz_cl.device):
        _lib.call("pn2_sa_all_mlp_max", B, N, D, ptr(xyz_cl), ptr(feat_cl), mlp.desc, ptr(out), out.shape[-1], out_offset,
                  _lib.stream_ptr(xyz_cl.device))
    return out


def three_nn_weights_cl(xyz1_cl, xyz2_cl):
    """-> idx (B, n, 3) int32, weight (B, n, 3): three_nn + sqrt + clamp + inverse-distance weights
    (model/pointnet_util.py:205-208) in one kernel."""
    xyz1_cl, xyz2_cl = _lib.check_f32(xyz1_cl, "xyz1"), _lib.check_f32(xyz2_cl, "xyz2")
    B, n, _ = xyz1_cl.shape
    m = xyz2_cl.shape[1]
    idx = torch.empty((B, n, 3), dtype=torch.int32, device=xyz1_cl.device)
    w = torch.empty((B, n, 3), dtype=torch.float32, device=xyz1_cl.device)
    with torch.cuda.device(xyz1_cl.device):
        _lib.call("pn2_three_nn_weights", B, n, m, ptr(xyz1_cl), ptr(xyz2_cl), ptr(idx), ptr(w),
                  _lib.stream_ptr(xyz1_cl.device))
    return idx, w


def fp_mlp_cl(feat1_cl, feat2_cl, idx, weight, mlp, n, row_order=None, out_dtype=torch.float32):
    """Fused 3-NN interpolation + skip concatenation + MLP.  -> (B, n, cout); with out_dtype=torch.uint8 -> (B, n)
    class predictions: arg-max over the output channels, fused into the last layer (tensor-core path only)."""
    feat1_cl, feat2_cl = _lib.check_f32(feat1_cl, "feat1", allow_bf16=True), _lib.check_f32(feat2_cl, "feat2", allow_bf16=True)
    idx, weight, row_order = _lib.check_i32(idx, "idx"), _lib.check_f32(weight, "weight"), _lib.check_i32(row_order, "row_order")
    B, m, D2 = feat2_cl.shape
    D1 = 0 if feat1_cl is None else feat1_cl.shape[2]
    if out_dtype == torch.uint8:
        if not (_PRECISION == "bf16" and mlp.bf16_ok()) or mlp.cout > 256:
            raise _lib.Pn2Error("fused arg-max output needs the tensor-core path and at most 256 output channels")
        out = torch.empty((B, n), dtype=torch.uint8, device=feat2_cl.device)
    else:
        out = torch.empty((B, n, mlp.cout), dtype=out_dtype, device=feat2_cl.device)
    with torch.cuda.device(feat2_cl.device):
        if _PRECISION == "bf16" and mlp.bf16_ok():
            _lib.call("pn2_fp_mlp_bf16", B, n, m, D1, D2, ptr(feat1_cl), ptr(feat2_cl), ptr(idx), ptr(weight), mlp.desc,
                      ptr(mlp.packed(D1)), ptr(row_order), ptr(out), _bf16_flags(feat2_cl, feat1_cl, out),
                      _lib.stream_ptr(feat2_cl.device))
        elif feat2_cl.dtype != torch.float32 or out.dtype != torch.float32 or (feat1_cl is not None and feat1_cl.dtype != torch.float32):
            raise _lib.Pn2Error("bf16 activations need the tensor-core path (set_mlp_precision('bf16') and widths it supports)")
        else:
            _lib.call("pn2_fp_mlp", B, n, m, D1, D2, ptr(feat1_cl), ptr(feat2_cl), ptr(idx), ptr(weight), mlp.desc, ptr(out),
                      _lib.stream_ptr(feat2_cl.device))
    return out


# ---------------------------------------------------------------------------------------------------
# reference surface
# ---------------------------------------------------------------------------------------------------

def sample_and_group(npoint, radius, nsample, xyz, points, returnfps=False, fps_idx=None):
    """xyz (B, N, 3), points (B, N, D) -> new_xyz (B, npoint, 3), new_points (B, npoint, nsample, 3 + D)
    with the centred xyz channels FIRST (reference :41).  `fps_idx` (B, npoint) int32: sampling indices computed by the
    caller (modules that sample the same cloud share one sampling, see models._MultiviewStackBase.forward)."""
    B, N, C = xyz.shape
    xyz_c = xyz.contiguous()
    xyz_cf = xyz.permute(0, 2, 1).contiguous()
    if fps_idx is None:
        fps_idx = pointnet2_utils.furthest_point_sample(xyz_c, npoint)
    new_xyz = pointnet2_utils.gather_operation(xyz_cf, fps_idx).permute(0, 2, 1).contiguous()
    idx = pointnet2_utils.ball_query(radius, nsample, xyz_c, new_xyz)
    grouped_xyz = pointnet2_utils.grouping_operation(xyz_cf, idx).permute(0, 2, 3, 1).contiguous()
    grouped_xyz_norm = grouped_xyz - new_xyz.view(B, npoint, 1, C)
    if points is not None:
        grouped_points = pointnet2_utils.grouping_operation(points.permute(0, 2, 1).contiguous(), idx)
        new_points = torch.cat([grouped_xyz_norm, grouped_points.permute(0, 2, 3, 1).contiguous()], dim=-1)
    else:
        new_points = grouped_xyz_norm
    if returnfps:
        return new_xyz, new_points, grouped_xyz, fps_idx
    return new_xyz, new_points


def sample_and_group_all(xyz, points):
    """One group of all N points; new_xyz is zeros and xyz is NOT centred (reference :50-67)."""
    B, N, C = xyz.shape
    new_xyz = torch.zeros(B, 1, C, device=xyz.device, dtype=xyz.dtype)
    grouped_xyz = xyz.reshape(B, 1, N, C)
    if points is not None:
        new_points = torch.cat([grouped_xyz, points.reshape(B, 1, N, -1)], dim=-1)
    else:
        new_points = grouped_xyz
    return new_xyz, new_points


class PointNetSetAbstraction(nn.Module):
    def __init__(self, npoint, radius, nsample, in_channel, mlp, group_all):
        super().__init__()
        self.npoint, self.radius, self.nsample = npoint, radius, nsample
        self.mlp_convs = nn.ModuleList()
        self.mlp_bns = nn.ModuleList()
        last = in_channel  # includes the 3 xyz channels (the caller adds them, reference :134)
        for out_channel in mlp:
            self.mlp_convs.append(nn.Conv2d(last, out_channel, 1))
            self.mlp_bns.append(nn.BatchNorm2d(out_channel))
            last = out_channel
        self.group_all = group_all
        self._fold = _FoldCache()

    def folded(self):
        return self._fold.get(self, self.mlp_convs, self.mlp_bns, [True] * len(self.mlp_convs))

    def train(self, mode=True):
        self._fold.clear()
        return super().train(mode)

    def _fused_ok(self, xyz, points):
        """Eval / no-autograd / fp32 (see _fusable) and a shape the fused kernel supports: up to PN2_MAX_LAYERS layers,
        nsample a power of two <= 128 (any N with group_all), widths within shared memory -- otherwise the reference's
        composition runs."""
        if len(self.mlp_convs) > _lib.PN2_MAX_LAYERS or not _fusable(self, xyz, points):
            return False
        return _fp32_supported(self.folded(), 3 + (0 if points is None else points.shape[1]), 0 if self.group_all else self.nsample)

    def forward_cl(self, xyz_cl, feat_cl, geometry=None, out_dtype=torch.float32):
        """Channel-last fused path: xyz (B, N, 3), feat (B, N, D) or None -> new_xyz (B, S, 3), (B, S, D').
        `geometry` = (new_xyz, ball_idx) lets several modules share one sampling / ball query.  With group_all: new_xyz
        is zeros (B, 1, 3) and the fp32 kernel pools whole clouds (geometry and out_dtype do not apply)."""
        if self.group_all:
            new_xyz = torch.zeros((xyz_cl.shape[0], 1, 3), dtype=torch.float32, device=xyz_cl.device)
            return new_xyz, sa_all_mlp_max_cl(xyz_cl, feat_cl, self.folded())
        if geometry is None:
            _, new_xyz = fps_gather_cl(xyz_cl, self.npoint)
            idx = pointnet2_utils.ball_query(self.radius, self.nsample, xyz_cl, new_xyz)
        else:
            new_xyz, idx = geometry
        out = sa_mlp_max_cl(xyz_cl, feat_cl, new_xyz, idx, _lib.ORDER_XYZ_FIRST, self.folded(), out_dtype=out_dtype)
        return new_xyz, out

    def forward(self, xyz, points, fps_idx=None):
        """xyz (B, 3, N), points (B, D, N) or None -> new_xyz (B, 3, S), new_points (B, D', S).  `fps_idx`: optional
        precomputed sampling indices (composed path only; an extension of the reference's signature)."""
        if self._fused_ok(xyz, points):
            new_xyz, out = self.forward_cl(to_channel_last(xyz), to_channel_last(points))
            return new_xyz.permute(0, 2, 1), to_channel_first(out)
        if self.group_all and _train_blocks(self, self.mlp_convs, self.mlp_bns, [xyz], [points]):
            out = train_mlp.sa_all_train(_cl_xyz(xyz), _cl_view(points) if points is not None else None, self.mlp_convs,
                                         self.mlp_bns)
            return torch.zeros((xyz.shape[0], 3, 1), dtype=torch.float32, device=xyz.device), out.permute(0, 2, 1)
        if not self.group_all and _train_blocks(self, self.mlp_convs, self.mlp_bns, [xyz], [points], self.nsample):
            xyz_cl = _cl_xyz(xyz)
            new_xyz = _sampled(xyz_cl, xyz, self.npoint, fps_idx)
            idx = pointnet2_utils.ball_query(self.radius, self.nsample, xyz_cl, new_xyz)
            out = train_mlp.sa_scale_train(xyz_cl, new_xyz, idx, _cl_view(points) if points is not None else None,
                                           _lib.ORDER_XYZ_FIRST, self.mlp_convs, self.mlp_bns)
            return new_xyz.permute(0, 2, 1), out.permute(0, 2, 1)
        xyz_t = xyz.permute(0, 2, 1)
        pts_t = points.permute(0, 2, 1) if points is not None else None
        if self.group_all:
            new_xyz, new_points = sample_and_group_all(xyz_t, pts_t)
        else:
            new_xyz, new_points = sample_and_group(self.npoint, self.radius, self.nsample, xyz_t, pts_t, fps_idx=fps_idx)
        if _train_fused(self, new_points, self.mlp_convs, self.mlp_bns):
            # (B, S, K, C) rows through the fused training chain, then the max over nsample (:109)
            Bq, S, K, C0 = new_points.shape
            a = train_mlp.fused_mlp_train(new_points.reshape(Bq * S * K, C0), self.mlp_convs, self.mlp_bns)
            new_points = a.view(Bq, S, K, -1).max(dim=2)[0].permute(0, 2, 1)
            return new_xyz.permute(0, 2, 1), new_points
        new_points = new_points.permute(0, 3, 2, 1)  # (B, C+D, nsample, npoint)
        for conv, bn in zip(self.mlp_convs, self.mlp_bns):
            new_points = F.relu(bn(conv(new_points)))
        new_points = torch.max(new_points, 2)[0]
        return new_xyz.permute(0, 2, 1), new_points


_CHILD_STREAMS = {}  # (device index, parent stream handle, i) -> side stream for independent branches of the composed path
_CHILD_LOCK = threading.Lock()


def _child_stream(device, parent, i):
    key = (device.index, parent.cuda_stream, i)
    with _CHILD_LOCK:
        st = _CHILD_STREAMS.get(key)
        if st is None:
            st = _CHILD_STREAMS[key] = torch.cuda.Stream(device)
    return st


class PointNetSetAbstractionMsg(nn.Module):
    parallel_scales = "capture"  # composed path: scales on separate streams while a CUDA graph is captured (True: always)

    def __init__(self, npoint, radius_list, nsample_list, in_channel, mlp_list):
        super().__init__()
        self.npoint, self.radius_list, self.nsample_list = npoint, radius_list, nsample_list
        self.conv_blocks = nn.ModuleList()
        self.bn_blocks = nn.ModuleList()
        for mlp in mlp_list:
            convs, bns = nn.ModuleList(), nn.ModuleList()
            last = in_channel + 3  # here in_channel EXCLUDES xyz (reference :125)
            for out_channel in mlp:
                convs.append(nn.Conv2d(last, out_channel, 1))
                bns.append(nn.BatchNorm2d(out_channel))
                last = out_channel
            self.conv_blocks.append(convs)
            self.bn_blocks.append(bns)
        self._folds = [_FoldCache() for _ in mlp_list]

    def folded(self, i):
        return self._folds[i].get(self, self.conv_blocks[i], self.bn_blocks[i], [True] * len(self.conv_blocks[i]))

    def train(self, mode=True):
        for f in self._folds:
            f.clear()
        return super().train(mode)

    def _fused_ok(self, xyz, points):
        if any(len(c) > _lib.PN2_MAX_LAYERS for c in self.conv_blocks) or not _fusable(self, xyz, points):
            return False
        c0 = 3 + (0 if points is None else points.shape[1])
        return all(_fp32_supported(self.folded(i), c0, k) for i, k in enumerate(self.nsample_list))

    def forward_cl(self, xyz_cl, feat_cl, geometry=None, out_dtype=torch.float32):
        """geometry = (new_xyz, [ball_idx per scale]) to share sampling / queries between modules."""
        if geometry is None:
            _, new_xyz = fps_gather_cl(xyz_cl, self.npoint)
            idxs = [pointnet2_utils.ball_query(r, k, xyz_cl, new_xyz) for r, k in zip(self.radius_list, self.nsample_list)]
        else:
            new_xyz, idxs = geometry
        mlps = [self.folded(i) for i in range(len(self.radius_list))]
        B = xyz_cl.shape[0]
        out = torch.empty((B, self.npoint, sum(m.cout for m in mlps)), dtype=out_dtype, device=xyz_cl.device)
        off = 0
        for idx, mlp in zip(idxs, mlps):
            # features first, centred xyz last (reference :157); scales concatenated in order (:170)
            sa_mlp_max_cl(xyz_cl, feat_cl, new_xyz, idx, _lib.ORDER_FEAT_FIRST, mlp, out=out, out_offset=off)
            off += mlp.cout
        return new_xyz, out

    def forward(self, xyz, points, fps_idx=None):
        """`fps_idx`: optional precomputed sampling indices (composed path only; an extension of the reference's signature)"""
        if self._fused_ok(xyz, points):
            new_xyz, out = self.forward_cl(to_channel_last(xyz), to_channel_last(points))
            return new_xyz.permute(0, 2, 1), to_channel_first(out)
        xyz_t = xyz.permute(0, 2, 1)
        B, N, C = xyz_t.shape
        S = self.npoint
        blocks = all(_train_blocks(self, self.conv_blocks[i], self.bn_blocks[i], [xyz], [points], k)
                     for i, k in enumerate(self.nsample_list))
        if blocks:
            xyz_c = _cl_xyz(xyz)
            feat_cl = _cl_view(points) if points is not None else None
            new_xyz = _sampled(xyz_c, xyz, S, fps_idx)
        else:
            pts_cf = points.contiguous() if points is not None else None
            xyz_c, xyz_cf = xyz_t.contiguous(), xyz.contiguous()
            if fps_idx is None:
                fps_idx = pointnet2_utils.furthest_point_sample(xyz_c, S)
            new_xyz = pointnet2_utils.gather_operation(xyz_cf, fps_idx).permute(0, 2, 1).contiguous()

        def scale(i):
            radius, K = self.radius_list[i], self.nsample_list[i]
            idx = pointnet2_utils.ball_query(radius, K, xyz_c, new_xyz)
            if blocks:  # (B, S, C_i) channel-last; features first, centred xyz last (:157)
                return train_mlp.sa_scale_train(xyz_c, new_xyz, idx, feat_cl, _lib.ORDER_FEAT_FIRST, self.conv_blocks[i],
                                                self.bn_blocks[i])
            grouped_xyz = pointnet2_utils.grouping_operation(xyz_cf, idx).permute(0, 2, 3, 1).contiguous()
            grouped_xyz = grouped_xyz - new_xyz.view(B, S, 1, C)
            if pts_cf is not None:
                gp = pointnet2_utils.grouping_operation(pts_cf, idx).permute(0, 2, 3, 1).contiguous()
                grouped = torch.cat([gp, grouped_xyz], dim=-1)
            else:
                grouped = grouped_xyz
            if _train_fused(self, grouped, self.conv_blocks[i], self.bn_blocks[i]):
                a = train_mlp.fused_mlp_train(grouped.reshape(B * S * K, grouped.shape[-1]), self.conv_blocks[i], self.bn_blocks[i])
                return a.view(B, S, K, -1).max(dim=2)[0].permute(0, 2, 1)
            grouped = grouped.permute(0, 3, 2, 1)  # (B, D, K, S)
            for conv, bn in zip(self.conv_blocks[i], self.bn_blocks[i]):
                grouped = F.relu(bn(conv(grouped)))
            return torch.max(grouped, 2)[0]

        # The scales are independent given the sampling.  While a CUDA graph is being captured (GraphedTrainStep) each
        # further scale runs on a stream of its own, so the replayed graph has parallel branches (autograd replays a
        # backward on its forward stream); eagerly the step is host bound and extra streams only cost host time.
        # Scale 0 is built LAST in both cases: the order in which the scales enter the autograd graph fixes the order in
        # which the gradients of their shared input are summed, so the one-stream and the multi-stream step agree bit for
        # bit, and with the side streams enqueued first the replayed MSG step measured 8.4 ms against 9.1 ms (4 scenes).
        n_scales = len(self.radius_list)
        par = xyz.is_cuda and n_scales > 1 and (self.parallel_scales is True or (
            self.parallel_scales == "capture" and torch.cuda.is_current_stream_capturing()))
        outs = [None] * n_scales
        if not par:
            for i in list(range(1, n_scales)) + [0]:
                outs[i] = scale(i)
        else:
            cur = torch.cuda.current_stream(xyz.device)
            sides = [_child_stream(xyz.device, cur, i) for i in range(1, n_scales)]
            for i, st in enumerate(sides, start=1):
                st.wait_stream(cur)
                with torch.cuda.stream(st):
                    outs[i] = scale(i)
            outs[0] = scale(0)
            for i, st in enumerate(sides, start=1):
                cur.wait_stream(st)
                if not torch.cuda.is_current_stream_capturing():
                    outs[i].record_stream(cur)  # allocated on the side stream, consumed on the caller's
        if blocks:
            return new_xyz.permute(0, 2, 1), torch.cat(outs, dim=2).permute(0, 2, 1)
        return new_xyz.permute(0, 2, 1), torch.cat(outs, dim=1)


class PointNetFeaturePropagation(nn.Module):
    def __init__(self, in_channel, mlp):
        super().__init__()
        self.mlp_convs = nn.ModuleList()
        self.mlp_bns = nn.ModuleList()
        last = in_channel
        for out_channel in mlp:
            self.mlp_convs.append(nn.Conv1d(last, out_channel, 1))
            self.mlp_bns.append(nn.BatchNorm1d(out_channel))
            last = out_channel
        self._fold = _FoldCache()

    def folded(self):
        return self._fold.get(self, self.mlp_convs, self.mlp_bns, [True] * len(self.mlp_convs))

    def train(self, mode=True):
        self._fold.clear()
        return super().train(mode)

    def _fused_ok(self, xyz1, xyz2, points1, points2):
        if len(self.mlp_convs) > _lib.PN2_MAX_LAYERS or not _fusable(self, xyz1, xyz2, points1, points2):
            return False
        return _fp32_supported(self.folded(), points2.shape[1] + (0 if points1 is None else points1.shape[1]), 0)

    def forward_cl(self, xyz1_cl, xyz2_cl, feat1_cl, feat2_cl, mlp=None, nn_weights=None, row_order=None,
                   out_dtype=torch.float32):
        """xyz1 (B, N, 3), xyz2 (B, S, 3), feat1 (B, N, D1) or None, feat2 (B, S, D2) -> (B, N, D').
        `mlp` overrides the folded stack (a network appends its head to the last block);
        `nn_weights` = (idx, weight) computed elsewhere (e.g. on a side stream); `row_order` (B, N) int32 = a
        spatially coherent processing order of the fine points (SpatialGrid.order), same result, cache-friendly gather."""
        mlp = mlp if mlp is not None else self.folded()
        n, m = xyz1_cl.shape[1], xyz2_cl.shape[1]
        if m == 1:
            idx = w = None
        elif nn_weights is not None:
            idx, w = nn_weights
        else:
            idx, w = three_nn_weights_cl(xyz1_cl, xyz2_cl)
        return fp_mlp_cl(feat1_cl, feat2_cl, idx, w, mlp, n, row_order=row_order, out_dtype=out_dtype)

    def forward(self, xyz1, xyz2, points1, points2):
        """xyz1 (B, 3, N), xyz2 (B, 3, S), points1 (B, D1, N) or None, points2 (B, D2, S) -> (B, D', N)"""
        if self._fused_ok(xyz1, xyz2, points1, points2):
            out = self.forward_cl(to_channel_last(xyz1), to_channel_last(xyz2), to_channel_last(points1),
                                  to_channel_last(points2))
            return to_channel_first(out)
        if _train_blocks(self, self.mlp_convs, self.mlp_bns, [xyz1, xyz2], [points1, points2]):
            idx, w = (None, None) if xyz2.shape[2] == 1 else _three_nn_weights_torch(_cl_xyz(xyz1), _cl_xyz(xyz2))
            out = train_mlp.fp_block_train(_cl_view(points1) if points1 is not None else None, _cl_view(points2), idx, w,
                                           self.mlp_convs, self.mlp_bns, xyz1.shape[2])
            return out.permute(0, 2, 1)
        xyz1_t = xyz1.permute(0, 2, 1).contiguous()
        xyz2_t = xyz2.permute(0, 2, 1).contiguous()
        B, N, _ = xyz1_t.shape
        S = xyz2_t.shape[1]
        if S == 1:
            interpolated = points2.permute(0, 2, 1).repeat(1, N, 1)
        else:
            idx, weight = _three_nn_weights_torch(xyz1_t, xyz2_t)
            interpolated = pointnet2_utils.three_interpolate(points2.contiguous(), idx, weight).permute(0, 2, 1)
        if points1 is not None:
            new_points = torch.cat([points1.permute(0, 2, 1), interpolated], dim=-1)  # skip features FIRST (:213)
        else:
            new_points = interpolated
        if _train_fused(self, new_points, self.mlp_convs, self.mlp_bns):
            a = train_mlp.fused_mlp_train(new_points.reshape(B * N, new_points.shape[-1]), self.mlp_convs, self.mlp_bns)
            return a.view(B, N, -1).permute(0, 2, 1)
        new_points = new_points.permute(0, 2, 1)
        for conv, bn in zip(self.mlp_convs, self.mlp_bns):
            new_points = F.relu(bn(conv(new_points)))
        return new_points
