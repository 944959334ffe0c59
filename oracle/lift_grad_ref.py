"""Gradient of the multi-view lifting with respect to the 2-D feature maps (TEST INFRASTRUCTURE ONLY).

Two CPU statements of the same thing:
  * `lift_grad_ref` -- a vectorised float64 restatement of the rule pn2_lift_views_grad implements (include/pn2_abi.h);
  * `composition_grad` -- torch autograd run through the reference's own composition: per (scene, view) the drop-in
    `projection.Projection` (a scatter of the maps onto the points, zero fill, transposed scatter as its backward), then the
    view reduction of model/pointnet2multiview.py -- F.max_pool1d over the stacked views (:39) or the first-view fill loop
    (:93-98, as oracle/projection_ref.lift_ref writes it).
tests/test_lift_grad_ref_cpu.py pins the first to the second on inputs built to hit every tie; the GPU tests then compare
the kernel with the first, bit for bit.
"""
import numpy as np
import torch
import torch.nn.functional as F


def lift_grad_ref(feats, pix, grad_out, reduce):
    """feats (B, V, C, H, W), pix (B, V, N) int (-1 = not lifted), grad_out (B, C, N) -> grad_feats (B, V, C, H, W) float64.

    max:   grad_out[b, c, i] goes to the first view (in view order) holding the maximum of channel c over the views, an
           invisible view taking part with 0; nothing reaches the maps when that view does not see the point.
    first: the whole column goes to the first view that sees the point with a column that is not all zero; without one,
           to view V-1 if it sees the point (the fill loop's last assignment), else nowhere."""
    feats = torch.as_tensor(feats).to(torch.float64)
    pix = torch.as_tensor(pix).to(torch.int64)
    grad_out = torch.as_tensor(grad_out).to(torch.float64)
    B, V, C, H, W = feats.shape
    N = pix.shape[-1]
    vis = pix >= 0                                                         # (B, V, N)
    pc = pix.clamp(min=0)
    x = torch.gather(feats.reshape(B, V, C, H * W), 3, pc[:, :, None, :].expand(B, V, C, N))
    x = torch.where(vis[:, :, None, :], x, torch.zeros((), dtype=torch.float64))   # (B, V, C, N), zeros where unseen
    views = torch.arange(V).view(1, V, 1, 1)
    if reduce == "max":
        best = x.max(dim=1, keepdim=True).values
        winner = torch.where(x == best, views, V).min(dim=1, keepdim=True).values  # first view holding the maximum
        take = (views == winner) & vis[:, :, None, :]                               # (B, V, C, N)
    else:
        ok = vis & (x != 0).any(dim=2)                                             # (B, V, N): seen, column not all zero
        first = torch.where(ok, torch.arange(V).view(1, V, 1), V).min(dim=1).values
        sel = torch.where(first < V, first, V - 1)                                 # (B, N)
        take = ((torch.arange(V).view(1, V, 1) == sel[:, None, :]) & vis)[:, :, None, :].expand(B, V, C, N)
    contrib = torch.where(take, grad_out[:, None, :, :].expand(B, V, C, N), torch.zeros((), dtype=torch.float64))
    grad = torch.zeros((B, V, C, H * W), dtype=torch.float64)
    grad.scatter_add_(3, pc[:, :, None, :].expand(B, V, C, N), contrib)
    return grad.reshape(B, V, C, H, W)


def index_vectors(pix_v):
    """pix (N,) of one view -> (indices_3d, indices_2d) in the reference's packed form ([count, ...], length N + 1)."""
    N = pix_v.shape[0]
    keep = torch.nonzero(pix_v >= 0).squeeze(1)
    ind3d = torch.zeros(N + 1, dtype=torch.int64, device=pix_v.device)
    ind2d = torch.zeros(N + 1, dtype=torch.int64, device=pix_v.device)
    ind3d[0] = ind2d[0] = keep.numel()
    ind3d[1:1 + keep.numel()] = keep
    ind2d[1:1 + keep.numel()] = pix_v[keep].to(torch.int64)
    return ind3d, ind2d


def composition_forward(feats, pix, reduce):
    """The reference's lifting under autograd: feats (B, V, C, H, W) (any float dtype, may require grad), pix (B, V, N)
    -> image features (B, C, N).  Projection.apply per (scene, view), stack, then the view reduction."""
    from pn2_b200.projection import Projection
    B, V = feats.shape[:2]
    N = pix.shape[-1]
    outs = []
    for b in range(B):
        maps = []
        for v in range(V):
            ind3d, ind2d = index_vectors(pix[b, v])
            maps.append(Projection.apply(feats[b, v], ind3d, ind2d, N))      # (C, N)
        stack = torch.stack(maps, dim=2)                                     # (C, N, V)
        if reduce == "max":
            outs.append(F.max_pool1d(stack, kernel_size=V).squeeze(2))
        else:
            final = stack[:, :, 0].clone()
            C = final.shape[0]
            for j in range(1, V):
                m = torch.nonzero((final == 0).sum(0) == C).squeeze(1)
                final[:, m] = stack[:, m, j]
            outs.append(final)
    return torch.stack(outs)


def composition_grad(feats, pix, grad_out, reduce):
    """d(sum(composition_forward * grad_out)) / d feats, float64 autograd on the CPU."""
    f = torch.as_tensor(feats).to(torch.float64).clone().requires_grad_(True)
    out = composition_forward(f, torch.as_tensor(pix).to(torch.int64), reduce)
    (out * torch.as_tensor(grad_out).to(torch.float64)).sum().backward()
    return f.grad


def tie_inputs(seed, B=2, V=3, C=3, H=4, W=5, N=96):
    """Small inputs that hit every tie of the two reductions: feature values from {-1, 0, 1}, about a third of the pixels
    with an all-zero column, every view seeing about 60 % of the points, many points per pixel, and dyadic grad_out
    (integers in [-4, 4] x 2^-3, so every sum is exact in fp32 whatever the order).  -> feats, pix (int32), grad_out."""
    rng = np.random.default_rng(seed)
    feats = rng.integers(-1, 2, size=(B, V, C, H, W)).astype(np.float32)
    zero_col = rng.random((B, V, H, W)) < 0.35
    feats[np.broadcast_to(zero_col[:, :, None], feats.shape)] = 0.0
    pix = rng.integers(0, H * W, size=(B, V, N)).astype(np.int32)
    pix[rng.random((B, V, N)) < 0.4] = -1
    grad_out = (rng.integers(-4, 5, size=(B, C, N)) * 0.125).astype(np.float32)
    return feats, pix, grad_out


def tie_cases(feats, pix):
    """Counts of the four situations the rule has to get right -> dict name -> count."""
    feats = torch.as_tensor(feats).to(torch.float64)
    pix = torch.as_tensor(pix).to(torch.int64)
    B, V, C, H, W = feats.shape
    N = pix.shape[-1]
    vis = pix >= 0
    x = torch.gather(feats.reshape(B, V, C, H * W), 3, pix.clamp(min=0)[:, :, None, :].expand(B, V, C, N))
    x = torch.where(vis[:, :, None, :], x, torch.zeros((), dtype=torch.float64))
    best = x.max(dim=1, keepdim=True).values
    at_max = x == best                                                    # (B, V, C, N)
    visible_at_max = (at_max & vis[:, :, None, :]).sum(dim=1)             # (B, C, N)
    views = torch.arange(V).view(1, V, 1, 1)
    winner = torch.where(at_max, views, V).min(dim=1).values              # (B, C, N)
    winner_visible = torch.gather(vis[:, :, None, :].expand(B, V, C, N), 1, winner[:, None]).squeeze(1)
    all_zero = ~(vis & (x != 0).any(dim=2)).any(dim=1)                    # (B, N): no seen non-zero column
    return {"max_tie_two_visible": int((visible_at_max >= 2).sum()),
            "max_won_by_invisible_zero": int((~winner_visible).sum()),
            "first_all_zero_last_visible": int((all_zero & vis[:, V - 1]).sum()),
            "first_all_zero_last_invisible": int((all_zero & ~vis[:, V - 1]).sum())}
