"""Multi-view 2D->3D feature lifting: the call surface of the reference's utils/projection.py
(ProjectionHelper :5-230, Projection :234-267) plus the batched fused operator `lift_views`.

Reference behaviour kept (SURVEY.md F3/F4, A.8/A.9):
  * NEAREST pixel (torch.round, half-to-even), never bilinear (utils/projection.py:204);
  * frustum test round(100*s)/100 < 0 against corners 2 / 4 (:108-120), bounds, depth-range and
    |depth - z| <= accuracy tests (:207-216);
  * compute_projection returns two int64 vectors of length num_points + 1, `[count, indices...]`
    (the tail beyond count is unspecified in the reference; zero here), or None when nothing projects;
  * two view reductions: max over views with zeros for invisible views
    (model/pointnet2multiview.py:39) and first-view-wins / fill-where-all-zero (:93-98).

The reference evaluates the projection with ~25 small torch ops and >= 4 host<->device round trips per
(scene, view) in the training loop (SURVEY.md 3.4); here the per-point work of ALL views of ALL scenes is
one kernel launch (csrc/lift.cu), and compute_projection is a thin single-view wrapper over it.
"""
import ctypes

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib
from ._lib import ptr


def _skeleton(intrinsic, ux, uy, depth):
    x = (ux - float(intrinsic[0][2])) / float(intrinsic[0][0])
    y = (uy - float(intrinsic[1][2])) / float(intrinsic[1][1])
    return [depth * x, depth * y, depth]


def frustum_corners(intrinsic, depth_min, depth_max, image_dims, camera_to_world):
    """camera_to_world (..., 4, 4) -> corners (..., 8, 4) in world coordinates (utils/projection.py:25-52)."""
    W, H = image_dims
    pts = []
    for d in (depth_min, depth_max):
        for (u, v) in ((0, 0), (W - 1, 0), (W - 1, H - 1), (0, H - 1)):
            pts.append(_skeleton(intrinsic, u, v, d) + [1.0])
    cam = torch.tensor(pts, dtype=torch.float32, device=camera_to_world.device)  # (8, 4) in camera space
    return torch.matmul(camera_to_world.unsqueeze(-3), cam.unsqueeze(-1)).squeeze(-1)


def frustum_normals(corners):
    """corners (..., 8, 4) -> inward plane normals (..., 6, 3) (utils/projection.py:54-95)."""
    c = corners[..., :3]

    def cross(a0, a1, b0, b1):
        return torch.cross(c[..., a1, :] - c[..., a0, :], c[..., b1, :] - c[..., b0, :], dim=-1)

    return torch.stack([cross(0, 3, 0, 1),   # front
                        cross(1, 2, 1, 5),   # right
                        cross(2, 3, 2, 6),   # roof
                        cross(3, 0, 3, 7),   # left
                        cross(0, 1, 0, 4),   # bottom
                        cross(5, 6, 5, 4)],  # back
                       dim=-2)


def _camera_corners(intrinsic, depth_min, depth_max, image_dims):
    """The eight camera-space frustum corners (24 Python floats), utils/projection.py:37-44."""
    W, H = image_dims
    cam = []
    for d in (depth_min, depth_max):
        for (u, v) in ((0, 0), (W - 1, 0), (W - 1, H - 1), (0, H - 1)):
            cam += _skeleton(intrinsic, u, v, d)  # Python floats, rounded to fp32 by ctypes as torch.Tensor(...) does
    return cam


def view_params(camera_to_world, intrinsic, depth_min, depth_max, image_dims):
    """camera_to_world (..., 4, 4) cuda -> (w2c (..., 4, 4), corner2 (..., 3), corner4 (..., 3), normals (..., 6, 3)):
    everything the lifting / frustum tests need per view, in ONE launch (pn2_lift_setup) instead of the ~25 torch ops of
    utils/projection.py:25-95 + torch.inverse (:178).  The inverse is an fp64 adjugate rounded once, so it agrees with
    torch.inverse to ~1 ulp rather than bitwise (see csrc/lift.cu)."""
    _lib.require_cuda(camera_to_world)
    c2w = camera_to_world.to(torch.float32).contiguous()
    lead = c2w.shape[:-2]
    nv = c2w.numel() // 16
    cam = (ctypes.c_float * 24)(*_camera_corners(intrinsic, depth_min, depth_max, image_dims))
    w2c_c = torch.empty((nv, 16), dtype=torch.float32, device=c2w.device)
    c2_c = torch.empty((nv, 3), dtype=torch.float32, device=c2w.device)
    c4_c = torch.empty((nv, 3), dtype=torch.float32, device=c2w.device)
    nrm_c = torch.empty((nv, 18), dtype=torch.float32, device=c2w.device)
    with torch.cuda.device(c2w.device):
        _lib.call("pn2_lift_setup", nv, ptr(c2w), cam, ptr(w2c_c), ptr(c2_c), ptr(c4_c), ptr(nrm_c), _lib.stream_ptr(c2w.device))
    return w2c_c.view(*lead, 4, 4), c2_c.view(*lead, 3), c4_c.view(*lead, 3), nrm_c.view(*lead, 6, 3)


def lift_views(points, feats, depth, camera_to_world, intrinsic, depth_min, depth_max, image_dims, accuracy,
               reduce="max", return_pixels=False, view_parameters=None):
    """Fused lifting for a batch.

    points (B, N, 3); feats (B, V, C, H, W) feature maps (e.g. ENet, C=128, H=32, W=41); depth (B, V, H, W);
    camera_to_world (B, V, 4, 4); intrinsic 4x4 (or 3x3) with fx, fy, cx, cy; image_dims = [W, H].
    reduce = "max" | "first".  Returns image_features (B, C, N) [, pix (B, V, N) int32 (-1 = not lifted),
    count (B, V) int32].  view_parameters = (w2c (B,V,4,4), corner2 (B,V,3), corner4 (B,V,3), normals (B,V,6,3)) replaces
    the internal `view_params(camera_to_world, ...)` call, for callers that already hold them (camera_to_world is then
    unused and may be None).

    Differentiable with respect to feats: when grad mode is on and feats.requires_grad, the output carries a grad_fn whose
    backward (pn2_lift_views_grad) is the gradient of the reference's composition -- Projection per view, then the view
    reduction -- computed in a fixed order (bit-reproducible).  points, depth and poses get no gradient (the lifting is
    piecewise constant in them); pix and count are not differentiable.  Without a gradient the call is the plain forward.
    """
    if feats.requires_grad and torch.is_grad_enabled():
        def run(f):  # called by the Function with grad mode off: the plain forward below, asked for pix
            return lift_views(points, f, depth, camera_to_world, intrinsic, depth_min, depth_max, image_dims, accuracy,
                              reduce=reduce, return_pixels=True, view_parameters=view_parameters)
        res = _LiftViews.apply(feats, run, reduce)
        return res if return_pixels else res[0]
    _lib.require_cuda(points, feats, depth)
    B, N, _ = points.shape
    _, V, C, H, W = feats.shape
    if [W, H] != [int(image_dims[0]), int(image_dims[1])]:
        raise _lib.Pn2Error("image_dims [W, H] = %s does not match the feature maps (H=%d, W=%d)" % (list(image_dims), H, W))
    dev = points.device
    intr = (ctypes.c_float * 4)(float(intrinsic[0][0]), float(intrinsic[1][1]), float(intrinsic[0][2]), float(intrinsic[1][2]))
    out = torch.empty((B, C, N), dtype=torch.float32, device=dev)
    pix = torch.empty((B, V, N), dtype=torch.int32, device=dev) if return_pixels else None
    count = torch.zeros((B, V), dtype=torch.int32, device=dev) if return_pixels else None
    points, feats, depth = _lib.check_f32(points, "points"), _lib.check_f32(feats, "feats"), _lib.check_f32(depth, "depth")
    red = _lib.REDUCE_FIRST if reduce == "first" else _lib.REDUCE_MAX
    if view_parameters is None and V * H * W * 16 <= 200 * 1024:
        # the per-view parameters are derived inside the projection kernel (same arithmetic as view_params / pn2_lift_setup)
        c2w = _lib.check_f32(camera_to_world, "camera_to_world")
        if c2w.numel() != B * V * 16:
            raise _lib.Pn2Error("camera_to_world must be (B, V, 4, 4) = (%d, %d, 4, 4)" % (B, V))
        cam = (ctypes.c_float * 24)(*_camera_corners(intrinsic, depth_min, depth_max, image_dims))
        with torch.cuda.device(dev):
            _lib.call("pn2_lift_views_poses", B, N, V, C, H, W, ptr(points), ptr(feats), ptr(depth), ptr(c2w), cam, intr,
                      float(depth_min), float(depth_max), float(accuracy), red, ptr(out), ptr(pix), ptr(count), _lib.stream_ptr(dev))
    else:
        if view_parameters is None:
            w2c, corner2, corner4, normals = view_params(camera_to_world, intrinsic, depth_min, depth_max, image_dims)
        else:
            w2c, corner2, corner4, normals = [_lib.check_f32(t, "view_parameters") for t in view_parameters]
            if w2c.numel() != B * V * 16 or corner2.numel() != B * V * 3 or corner4.numel() != B * V * 3 or normals.numel() != B * V * 18:
                raise _lib.Pn2Error("view_parameters do not match (B, V) = (%d, %d)" % (B, V))
        with torch.cuda.device(dev):
            _lib.call("pn2_lift_views", B, N, V, C, H, W, ptr(points), ptr(feats), ptr(depth), ptr(w2c), ptr(corner2),
                      ptr(corner4), ptr(normals), intr, float(depth_min), float(depth_max), float(accuracy), red, ptr(out), ptr(pix),
                      ptr(count), _lib.stream_ptr(dev))
    if return_pixels:
        return out, pix, count
    return out


def lift_views_grad(feats, pix, grad_out, reduce="max"):
    """Backward of lift_views with respect to the feature maps (pn2_lift_views_grad): feats (B, V, C, H, W) as given to
    the forward, pix (B, V, N) int32 as it returned them, grad_out (B, C, N) -> grad_feats (B, V, C, H, W).  Every
    contribution to one element is summed in ascending point index, in fp32: the result is bit-reproducible."""
    feats, grad_out = _lib.check_f32(feats, "feats"), _lib.check_f32(grad_out, "grad_out")
    pix = _lib.check_i32(pix, "pix")
    B, V, C, H, W = feats.shape
    N = pix.shape[-1]
    if tuple(pix.shape) != (B, V, N) or tuple(grad_out.shape) != (B, C, N):
        raise _lib.Pn2Error("lift_views_grad: pix must be (B, V, N) and grad_out (B, C, N) for feats (B, V, C, H, W) = %s"
                            % (tuple(feats.shape),))
    grad = torch.empty((B, V, C, H, W), dtype=torch.float32, device=feats.device)
    red = _lib.REDUCE_FIRST if reduce == "first" else _lib.REDUCE_MAX
    with torch.cuda.device(feats.device):
        _lib.call("pn2_lift_views_grad", B, N, V, C, H, W, ptr(feats), ptr(pix), red, ptr(grad_out), ptr(grad),
                  _lib.stream_ptr(feats.device))
    return grad


class _LiftViews(Function):
    """lift_views under autograd: the forward always asks the kernels for pix (what the backward needs); the backward is
    pn2_lift_views_grad.  Only feats is differentiable."""

    @staticmethod
    def forward(ctx, feats, run, reduce):
        out, pix, count = run(feats)
        ctx.save_for_backward(feats, pix)
        ctx.reduce = reduce
        ctx.mark_non_differentiable(pix, count)
        return out, pix, count

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out, *_):
        feats, pix = ctx.saved_tensors
        return lift_views_grad(feats, pix, grad_out, ctx.reduce), None, None


def frustum_counts(points, camera_to_world, intrinsic, depth_min, depth_max, image_dims, view_parameters=None):
    """points (N, 3) cuda fp32, camera_to_world (P, 4, 4) -> (P,) int32: points inside each pose's viewing frustum.
    One launch for all poses of a scene; replaces the loader's per-pose-file loop over points_in_frustum_cpu
    (data_utils/ScanNetDataLoader.py:91-97).  view_parameters = (corner2 (P,3), corner4 (P,3), normals (P,6,3)) replaces
    the internal view_params call."""
    points = _lib.check_f32(points, "points")
    if view_parameters is None:
        _, c2, c4, normals = view_params(camera_to_world, intrinsic, depth_min, depth_max, image_dims)
    else:
        c2, c4, normals = [_lib.check_f32(t, "view_parameters") for t in view_parameters]
    P, N = c2.numel() // 3, points.shape[0]
    counts = torch.zeros((P,), dtype=torch.int32, device=points.device)
    points = points.contiguous()
    with torch.cuda.device(points.device):
        _lib.call("pn2_frustum_count", N, P, ptr(points), ptr(c2), ptr(c4), ptr(normals), ptr(counts), _lib.stream_ptr(points.device))
    return counts


def best_views(points, camera_to_world, num_images, intrinsic, depth_min, depth_max, image_dims, min_points=100):
    """The loader's selection rule (data_utils/ScanNetDataLoader.py:98-105): repeatedly take the pose that sees most
    points; after the first, a pose is only accepted if it sees more than `min_points`, otherwise the first is repeated.
    Ties resolve to the lowest pose index (dict insertion order in the reference).  -> list of pose indices."""
    counts = frustum_counts(points, camera_to_world, intrinsic, depth_min, depth_max, image_dims).cpu().tolist()
    remaining = dict(enumerate(counts))
    chosen = []
    for i in range(num_images):
        if not remaining:
            chosen.append(chosen[0])
            continue
        best = max(remaining, key=remaining.get)
        if i == 0 or remaining[best] > min_points:
            chosen.append(best)
            del remaining[best]
        else:
            chosen.append(chosen[0])
    return chosen


class ProjectionHelper:
    def __init__(self, intrinsic, depth_min, depth_max, image_dims, accuracy):
        self.intrinsic = intrinsic
        self.depth_min = depth_min
        self.depth_max = depth_max
        self.image_dims = image_dims
        self.accuracy = accuracy

    def depth_to_skeleton(self, ux, uy, depth):
        return torch.Tensor(_skeleton(self.intrinsic, ux, uy, depth))

    def skeleton_to_depth(self, p):
        x = (p[0] * self.intrinsic[0][0]) / p[2] + self.intrinsic[0][2]
        y = (p[1] * self.intrinsic[1][1]) / p[2] + self.intrinsic[1][2]
        return torch.Tensor([x, y, p[2]])

    def compute_frustum_corners(self, camera_to_world):
        """(4, 4) -> (8, 4, 1), as the reference returns it"""
        return frustum_corners(self.intrinsic, self.depth_min, self.depth_max, self.image_dims, camera_to_world).unsqueeze(-1)

    def compute_frustum_normals(self, corner_coords):
        return frustum_normals(corner_coords.reshape(8, 4))

    def _frustum_mask(self, corner_coords, normals, new_pts):
        c = corner_coords.reshape(8, 4)
        mask = torch.ones(new_pts.shape[0], dtype=torch.bool, device=new_pts.device)
        for k in range(6):
            rel = new_pts - (c[2, :3] if k < 3 else c[4, :3])
            mask &= (torch.round(torch.mm(rel, normals[k].unsqueeze(1)) * 100) / 100 < 0).squeeze(1)
        return mask

    def points_in_frustum(self, corner_coords, normals, new_pts, return_mask=False):
        mask = self._frustum_mask(corner_coords.cuda(), normals.cuda(), new_pts.cuda())
        return mask if return_mask else torch.sum(mask)

    def points_in_frustum_cpu(self, corner_coords, normals, new_pts, return_mask=False):
        mask = self._frustum_mask(corner_coords, normals, new_pts)
        return mask if return_mask else torch.sum(mask)

    def compute_projection(self, points, depth, camera_to_world, num_points):
        """points (num_points, 3) cuda, depth (H, W), camera_to_world (4, 4) -> (indices_3d, indices_2d) int64
        vectors of length num_points + 1 ([count, ...]) or None when no point projects."""
        W, H = int(self.image_dims[0]), int(self.image_dims[1])
        dummy = torch.zeros((1, 1, 0, H, W), dtype=torch.float32, device=points.device)
        _, pix, _ = lift_views(points[:num_points].reshape(1, num_points, 3), dummy, depth.reshape(1, 1, H, W),
                               camera_to_world.reshape(1, 1, 4, 4), self.intrinsic, self.depth_min, self.depth_max,
                               self.image_dims, self.accuracy, return_pixels=True)
        pix = pix.reshape(-1)
        keep = torch.nonzero(pix >= 0).squeeze(1)
        n = int(keep.numel())
        if n == 0:
            return None
        ind3d = torch.zeros(num_points + 1, dtype=torch.int64, device=points.device)
        ind2d = torch.zeros(num_points + 1, dtype=torch.int64, device=points.device)
        ind3d[0] = n
        ind2d[0] = n
        ind3d[1:1 + n] = keep
        ind2d[1:1 + n] = pix[keep].to(torch.int64)
        return ind3d, ind2d


class Projection(Function):
    """Scatter of 2-D feature columns onto points from precomputed index vectors (utils/projection.py:234-267).
    Kept for calling code that already holds (indices_3d, indices_2d); `lift_views` is the fused path.
    The backward is the transposed scatter (the reference's own backward is broken on torch >= 1.0, SURVEY.md 5)."""

    @staticmethod
    def forward(ctx, label, lin_indices_3d, lin_indices_2d, num_points):
        ctx.save_for_backward(lin_indices_3d, lin_indices_2d)
        ctx.shape = label.shape
        C = 1 if label.dim() == 2 else label.shape[0]
        out = label.new_zeros((C, num_points))
        n = int(lin_indices_3d[0])
        if n > 0:
            vals = torch.index_select(label.reshape(C, -1), 1, lin_indices_2d[1:1 + n])
            out[:, lin_indices_3d[1:1 + n]] = vals
        return out

    @staticmethod
    def backward(ctx, grad_output):
        ind3d, ind2d = ctx.saved_tensors
        C = grad_output.shape[0]
        grad = grad_output.new_zeros((C,) + (tuple(ctx.shape[-2:]) if len(ctx.shape) >= 2 else ()))
        n = int(ind3d[0])
        if n > 0:
            vals = torch.index_select(grad_output.contiguous(), 1, ind3d[1:1 + n])
            grad.reshape(C, -1).index_put_((torch.arange(C, device=grad.device)[:, None], ind2d[1:1 + n][None, :]),
                                           vals, accumulate=True)
        return grad.reshape(ctx.shape), None, None, None
