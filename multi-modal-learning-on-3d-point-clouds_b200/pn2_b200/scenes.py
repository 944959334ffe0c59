"""Synthetic inputs shaped like the reference's data (there is no network access for ScanNet / nuScenes).

scannet_scene follows the crop logic of data_utils/ScanNetDataLoader.py:394-418: a 1.5 m-class column
of an indoor scan in ABSOLUTE scene coordinates (not normalised), from which `npoints` points are
drawn WITH replacement (:410) -- so exact duplicates, hence exact FPS ties, are the norm.
Generators are numpy-only and seeded: the same (scene_id, npoints) always gives the same arrays.
"""
import numpy as np


def _surface_points(rng, n_surface):
    """Points on a floor, two walls and a few boxes inside a 1.9 x 1.9 x 2.7 m column (local frame)."""
    sx, sy, sz = 1.9, 1.9, 2.7
    parts = []
    n_floor = int(n_surface * 0.35)
    parts.append(np.stack([rng.uniform(0, sx, n_floor), rng.uniform(0, sy, n_floor), np.zeros(n_floor)], 1))
    n_wall = int(n_surface * 0.2)
    parts.append(np.stack([np.zeros(n_wall), rng.uniform(0, sy, n_wall), rng.uniform(0, sz, n_wall)], 1))
    parts.append(np.stack([rng.uniform(0, sx, n_wall), np.zeros(n_wall), rng.uniform(0, sz, n_wall)], 1))
    n_boxes = int(rng.integers(3, 7))
    remaining = n_surface - n_floor - 2 * n_wall
    per_box = max(remaining // n_boxes, 1)
    for _ in range(n_boxes):
        size = rng.uniform([0.2, 0.2, 0.2], [0.8, 0.8, 1.2])
        org = rng.uniform([0.05, 0.05, 0.0], [sx - size[0] - 0.05, sy - size[1] - 0.05, 0.3])
        # sample the five visible faces of the box
        face = rng.integers(0, 5, per_box)
        u, v = rng.uniform(0, 1, per_box), rng.uniform(0, 1, per_box)
        p = np.zeros((per_box, 3))
        top = face == 0
        p[top] = np.stack([u[top] * size[0], v[top] * size[1], np.full(top.sum(), size[2])], 1)
        for f, (ax_fixed, val) in zip((1, 2, 3, 4), ((0, 0.0), (0, size[0]), (1, 0.0), (1, size[1]))):
            msk = face == f
            other = 1 - ax_fixed
            q = np.zeros((msk.sum(), 3))
            q[:, ax_fixed] = val
            q[:, other] = u[msk] * size[other]
            q[:, 2] = v[msk] * size[2]
            p[msk] = q
        parts.append(p + org)
    pts = np.concatenate(parts, 0)
    pts += rng.normal(0.0, 0.005, pts.shape)  # 5 mm sensor noise
    return pts


def scannet_scene(scene_id, npoints=8192, n_surface=20000):
    """-> (xyz (npoints, 3) float32 absolute coordinates, rgb (npoints, 3) float32 in [-0.5, 0.5])"""
    rng = np.random.default_rng(1000 + int(scene_id))
    pts = _surface_points(rng, n_surface)
    origin = np.array([rng.uniform(0, 6), rng.uniform(0, 6), 0.0])
    pts = pts + origin
    choice = rng.choice(pts.shape[0], npoints, replace=True)
    xyz = pts[choice].astype(np.float32)
    rgb = rng.uniform(-0.5, 0.5, (npoints, 3)).astype(np.float32)
    return xyz, rgb


def scannet_batch(first_scene_id, batch, npoints=8192):
    """-> points (batch, npoints, 6) float32 [xyz | rgb], the loader's layout (train_scannet_semseg.py:123)"""
    out = np.empty((batch, npoints, 6), dtype=np.float32)
    for i in range(batch):
        xyz, rgb = scannet_scene(first_scene_id + i, npoints)
        out[i, :, :3], out[i, :, 3:] = xyz, rgb
    return out


def scannet_room(scene_id, n_points, extent):
    """A whole synthetic room, the input of pn2_b200.whole_scene: a floor, four walls and furniture boxes in a room of
    extent x (0.6 .. 1) * extent metres (extent > 0.5), 2.7 m high, with 5 mm sensor noise.
    -> (xyz (n_points, 3) float32 absolute coordinates, rgb (n_points, 3) float32 in [-0.5, 0.5], labels (n_points,)
    int64: floor 1, walls 2, each box one class in 3..20, and about 5 % unannotated points (label 0) on every surface)."""
    rng = np.random.default_rng(5000 + int(scene_id))
    sx, sy, sz = float(extent), float(extent) * rng.uniform(0.6, 1.0), 2.7
    n_floor, n_wall = int(n_points * 0.3), int(n_points * 0.1)
    n_box_total = n_points - n_floor - 4 * n_wall
    parts, labels = [], []
    parts.append(np.stack([rng.uniform(0, sx, n_floor), rng.uniform(0, sy, n_floor), np.zeros(n_floor)], 1))
    labels.append(np.full(n_floor, 1))
    for ax, val in ((0, 0.0), (0, sx), (1, 0.0), (1, sy)):
        w = np.empty((n_wall, 3))
        w[:, ax] = val
        w[:, 1 - ax] = rng.uniform(0, sy if ax == 0 else sx, n_wall)
        w[:, 2] = rng.uniform(0, sz, n_wall)
        parts.append(w)
        labels.append(np.full(n_wall, 2))
    n_boxes = max(int(sx * sy / 4), 3)
    counts = np.full(n_boxes, n_box_total // n_boxes)
    counts[: n_box_total - counts.sum()] += 1
    for cnt in counts:
        size = rng.uniform(0.2, 1.0, 3) * np.array([min(1.5, sx / 2), min(1.5, sy / 2), 1.5])
        org = np.array([rng.uniform(0.05, sx - size[0] - 0.05), rng.uniform(0.05, sy - size[1] - 0.05), 0.0])
        u, v, face = rng.uniform(0, 1, cnt), rng.uniform(0, 1, cnt), rng.integers(0, 5, cnt)
        p = np.stack([u * size[0], v * size[1], np.full(cnt, size[2])], 1)  # top face
        for f, (ax, val) in zip((1, 2, 3, 4), ((0, 0.0), (0, size[0]), (1, 0.0), (1, size[1]))):
            m = face == f
            p[m, ax] = val
            p[m, 1 - ax] = u[m] * size[1 - ax]
            p[m, 2] = v[m] * size[2]
        parts.append(p + org)
        labels.append(np.full(cnt, rng.integers(3, 21)))
    xyz = np.concatenate(parts, 0) + rng.normal(0.0, 0.005, (n_points, 3))
    xyz += np.array([rng.uniform(-5, 5), rng.uniform(-5, 5), 0.0])
    labels = np.concatenate(labels).astype(np.int64)
    labels[rng.random(n_points) < 0.05] = 0
    perm = rng.permutation(n_points)  # scan order is not surface order
    rgb = (rng.uniform(-0.5, 0.5, (n_points, 3)) * 0.2 + (labels[:, None] * np.array([0.37, 0.61, 0.83])) % 1.0 - 0.5).clip(-0.5, 0.5)
    return xyz[perm].astype(np.float32), rgb[perm].astype(np.float32), labels[perm]


def lidar_sweep(scene_id, npoints=None):
    """nuScenes-shaped synthetic 32-beam sweep (data_utils/NuScenesDataLoader.py:462-473): rays at
    elevations -30.67..+10.67 deg x 1085 azimuths onto a ground plane at z=-1.84 m plus boxes, range
    < 52 m.  -> (xyz (n, 3), feat (n, 2) = [intensity in [0,1], time in [0,0.5]]); n ~ 30-35k, or
    exactly `npoints` (sub/over-sampled with replacement) when given."""
    rng = np.random.default_rng(4000 + int(scene_id))
    elev = np.deg2rad(np.linspace(-30.67, 10.67, 32))
    azim = np.linspace(-np.pi, np.pi, 1085, endpoint=False)
    e, a = np.meshgrid(elev, azim, indexing="ij")
    d = np.stack([np.cos(e) * np.cos(a), np.cos(e) * np.sin(a), np.sin(e)], -1).reshape(-1, 3)
    rng_max = 52.0
    t = np.full(d.shape[0], np.inf)
    down = d[:, 2] < -1e-3
    t[down] = -1.84 / d[down, 2]
    n_boxes = int(rng.integers(20, 41))
    for _ in range(n_boxes):
        c = np.array([rng.uniform(-40, 40), rng.uniform(-40, 40), -1.84])
        s = rng.uniform([1.5, 1.5, 1.2], [6.0, 2.5, 3.0])
        lo, hi = c - np.array([s[0] / 2, s[1] / 2, 0]), c + np.array([s[0] / 2, s[1] / 2, s[2]])
        with np.errstate(divide="ignore", invalid="ignore"):
            t0, t1 = lo / d, hi / d
        tmin = np.nanmax(np.minimum(t0, t1), axis=1)
        tmax = np.nanmin(np.maximum(t0, t1), axis=1)
        hit = (tmax >= tmin) & (tmin > 0.5)
        t = np.where(hit & (tmin < t), tmin, t)
    keep = np.isfinite(t) & (t < rng_max)
    xyz = (d[keep] * t[keep, None] + rng.normal(0, 0.02, (keep.sum(), 3))).astype(np.float32)
    if npoints is not None:
        xyz = xyz[rng.choice(xyz.shape[0], npoints, replace=xyz.shape[0] < npoints)]
    feat = np.stack([rng.uniform(0, 1, xyz.shape[0]), rng.uniform(0, 0.5, xyz.shape[0])], 1).astype(np.float32)
    return xyz, feat


def uniform_cloud(seed, n, scale=1.0):
    """Microbench cloud: n points uniform in [0, scale)^3 (SURVEY.md 8d config 5)."""
    rng = np.random.default_rng(seed)
    return (rng.random((n, 3)) * scale).astype(np.float32)


# ---- multi-view inputs (SURVEY.md 8d config 3) -------------------------------------------------------

SCANNET_INTRINSIC = np.array([[37.01983, 0, 20, 0], [0, 38.52470, 15.5, 0], [0, 0, 1, 0], [0, 0, 0, 1]], dtype=np.float32)
SCANNET_IMAGE_DIMS = [41, 32]          # [W, H]  (train_scannet_multiview_semseg.py:109-110)
SCANNET_DEPTH_RANGE = (0.1, 4.0)
SCANNET_ACCURACY = 0.05


def look_at_pose(eye, target):
    """camera_to_world (4, 4) of a pinhole camera at `eye` looking at `target` (x right, y down, z forward)."""
    fwd = target - eye
    fwd = fwd / np.linalg.norm(fwd)
    right = np.cross(fwd, np.array([0.0, 0.0, 1.0]))
    right = right / np.linalg.norm(right)
    down = np.cross(fwd, right)
    m = np.eye(4)
    m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = right, down, fwd, eye
    return m.astype(np.float32)


def multiview_inputs(scene_id, xyz, num_views=3, channels=128):
    """Poses, z-buffered depth maps and random feature maps for one scene.

    xyz (N, 3).  Cameras sit 1.5-3 m from the column centre looking at it; each depth map is the
    z-buffer of the scene's own points on the 41x32 grid, so front-most points pass the 0.05 m test.
    -> feats (V, C, 32, 41) ~ N(0,1), depth (V, 32, 41), poses (V, 4, 4)"""
    rng = np.random.default_rng(3000 + int(scene_id))
    W, H = SCANNET_IMAGE_DIMS
    fx, fy, cx, cy = SCANNET_INTRINSIC[0, 0], SCANNET_INTRINSIC[1, 1], SCANNET_INTRINSIC[0, 2], SCANNET_INTRINSIC[1, 2]
    centre = xyz.mean(0).astype(np.float64)
    poses, depths = [], []
    for _ in range(num_views):
        ang = rng.uniform(0, 2 * np.pi)
        dist = rng.uniform(1.5, 3.0)
        eye = centre + np.array([np.cos(ang) * dist, np.sin(ang) * dist, rng.uniform(0.3, 1.5)])
        pose = look_at_pose(eye, centre)
        w2c = np.linalg.inv(pose.astype(np.float64))
        cam = xyz.astype(np.float64) @ w2c[:3, :3].T + w2c[:3, 3]
        z = cam[:, 2]
        with np.errstate(divide="ignore", invalid="ignore"):
            u = np.rint(cam[:, 0] * fx / z + cx)
            v = np.rint(cam[:, 1] * fy / z + cy)
        ok = (z > 0.05) & (u >= 0) & (u < W) & (v >= 0) & (v < H)
        depth = np.full(H * W, np.inf)
        np.minimum.at(depth, (v[ok] * W + u[ok]).astype(np.int64), z[ok])
        depth[~np.isfinite(depth)] = 0.0
        poses.append(pose)
        depths.append(depth.reshape(H, W).astype(np.float32))
    feats = rng.standard_normal((num_views, channels, H, W)).astype(np.float32)
    return feats, np.stack(depths), np.stack(poses)
