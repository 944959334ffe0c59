"""numpy restatement of the whole-scene protocol of pn2_b200/whole_scene.py (TEST INFRASTRUCTURE ONLY: tests/ compare the
device against it).

Evaluation blocks follow the PointNet++ ScanNet whole-scene loader: a loop over 1.5 m columns (i outer, j inner), boolean
masks for the 0.2 m padded block and its 0.001 m core, `npoints` draws with replacement, blocks with < 1 % core draws
dropped.  np.random.choice is replaced by a seeded counter hash so that device and oracle draw the same indices.
Labelling covers every non-empty padded block with strided chunks and votes once per (block, point).
"""
import numpy as np

BLOCK, PAD, CORE, MIN_CORE = 1.5, 0.2, 0.001, 0.01
_GOLDEN = np.uint64(0x9E3779B97F4A7C15)


def mix(x):
    """splitmix64 finaliser on uint64 arrays (wrapping arithmetic)"""
    x = np.asarray(x, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
    return x


def slot_hash(seed, block_id, slots):
    """h = mix(seed * 0x9E3779B97F4A7C15 + ((block_id << 32) | slot)) for each slot, uint64"""
    s = np.asarray(slots, dtype=np.uint64)
    with np.errstate(over="ignore"):
        base = np.array([seed], dtype=np.uint64) * _GOLDEN
        return mix(base + ((np.uint64(block_id) << np.uint64(32)) | s))


def sample_positions(seed, block_id, npoints, count):
    """segment positions read by slots 0 .. npoints-1: ((h >> 32) * count) >> 32"""
    h = slot_hash(seed, block_id, np.arange(npoints))
    return ((h >> np.uint64(32)) * np.uint64(count)) >> np.uint64(32)


def grid(xyz):
    """-> cmin (3,) fp32, cmax (3,) fp32, nx, ny"""
    cmin, cmax = xyz.min(axis=0), xyz.max(axis=0)
    ext = cmax - cmin  # fp32 subtraction
    nx = int(np.ceil(np.float64(ext[0]) / BLOCK))
    ny = int(np.ceil(np.float64(ext[1]) / BLOCK))
    return cmin, cmax, nx, ny


def _box(cmin, i, j):
    """the loader's curmin / curmax of column (i, j) in x and y: fp32 minimum widened, plus a Python float"""
    lo = np.array([np.float64(cmin[0]) + i * BLOCK, np.float64(cmin[1]) + j * BLOCK])
    hi = np.array([np.float64(cmin[0]) + (i + 1) * BLOCK, np.float64(cmin[1]) + (j + 1) * BLOCK])
    return lo, hi


def _inside(xy, lo, hi, margin):
    # z sets no condition: the loader's z range [cmin_z, cmin_z + fl32(cmax_z - cmin_z)] holds every point with room to spare
    return np.sum((xy >= (lo - margin)) * (xy <= (hi + margin)), axis=1) == 2


def segments(xyz):
    """Step 1-2: list of (block_id, scene indices of the padded block ascending, core mask) for every block, empty ones
    included, in block_id order.  Raises ValueError on a zero extent."""
    cmin, _, nx, ny = grid(xyz)
    if nx == 0 or ny == 0:
        raise ValueError("scene has zero extent in x or y")
    xy = xyz[:, :2].astype(np.float64)
    out = []
    for i in range(nx):
        for j in range(ny):
            lo, hi = _box(cmin, i, j)
            idx = np.nonzero(_inside(xy, lo, hi, PAD))[0]
            core = _inside(xy[idx], lo, hi, CORE)
            out.append((i * ny + j, idx, core))
    return out


def scene_blocks(xyz, feats, labels=None, labelweights=None, npoints=8192, seed=0):
    """Steps 1-5 -> dict block_id (nb,), point_index (nb, npoints), points (nb, npoints, 3 + C), target (nb, npoints)
    int64 or None, weights (nb, npoints) fp32."""
    rows = np.concatenate([xyz, feats], axis=1).astype(np.float32)
    kept, index, target, weights = [], [], [], []
    for b, idx, core in segments(xyz):
        if len(idx) == 0:
            continue
        choice = sample_positions(seed, b, npoints, len(idx)).astype(np.int64)
        mask = core[choice]
        if np.sum(mask) / float(len(mask)) < MIN_CORE:
            continue
        pidx = idx[choice]
        w = mask.astype(np.float32)
        if labels is not None:
            t = labels[pidx].astype(np.int64)
            target.append(t)
            if labelweights is not None:
                w = labelweights.astype(np.float32)[t] * w
        kept.append(b)
        index.append(pidx)
        weights.append(w)
    if not kept:
        raise ValueError("no block of the scene has enough core points")
    index = np.stack(index).astype(np.int32)
    return {"block_id": np.array(kept, dtype=np.int64), "point_index": index, "points": rows[index],
            "target": np.stack(target) if labels is not None else None, "weights": np.stack(weights).astype(np.float32)}


def scene_chunks(xyz, feats, npoints=8192):
    """Step 6 cover -> point_index (n_chunks, npoints) int32, sizes (n_chunks,) int32, points (n_chunks, npoints, 3 + C)"""
    rows = np.concatenate([xyz, feats], axis=1).astype(np.float32)
    index, sizes = [], []
    for _, idx, _ in segments(xyz):
        count = len(idx)
        if count == 0:
            continue
        k = -(-count // npoints)
        for c in range(k):
            size = -(-(count - c) // k)
            index.append(idx[c + k * (np.arange(npoints) % size)])
            sizes.append(size)
    index = np.stack(index).astype(np.int32)
    return index, np.array(sizes, dtype=np.int32), rows[index]


def scene_votes(point_index, sizes, pred, n, num_classes):
    """votes (n, num_classes) int32: one per valid slot (s < sizes[chunk]) at [point, pred]"""
    votes = np.zeros((n, num_classes), dtype=np.int32)
    valid = np.arange(point_index.shape[1])[None, :] < sizes[:, None]
    np.add.at(votes, (point_index[valid], pred[valid].astype(np.int64)), 1)
    return votes


def padded_block_count(xyz):
    """number of padded blocks holding each point"""
    cnt = np.zeros(xyz.shape[0], dtype=np.int64)
    for _, idx, _ in segments(xyz):
        cnt[idx] += 1
    return cnt
