"""Whole-scene segmentation on the device: from a whole scan to the 1.5 m columns the networks take, and back to one
label per scan point.

- `scene_blocks` is the evaluation tiling of the PointNet++ ScanNet whole-scene loader (train_scannet_semseg.py:182-237
  evaluates on it): 1.5 m blocks in x / y padded by 0.2 m, `npoints` draws per block with replacement, weights =
  labelweights[label] * "inside the block's 0.001 m core", blocks with fewer than 1 % core draws dropped.  Its output
  feeds `predict()` and `pc_util.EvalCounters` directly.
- `segment_scene` labels every point: every non-empty padded block is cut into strided chunks of `npoints` that cover
  all of its points, each chunk is classified with `predict()`, and every (block, point) casts one vote.
- `SceneBank.crops` is the training side (ScanNetDataLoader.py:394-418, as train_scannet_semseg.py:64 uses it): per
  crop up to ten random 1.5 m columns of a scene held on the device, the first that is >= 70 % labelled and whose core
  occupies >= 2 % of its 31 x 31 x 62 voxels, then `npoints` draws with replacement from the column padded by 0.2 m.

The draws use a seeded counter hash instead of np.random.choice, so a run is reproducible and oracle/whole_scene_ref.py
and oracle/scene_crops_ref.py restate it exactly.  Block cutting, sampling, gathering, voting and cropping are kernels
of csrc/scene_blocks.cu.  The evaluation side reads one 40-byte record per scene for the block or chunk count: its
output sizes depend on the data, so it is not graph-captured.  Training crops have a fixed shape, read nothing back
and can be captured in a CUDA graph.
"""
import collections

import numpy as np
import torch

from . import _lib
from ._lib import Pn2Error, ptr

BLOCK, PAD, CORE, MIN_CORE = 1.5, 0.2, 0.001, 0.01  # the kernels' constants (csrc/scene_blocks.cu)
MAX_BLOCKS = 1 << 16

SceneBlocks = collections.namedtuple("SceneBlocks", "points target weights block_id point_index")
SceneBlocks.__doc__ = """Kept evaluation blocks in ascending block id (= i * ny + j): points (nb, npoints, 3 + C) fp32
[xyz | feats] rows, target (nb, npoints) int64 (None without labels), weights (nb, npoints) fp32, block_id (nb,) int64,
point_index (nb, npoints) int32 = scene index of each row."""


def _scene(xyz, feats):
    _lib.require_cuda(xyz, feats)
    if xyz.dim() != 2 or xyz.shape[1] != 3:
        raise Pn2Error("xyz must be (N, 3) (got %s)" % (tuple(xyz.shape),))
    if feats.dim() != 2 or feats.shape[0] != xyz.shape[0]:
        raise Pn2Error("feats must be (N, C) with N = %d (got %s)" % (xyz.shape[0], tuple(feats.shape)))
    return _lib.check_f32(xyz, "xyz"), _lib.check_f32(feats, "feats")


def _index(xyz):
    """pn2_scene_index -> grid record (pn2_scene_grid, 10 words), seg_start, pos"""
    n = xyz.shape[0]
    dev = xyz.device
    grid = torch.empty(10, dtype=torch.int32, device=dev)
    seg_start = torch.empty(MAX_BLOCKS + 2, dtype=torch.int32, device=dev)
    # a size the library refuses gets no buffer: the call reports it instead of a huge allocation
    pos = torch.empty(4 * n, dtype=torch.int32, device=dev) if 1 <= 4 * n < 1 << 31 else None
    _lib.call("pn2_scene_index", n, ptr(xyz), ptr(grid), ptr(seg_start), ptr(pos), _lib.stream_ptr(dev))
    return grid, seg_start, pos


def _read_grid(grid):
    """The one host read of a pass: (nx, ny, count)."""
    nx, ny, count = (int(v) for v in grid[6:9].cpu())
    if nx == 0 or ny == 0:
        raise ValueError("the scene has zero extent in x or y: there is no 1.5 m block to cut")
    return nx, ny, count


def scene_blocks(xyz, feats, labels=None, labelweights=None, npoints=8192, seed=0):
    """xyz (N, 3) fp32, feats (N, C) fp32, labels (N,) integer or None, labelweights (num_classes,) fp32 or None (ones),
    cuda tensors -> SceneBlocks.  Labels outside [0, num_classes) get weight 0.  Raises ValueError when the scene has zero
    extent in x or y or no block keeps 1 % core points, Pn2Error for bad arguments (CPU tensors, npoints < 1, N == 0,
    4N >= 2^31, more than 2^16 blocks)."""
    xyz, feats = _scene(xyz, feats)
    _lib.require_cuda(labels, labelweights)
    n, c = xyz.shape[0], feats.shape[1]
    if labels is not None:
        if labels.shape != (n,) or labels.dtype.is_floating_point or labels.dtype == torch.bool:
            raise Pn2Error("labels must be (N,) integer (got %s %s)" % (tuple(labels.shape), labels.dtype))
        labels = labels.to(torch.int64).contiguous()
    if labelweights is not None:
        if labels is None:
            raise Pn2Error("labelweights need labels")
        if labelweights.dim() != 1:
            raise Pn2Error("labelweights must be (num_classes,)")
        labelweights = _lib.check_f32(labelweights, "labelweights")
    if not 0 <= int(seed) < 1 << 64:
        raise Pn2Error("seed must be in [0, 2^64)")
    dev = xyz.device
    with torch.cuda.device(dev):
        st = _lib.stream_ptr(dev)
        grid, seg_start, pos = _index(xyz)
        kept = torch.empty(MAX_BLOCKS, dtype=torch.int32, device=dev)
        _lib.call("pn2_scene_keep", int(npoints), int(seed), ptr(xyz), ptr(grid), ptr(seg_start), ptr(pos), ptr(kept), st)
        nx, ny, nb = _read_grid(grid)
        point_index = torch.empty((nb, npoints), dtype=torch.int32, device=dev)
        points = torch.empty((nb, npoints, 3 + c), dtype=torch.float32, device=dev)
        target = None if labels is None else torch.empty((nb, npoints), dtype=torch.int64, device=dev)
        weights = torch.empty((nb, npoints), dtype=torch.float32, device=dev)
        num_classes = 0 if labelweights is None else labelweights.shape[0]
        _lib.call("pn2_scene_sample", nx, ny, nb, int(npoints), int(seed), c, ptr(xyz), ptr(feats), ptr(labels), ptr(labelweights),
                  num_classes, ptr(grid), ptr(seg_start), ptr(pos), ptr(kept), ptr(point_index), ptr(points), ptr(target),
                  ptr(weights), st)
        if nb == 0:
            raise ValueError("no block of the scene keeps %g of its samples in its core" % MIN_CORE)
        return SceneBlocks(points, target, weights, kept[:nb].to(torch.int64), point_index)


def scene_chunks(xyz, feats, npoints=8192):
    """The labelling cover: every non-empty padded block with count points is cut into k = ceil(count / npoints) chunks,
    chunk c holding its segment positions c, c+k, c+2k, ... (ascending scene index), padded to npoints by repeating them.
    -> points (n_chunks, npoints, 3 + C) fp32, point_index (n_chunks, npoints) int32, sizes (n_chunks,) int32 (the
    number of distinct leading slots of each chunk), chunks in (block id, c) order."""
    xyz, feats = _scene(xyz, feats)
    c = feats.shape[1]
    dev = xyz.device
    with torch.cuda.device(dev):
        st = _lib.stream_ptr(dev)
        grid, seg_start, pos = _index(xyz)
        first = torch.empty(MAX_BLOCKS + 1, dtype=torch.int32, device=dev)
        _lib.call("pn2_scene_chunks", int(npoints), ptr(grid), ptr(seg_start), ptr(first), st)
        nx, ny, n_chunks = _read_grid(grid)
        point_index = torch.empty((n_chunks, npoints), dtype=torch.int32, device=dev)
        sizes = torch.empty((n_chunks,), dtype=torch.int32, device=dev)
        points = torch.empty((n_chunks, npoints, 3 + c), dtype=torch.float32, device=dev)
        _lib.call("pn2_scene_chunk_rows", nx, ny, n_chunks, int(npoints), c, ptr(xyz), ptr(feats), ptr(grid), ptr(seg_start), ptr(pos),
                  ptr(first), ptr(point_index), ptr(sizes), ptr(points), st)
    return points, point_index, sizes


def _votes(point_index, sizes, pred_u8, n, num_classes, labels):
    _lib.require_cuda(point_index, sizes, pred_u8)
    point_index, sizes = _lib.check_i32(point_index, "point_index"), _lib.check_i32(sizes, "sizes")
    if pred_u8.dtype != torch.uint8 or pred_u8.shape != point_index.shape or sizes.shape != point_index.shape[:1]:
        raise Pn2Error("pred_u8 must be uint8 shaped like point_index (n_chunks, npoints), sizes (n_chunks,)")
    pred_u8 = pred_u8.contiguous()
    dev = point_index.device
    votes = torch.empty((n, num_classes), dtype=torch.int32, device=dev)
    out = torch.empty((n,), dtype=torch.uint8, device=dev) if labels else None
    with torch.cuda.device(dev):
        _lib.call("pn2_scene_votes", point_index.shape[0], point_index.shape[1], ptr(point_index), ptr(sizes), ptr(pred_u8), int(n),
                  int(num_classes), ptr(votes), ptr(out), _lib.stream_ptr(dev))
    return votes, out


def scene_votes(point_index, sizes, pred_u8, n, num_classes):
    """votes (n, num_classes) int32: one vote votes[point, pred] for every slot s < sizes[chunk] of the chunks of
    scene_chunks (so a point gets exactly one vote from every padded block holding it); integer atomics, exact."""
    return _votes(point_index, sizes, pred_u8, n, num_classes, False)[0]


def segment_scene(net, xyz, feats, npoints=8192, batch=32):
    """One label per scene point: scene_chunks, then net.predict over groups of at most `batch` chunks (under the current
    set_mlp_precision), then scene_votes and the first-maximum arg-max of the votes (the lowest class wins a tie, as with
    np.argmax).  net: a PointNet2SemSeg (a module with predict(xyz, points)) in eval().
    -> labels (N,) uint8, votes (N, num_classes) int32."""
    if net.training:
        raise ValueError("segment_scene needs the network in eval()")
    if batch < 1:
        raise ValueError("batch must be >= 1")
    points, point_index, sizes = scene_chunks(xyz, feats, npoints)
    num_classes = net.conv2.out_channels
    preds = torch.empty(point_index.shape, dtype=torch.uint8, device=points.device)
    with torch.no_grad():
        for s in range(0, points.shape[0], batch):
            x = points[s:s + batch].permute(0, 2, 1)
            preds[s:s + batch] = net.predict(x[:, :3], x[:, 3:])
    votes, labels = _votes(point_index, sizes, preds, xyz.shape[0], num_classes, True)
    return labels, votes


SceneCrops = collections.namedtuple("SceneCrops", "points target weights point_index center tries valid")
SceneCrops.__doc__ = """One training batch of B crops: points (B, npoints, 3 + C) fp32 [xyz | feats] rows, target (B, npoints)
int64 labels, weights (B, npoints) fp32, point_index (B, npoints) int32 bank rows, center (B,) int32 scene-local index of
the column's centre, tries (B,) int32 in 1..10 (the try taken), valid (B,) uint8 (whether that try passed the loader's
test; the tenth is taken when none does).  A crop whose scene id lies outside [0, S) has tries = 0, valid = 0,
center = -1, point_index = -1 and zero rows, targets and weights."""


class SceneBank:
    """S scenes resident on the device, the source of training crops.

        bank = SceneBank(xyz, feats, labels, offsets)   # packed: scene k = rows offsets[k] .. offsets[k + 1]
        lw = bank.label_weights(21)
        crops = bank.crops(scene_ids, lw)               # scene_ids (B,) int32 cuda

    xyz (N, 3) fp32, feats (N, C) fp32, labels (N,) int64, offsets (S + 1,) int64, all cuda tensors.  The constructor
    validates them once on the host (offsets strictly increasing from 0 to N) and computes per-scene bounds.  `step` is
    a device int64 counter: every `crops` call draws with it and increments it on the stream, so consecutive calls and
    the replays of a captured graph draw new batches, and `bank.step.fill_(k)` replays the draws of call k."""

    def __init__(self, xyz, feats, labels, offsets):
        _lib.require_cuda(xyz, feats, labels, offsets)
        xyz, feats = _scene(xyz, feats)
        n = xyz.shape[0]
        if labels.shape != (n,) or labels.dtype != torch.int64:
            raise Pn2Error("labels must be (N,) int64 with N = %d (got %s %s)" % (n, tuple(labels.shape), labels.dtype))
        if offsets.dim() != 1 or offsets.shape[0] < 2 or offsets.dtype != torch.int64:
            raise Pn2Error("offsets must be (S + 1,) int64 with S >= 1 (got %s %s)" % (tuple(offsets.shape), offsets.dtype))
        if n >= 1 << 31:
            raise Pn2Error("a bank holds fewer than 2^31 points (got %d)" % n)
        off = offsets.cpu()
        sizes = off[1:] - off[:-1]
        if int(off[0]) != 0 or int(off[-1]) != n or not bool((sizes > 0).all()):
            raise Pn2Error("offsets must increase strictly from 0 to N = %d" % n)
        self.xyz, self.feats, self.labels, self.offsets = xyz, feats, labels.contiguous(), offsets.contiguous()
        self.num_scenes, self.max_count = int(off.shape[0]) - 1, int(sizes.max())
        dev = xyz.device
        self.bounds = torch.empty((self.num_scenes, 6), dtype=torch.float32, device=dev)
        self.step = torch.zeros(1, dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            _lib.call("pn2_scene_bank_bounds", self.num_scenes, n, ptr(self.xyz), ptr(self.offsets), ptr(self.bounds), _lib.stream_ptr(dev))

    def label_weights(self, num_classes=21):
        """The loader's train-split class weights, (num_classes,) fp32 cuda: w = histogram of all labels over bins
        0 .. num_classes - 1 (the last bin closed, so a label equal to num_classes counts in it), w = fl32(w) / sum(w),
        1 / log(1.2 + w).  The counts are taken on the device; the num_classes-element formula runs in numpy float32, so
        it equals the loader's numbers exactly."""
        if num_classes < 1:
            raise ValueError("num_classes must be >= 1")
        lab = self.labels[(self.labels >= 0) & (self.labels <= num_classes)].clamp(max=num_classes - 1)
        w = torch.bincount(lab, minlength=num_classes).cpu().numpy().astype(np.float32)
        w = w / np.sum(w)
        w = (1 / np.log(1.2 + w)).astype(np.float32)
        return torch.from_numpy(w).to(self.xyz.device)

    def crops(self, scene_ids, labelweights=None, npoints=8192, seed=0):
        """scene_ids (B,) int32 cuda, labelweights (num_classes,) fp32 cuda or None -> SceneCrops.  weights =
        labelweights[target] * core, or the core mask without labelweights, 0 for a label outside [0, num_classes).
        Makes no host read and no synchronisation (capturable in a CUDA graph).  Pn2Error for bad arguments: CPU
        tensors, B < 1, npoints < 1, B * npoints >= 2^31."""
        _lib.require_cuda(scene_ids, labelweights)
        scene_ids = _lib.check_i32(scene_ids, "scene_ids")
        if scene_ids.dim() != 1:
            raise Pn2Error("scene_ids must be (B,) int32 (got %s)" % (tuple(scene_ids.shape),))
        if labelweights is not None:
            if labelweights.dim() != 1:
                raise Pn2Error("labelweights must be (num_classes,)")
            labelweights = _lib.check_f32(labelweights, "labelweights")
        if not 0 <= int(seed) < 1 << 64:
            raise Pn2Error("seed must be in [0, 2^64)")
        b, c, dev = scene_ids.shape[0], self.feats.shape[1], self.xyz.device
        if b < 1 or npoints < 1 or b * npoints >= 1 << 31:  # no buffers for a size the library refuses
            point_index = points = target = weights = center = tries = valid = None
        else:
            point_index = torch.empty((b, npoints), dtype=torch.int32, device=dev)
            points = torch.empty((b, npoints, 3 + c), dtype=torch.float32, device=dev)
            target = torch.empty((b, npoints), dtype=torch.int64, device=dev)
            weights = torch.empty((b, npoints), dtype=torch.float32, device=dev)
            center = torch.empty((b,), dtype=torch.int32, device=dev)
            tries = torch.empty((b,), dtype=torch.int32, device=dev)
            valid = torch.empty((b,), dtype=torch.uint8, device=dev)
        num_classes = 0 if labelweights is None else labelweights.shape[0]
        with torch.cuda.device(dev):
            _lib.call("pn2_scene_crops", self.num_scenes, self.xyz.shape[0], c, self.max_count, ptr(self.xyz), ptr(self.feats),
                      ptr(self.labels), ptr(self.offsets), ptr(self.bounds), b, ptr(scene_ids), int(npoints), int(seed),
                      ptr(self.step), ptr(labelweights), num_classes, ptr(point_index), ptr(points), ptr(target), ptr(weights),
                      ptr(center), ptr(tries), ptr(valid), _lib.stream_ptr(dev))
        return SceneCrops(points, target, weights, point_index, center, tries, valid)
