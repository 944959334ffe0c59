"""Whole-scene segmentation on the device (csrc/scene_blocks.cu, pn2_b200/whole_scene.py) bit-exact against the numpy
restatement of the protocol (oracle/whole_scene_ref.py): block order, index maps, rows, targets, weights, chunk tables
and votes; boundary points, the 1 % core threshold, empty blocks, errors; segment_scene and the evaluation counters."""
import numpy as np
import pytest
import torch

from oracle import pc_util_ref
from oracle import whole_scene_ref as ref
from pn2_b200 import Pn2Error, pc_util, scenes, whole_scene
from pn2_b200.models import PointNet2SemSeg
from pn2_b200.pointnet_util import set_mlp_precision

pytestmark = pytest.mark.gpu

C = 21
LABELWEIGHTS = (1.0 + np.arange(C) / 7.0).astype(np.float32) ** 1.5  # non-uniform


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def check_blocks(dev, xyz, feats, labels=None, labelweights=None, npoints=8192, seed=0):
    want = ref.scene_blocks(xyz, feats, labels, labelweights, npoints, seed)
    got = whole_scene.scene_blocks(_t(xyz, dev), _t(feats, dev), None if labels is None else _t(labels, dev),
                                   None if labelweights is None else _t(labelweights, dev), npoints, seed)
    np.testing.assert_array_equal(got.block_id.cpu().numpy(), want["block_id"])
    np.testing.assert_array_equal(got.point_index.cpu().numpy(), want["point_index"])
    np.testing.assert_array_equal(got.points.cpu().numpy(), want["points"])
    np.testing.assert_array_equal(got.weights.cpu().numpy(), want["weights"])
    if labels is None:
        assert got.target is None
    else:
        np.testing.assert_array_equal(got.target.cpu().numpy(), want["target"])
    return got, want


def check_chunks(dev, xyz, feats, npoints=8192):
    index, sizes, pts = ref.scene_chunks(xyz, feats, npoints)
    got_pts, got_index, got_sizes = whole_scene.scene_chunks(_t(xyz, dev), _t(feats, dev), npoints)
    np.testing.assert_array_equal(got_index.cpu().numpy(), index)
    np.testing.assert_array_equal(got_sizes.cpu().numpy(), sizes)
    np.testing.assert_array_equal(got_pts.cpu().numpy(), pts)
    # votes of arbitrary predictions, and every point votes once per padded block holding it
    rng = np.random.default_rng(1)
    pred = rng.integers(0, C, index.shape).astype(np.uint8)
    votes = whole_scene.scene_votes(got_index, got_sizes, _t(pred, dev), xyz.shape[0], C).cpu().numpy()
    np.testing.assert_array_equal(votes, ref.scene_votes(index, sizes, pred, xyz.shape[0], C))
    np.testing.assert_array_equal(votes.sum(1), ref.padded_block_count(xyz))
    return got_index, got_sizes


@pytest.mark.parametrize("room,n,extent,npoints", [(0, 3000, 1.0, 8192), (1, 100000, 5.0, 8192), (2, 250000, 9.5, 8192),
                                                   (3, 60000, 6.0, 1024)])
def test_rooms_match_the_oracle(cuda, room, n, extent, npoints):
    xyz, rgb, labels = scenes.scannet_room(room, n, extent)
    got, _ = check_blocks(cuda, xyz, rgb, labels, LABELWEIGHTS, npoints, seed=room + 11)
    if extent < 1.5:
        assert got.block_id.tolist() == [0]
    check_blocks(cuda, xyz, rgb, npoints=npoints, seed=5)          # no labels: weights = core
    check_chunks(cuda, xyz, rgb, npoints)


def _boundary_scene():
    """Points on fp32 values at and next to cmin + i*1.5 +- 0.2 and +- 0.001 along x and y."""
    c0 = np.float32(0.3)
    vals = [c0, np.float32(c0 + 4.5)]
    for i in range(4):
        for m in (0.2, 0.001):
            for sgn in (-1, 1):
                v = np.float32(np.float64(c0) + i * 1.5 + sgn * m)
                vals += [np.nextafter(v, np.float32(-np.inf)), v, np.nextafter(v, np.float32(np.inf))]
    vals = np.array([v for v in vals if c0 <= v <= c0 + np.float32(4.5)], dtype=np.float32)
    gx, gy = np.meshgrid(vals, vals, indexing="ij")
    xyz = np.stack([gx.ravel(), gy.ravel(), np.zeros(gx.size, np.float32)], 1).astype(np.float32)
    return xyz


def test_boundary_points_and_an_extent_that_is_a_multiple_of_the_block(cuda):
    xyz = _boundary_scene()
    assert np.float32(xyz[:, 0].max() - xyz[:, 0].min()) == np.float32(4.5)  # exactly 3 blocks
    assert ref.grid(xyz)[2:] == (3, 3)
    feats = np.arange(xyz.shape[0], dtype=np.float32)[:, None]
    labels = np.arange(xyz.shape[0]) % C
    for npoints in (64, 4096):
        check_blocks(cuda, xyz, feats, labels, LABELWEIGHTS, npoints, seed=npoints)
        check_chunks(cuda, xyz, feats, npoints)


def test_core_threshold_below_at_and_above(cuda):
    # block 1 along x: 99 points in its padding only (x = 1.4), one core point (x = 2.0), one more padding point (3.15)
    rng = np.random.default_rng(0)
    xs = np.concatenate([[0.0], np.full(99, 1.4), [2.0, 3.15]]).astype(np.float32)
    xyz = np.stack([xs, rng.uniform(0, 0.5, xs.size), np.zeros(xs.size)], 1).astype(np.float32)
    feats = np.zeros((xs.size, 1), np.float32)
    npoints = 100  # threshold 0.01 * 100 = exactly one core draw
    seg = [idx for b, idx, _ in ref.segments(xyz) if b == 1][0]
    found = {}
    for seed in range(400):
        pos = ref.sample_positions(seed, 1, npoints, len(seg)).astype(np.int64)
        found.setdefault(int(np.sum(seg[pos] == 100)), seed)
    assert {0, 1, 2} <= set(found)
    for core, seed in found.items():
        got, _ = check_blocks(cuda, xyz, feats, npoints=npoints, seed=seed)
        assert (1 in got.block_id.tolist()) == (core >= 1), core


def test_empty_blocks_are_skipped(cuda):
    rng = np.random.default_rng(2)
    a = rng.uniform(0, 1, (3000, 3))
    b = rng.uniform(0, 1, (3000, 3)) + np.array([6.0, 4.0, 0.0])
    xyz = np.concatenate([a, b]).astype(np.float32)
    rgb = rng.uniform(-0.5, 0.5, xyz.shape).astype(np.float32)
    labels = rng.integers(0, C, xyz.shape[0])
    got, _ = check_blocks(cuda, xyz, rgb, labels, LABELWEIGHTS, 2048, seed=3)
    # 5 x 4 blocks, 15 of them empty; blocks 14 and 15 hold padding points of the far cluster only
    assert got.block_id.tolist() == [0, 18, 19]
    _, sizes = check_chunks(cuda, xyz, rgb, 2048)
    assert sizes.shape[0] == 8  # 2 for the 3000 points of block 0, 6 for blocks 14, 15, 18, 19


def test_errors(cuda):
    xyz = np.zeros((10, 3), np.float32)
    xyz[:, 1] = np.linspace(0, 3, 10)
    feats = np.zeros((10, 3), np.float32)
    with pytest.raises(ValueError):
        whole_scene.scene_blocks(_t(xyz, cuda), _t(feats, cuda))      # zero extent in x
    with pytest.raises(ValueError):
        whole_scene.scene_chunks(_t(xyz[:, [1, 0, 2]], cuda), _t(feats, cuda))  # zero extent in y
    far = np.array([[0, 0, 0], [400, 400, 0]], np.float32)               # 267 x 267 blocks
    with pytest.raises(Pn2Error, match="at most 65536"):
        whole_scene.scene_blocks(_t(far, cuda), _t(feats[:2], cuda))
    with pytest.raises(Pn2Error, match="at most 65536"):
        whole_scene.scene_chunks(_t(far, cuda), _t(feats[:2], cuda))
    with pytest.raises(Pn2Error, match="n >= 1"):
        whole_scene.scene_blocks(torch.zeros((0, 3), device=cuda), torch.zeros((0, 3), device=cuda))
    ok = np.stack([np.linspace(0, 3, 10), np.linspace(0, 3, 10), np.zeros(10)], 1).astype(np.float32)
    with pytest.raises(Pn2Error, match="npoints"):
        whole_scene.scene_blocks(_t(ok, cuda), _t(feats, cuda), npoints=0)
    with pytest.raises(Pn2Error, match="npoints"):
        whole_scene.scene_chunks(_t(ok, cuda), _t(feats, cuda), npoints=0)


@pytest.fixture(scope="module")
def net(cuda):
    torch.manual_seed(0)
    return PointNet2SemSeg(C).eval().to(cuda)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_segment_scene_equals_the_oracle_vote(cuda, net, precision):
    xyz, rgb, _ = scenes.scannet_room(7, 60000, 4.5)
    prev = set_mlp_precision(precision)
    try:
        labels, votes = whole_scene.segment_scene(net, _t(xyz, cuda), _t(rgb, cuda), batch=4)
        labels2, votes2 = whole_scene.segment_scene(net, _t(xyz, cuda), _t(rgb, cuda), batch=4)
        pts, index, sizes = whole_scene.scene_chunks(_t(xyz, cuda), _t(rgb, cuda))
        with torch.no_grad():
            pred = torch.cat([net.predict(x.permute(0, 2, 1)[:, :3], x.permute(0, 2, 1)[:, 3:]) for x in pts.split(4)])
    finally:
        set_mlp_precision(prev)
    assert torch.equal(labels, labels2) and torch.equal(votes, votes2)
    want = ref.scene_votes(index.cpu().numpy(), sizes.cpu().numpy(), pred.cpu().numpy(), xyz.shape[0], C)
    np.testing.assert_array_equal(votes.cpu().numpy(), want)
    np.testing.assert_array_equal(labels.cpu().numpy(), np.argmax(want, axis=1))
    np.testing.assert_array_equal(want.sum(1), ref.padded_block_count(xyz))
    assert labels.dtype == torch.uint8 and labels.shape == (xyz.shape[0],)


def test_evaluation_counters_match_the_host_loop(cuda, net):
    xyz, rgb, labels = scenes.scannet_room(8, 120000, 6.0)
    blocks = whole_scene.scene_blocks(_t(xyz, cuda), _t(rgb, cuda), _t(labels, cuda), _t(LABELWEIGHTS, cuda), seed=1)
    ctr = pc_util.EvalCounters(C, cuda, res=0.02)
    preds = []
    with torch.no_grad():
        for s in range(0, blocks.points.shape[0], 8):
            pts = blocks.points[s:s + 8]
            x = pts.permute(0, 2, 1)
            pred = net.predict(x[:, :3], x[:, 3:])
            ctr.update(pts, blocks.target[s:s + 8], pred, blocks.weights[s:s + 8])
            preds.append(pred.cpu().numpy())
    res = ctr.result()
    pts, target, weights = blocks.points.cpu().numpy(), blocks.target.cpu().numpy(), blocks.weights.cpu().numpy()
    pred = np.concatenate(preds).astype(np.int64)
    want = pc_util_ref.voxel_accuracy_counts(pts, target, pred, weights, C, res=0.02)
    for k, v in want.items():
        np.testing.assert_array_equal(np.asarray(res[k]), np.asarray(v), err_msg=k)
    w = weights > 0
    assert res["total_seen"] == int(np.sum((target > 0) & w))
    assert res["total_correct"] == int(np.sum((pred == target) & (target > 0) & w))
    for l in range(C):
        assert res["total_seen_class"][l] == int(np.sum((target == l) & w))
        assert res["total_correct_class"][l] == int(np.sum((pred == l) & (target == l) & w))
        assert res["total_union_class"][l] == int(np.sum(((pred == l) | (target == l)) & w))
