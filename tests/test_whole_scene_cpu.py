"""Whole-scene protocol without a GPU: the oracle (oracle/whole_scene_ref.py) on hand-built scenes with known blocks, the
sampling hash against fixed values, argument validation of the scene entry points and CPU tensors refused."""
import numpy as np
import pytest
import torch

from oracle import whole_scene_ref as ref
from pn2_b200 import Pn2Error, scenes, whole_scene

M64 = (1 << 64) - 1


def _mix_int(x):
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & M64
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & M64
    return x ^ (x >> 31)


def test_hash_matches_fixed_values():
    # splitmix64 finaliser values, independent of the oracle's numpy arithmetic
    assert _mix_int(0) == 0
    assert _mix_int(1) == 0x5692161D100B05E5
    for seed, b, s in [(0, 0, 1), (0, 3, 17), (7, 65535, 8191), (M64, 12, 4095), (123456789, 1, 0)]:
        h = _mix_int((seed * 0x9E3779B97F4A7C15 + ((b << 32) | s)) & M64)
        assert int(ref.slot_hash(seed, b, [s])[0]) == h
        for count in (1, 3, 8192, 400000):
            assert int(ref.sample_positions(seed, b, s + 1, count)[s]) == ((h >> 32) * count) >> 32
    assert [int(v) for v in ref.slot_hash(0, 0, [0, 1, 2])] == [0, 6238072747940578789, 15839785061582574730]
    assert int(ref.slot_hash(M64, 65535, [8191])[0]) == 612360328681266987


def _line(xs, ys=None):
    xs = np.asarray(xs, dtype=np.float32)
    ys = np.linspace(0, 0.5, len(xs)).astype(np.float32) if ys is None else np.asarray(ys, dtype=np.float32)  # one block in y
    return np.stack([xs, ys, np.zeros_like(xs)], 1)


def test_segments_of_a_hand_built_scene():
    # x extent 3.15 -> 3 blocks along x, 1 along y; padded x ranges [-0.2, 1.7], [1.3, 3.2], [2.8, 4.7]
    xyz = _line([0.0, 1.45, 3.15, 2.0, 1.35])
    segs = ref.segments(xyz)
    assert [b for b, _, _ in segs] == [0, 1, 2]
    assert [list(idx) for _, idx, _ in segs] == [[0, 1, 4], [1, 2, 3, 4], [2]]
    # cores [-0.001, 1.501], [1.499, 3.001], [2.999, 4.501]
    assert [list(core) for _, _, core in segs] == [[True, True, True], [False, False, True, False], [True]]
    np.testing.assert_array_equal(ref.padded_block_count(xyz), [1, 2, 2, 1, 2])


def test_a_block_without_core_samples_is_dropped():
    xyz = _line([0.0, 1.45, 3.15])  # block 1 holds 1.45 and 3.15, both in its padding only
    out = ref.scene_blocks(xyz, np.zeros((3, 0), np.float32), npoints=16)
    np.testing.assert_array_equal(out["block_id"], [0, 2])
    assert out["target"] is None
    np.testing.assert_array_equal(out["weights"][1], np.ones(16, np.float32))
    assert set(out["point_index"][1]) == {2}


def test_corner_point_lies_in_four_blocks_and_block_ids_run_i_outer():
    xyz = np.array([[0, 0, 0], [3, 3, 1], [1.5, 1.5, 0.5], [0.1, 2.9, 0]], dtype=np.float32)
    segs = ref.segments(xyz)
    assert [b for b, _, _ in segs] == [0, 1, 2, 3]
    assert ref.padded_block_count(xyz)[2] == 4
    assert list(segs[1][1]) == [2, 3]   # block (0, 1): x in [-0.2, 1.7], y in [1.3, 3.2]
    assert list(segs[2][1]) == [2]      # block (1, 0)


def test_chunks_cover_every_point_of_a_block_once():
    rng = np.random.default_rng(0)
    xyz = rng.uniform(0, 1.4, (1000, 3)).astype(np.float32)  # one block of 1000 points
    index, sizes, pts = ref.scene_chunks(xyz, xyz[:, :1], npoints=300)
    assert index.shape == (4, 300) and list(sizes) == [250, 250, 250, 250]
    valid = np.concatenate([index[c, :sizes[c]] for c in range(4)])
    np.testing.assert_array_equal(np.sort(valid), np.arange(1000))
    np.testing.assert_array_equal(index[1, :3], [1, 5, 9])
    np.testing.assert_array_equal(index[1, 250:253], index[1, :3])  # repeats pad the chunk
    np.testing.assert_array_equal(pts[..., :3], xyz[index])
    votes = ref.scene_votes(index, sizes, np.zeros_like(index, dtype=np.uint8), 1000, 3)
    np.testing.assert_array_equal(votes[:, 0], np.ones(1000))


def test_zero_extent_raises():
    with pytest.raises(ValueError):
        ref.segments(_line([1.0, 1.0], [0.0, 2.0]))
    with pytest.raises(ValueError):
        ref.segments(_line([0.0, 2.0], [1.0, 1.0]))


def test_room_generator_is_seeded():
    a = scenes.scannet_room(3, 5000, 6.0)
    b = scenes.scannet_room(3, 5000, 6.0)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    xyz, rgb, labels = a
    assert xyz.shape == (5000, 3) and rgb.shape == (5000, 3) and labels.shape == (5000,)
    assert xyz.dtype == np.float32 and rgb.dtype == np.float32
    assert (labels == 0).any() and labels.max() <= 20 and np.abs(rgb).max() <= 0.5
    assert 5.9 < np.ptp(xyz[:, 0]) < 6.1


def test_argument_validation_without_gpu():
    from pn2_b200 import _lib
    lib = _lib.load()
    err = lib.pn2_last_error
    assert lib.pn2_scene_index(0, None, None, None, None, None) == 1 and b"n >= 1" in err()
    assert lib.pn2_scene_index(1 << 29, None, None, None, None, None) == 1 and b"2^31" in err()
    assert lib.pn2_scene_index(8, None, None, None, None, None) == 1 and b"null pointer" in err()
    assert lib.pn2_scene_keep(0, 0, None, None, None, None, None, None) == 1 and b"npoints" in err()
    assert lib.pn2_scene_chunks(0, None, None, None, None) == 1 and b"npoints" in err()
    args = [0, 8192, 0, 3] + [None] * 4 + [0] + [None] * 9
    assert lib.pn2_scene_sample(300, 300, *args) == 1 and b"at most 65536" in err()
    assert lib.pn2_scene_sample(0, 4, *args) == 1 and b"empty grid" in err()
    assert lib.pn2_scene_sample(4, 4, 0, 0, 0, 3, *[None] * 4, 0, *[None] * 9) == 1 and b"bad dims" in err()
    assert lib.pn2_scene_sample(4, 4, 0, 8192, 0, 3, *[None] * 4, 0, *[None] * 9) == 0  # no kept block: nothing to do
    assert lib.pn2_scene_chunk_rows(256, 257, 4, 8192, 3, *[None] * 10) == 1 and b"at most 65536" in err()
    assert lib.pn2_scene_votes(1, 8192, None, None, None, 10, 300, None, None, None) == 1 and b"num_classes" in err()
    assert lib.pn2_scene_votes(1, 8192, None, None, None, 10, 21, None, None, None) == 1 and b"null pointer" in err()


def test_cpu_tensors_are_refused():
    xyz, feats = torch.zeros(16, 3), torch.zeros(16, 3)
    with pytest.raises(Pn2Error):
        whole_scene.scene_blocks(xyz, feats)
    with pytest.raises(Pn2Error):
        whole_scene.scene_chunks(xyz, feats)
    idx = torch.zeros(1, 8, dtype=torch.int32)
    with pytest.raises(Pn2Error):
        whole_scene.scene_votes(idx, torch.ones(1, dtype=torch.int32), torch.zeros(1, 8, dtype=torch.uint8), 16, 21)
    from pn2_b200.models import PointNet2SemSeg
    with pytest.raises(Pn2Error):
        whole_scene.segment_scene(PointNet2SemSeg(21).eval(), xyz, feats)
    with pytest.raises(ValueError):
        whole_scene.segment_scene(PointNet2SemSeg(21), xyz, feats)  # needs eval()
