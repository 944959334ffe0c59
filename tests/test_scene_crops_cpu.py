"""Training crops without a GPU: the oracle (oracle/scene_crops_ref.py) against the training loader's loop as written,
the draw hash against fixed values, hand-built columns at the loader's thresholds and voxel-key corner cases, argument
validation of the crop entry points and CPU tensors refused."""
import numpy as np
import pytest
import torch

from oracle import scene_crops_ref as ref
from pn2_b200 import Pn2Error, scenes, whole_scene

M64 = (1 << 64) - 1
C = 21
LABELWEIGHTS = (1.0 + np.arange(C) / 7.0).astype(np.float32) ** 1.5


def _mix_int(x):
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & M64
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & M64
    return x ^ (x >> 31)


def _literal_loop(point_set, semantic_seg, labelweights, npoints, choice):
    """ScannetDataset.__getitem__ of the training loader, with np.random.choice injected as `choice`."""
    coordmax = np.max(point_set, axis=0)
    coordmin = np.min(point_set, axis=0)
    isvalid = False
    for i in range(10):
        curcenter = point_set[choice(len(semantic_seg), 1)[0], :]
        curmin = curcenter - [0.75, 0.75, 1.5]
        curmax = curcenter + [0.75, 0.75, 1.5]
        curmin[2] = coordmin[2]
        curmax[2] = coordmax[2]
        curchoice = np.sum((point_set >= (curmin - 0.2)) * (point_set <= (curmax + 0.2)), axis=1) == 3
        cur_point_set = point_set[curchoice, :]
        cur_semantic_seg = semantic_seg[curchoice]
        if len(cur_semantic_seg) == 0:
            continue
        mask = np.sum((cur_point_set >= (curmin - 0.01)) * (cur_point_set <= (curmax + 0.01)), axis=1) == 3
        vidx = np.ceil((cur_point_set[mask, :] - curmin) / (curmax - curmin) * [31.0, 31.0, 62.0])
        vidx = np.unique(vidx[:, 0] * 31.0 * 62.0 + vidx[:, 1] * 62.0 + vidx[:, 2])
        isvalid = np.sum(cur_semantic_seg > 0) / len(cur_semantic_seg) >= 0.7 and len(vidx) / 31.0 / 31.0 / 62.0 >= 0.02
        if isvalid:
            break
    choice = choice(len(cur_semantic_seg), npoints, replace=True)
    point_set = cur_point_set[choice, :]
    semantic_seg = cur_semantic_seg[choice]
    mask = mask[choice]
    sample_weight = labelweights[semantic_seg]
    sample_weight *= mask
    return point_set, semantic_seg, sample_weight, i + 1, isvalid


def _hash_choice(h, b):
    """np.random.choice replaced by the crop hash of crop b: the k-th single draw is the centre of try k."""
    tries = [0]

    def choice(n, size, replace=False):
        if size == 1:
            tries[0] += 1
            return [ref.centre(h, b, tries[0] - 1, n)]
        return ref.sample_positions(h, b, size, n).astype(np.int64)
    return choice


@pytest.mark.parametrize("room,n,extent,seed,step", [(0, 20000, 3.0, 0, 0), (1, 60000, 5.0, 7, 3), (2, 30000, 4.0, 1, 11)])
def test_oracle_equals_the_literal_loop(room, n, extent, seed, step):
    xyz, rgb, labels = scenes.scannet_room(room, n, extent)
    ids = [0, 0, 0, 0]
    out = ref.scene_crops(xyz, rgb, labels, np.array([0, n]), ids, LABELWEIGHTS, npoints=512, seed=seed, step=step)
    h = ref.draw_hash(seed, step)
    for b in range(len(ids)):
        pts, seg, w, tries, valid = _literal_loop(xyz, labels, LABELWEIGHTS, 512, _hash_choice(h, b))
        np.testing.assert_array_equal(out["points"][b, :, :3], pts)
        np.testing.assert_array_equal(out["target"][b], seg)
        np.testing.assert_array_equal(out["weights"][b], w)
        assert out["tries"][b] == tries and out["valid"][b] == valid


def test_oracle_equals_the_literal_loop_through_late_tries():
    xyz, labels = _late_tries_scene()
    ids = [0] * 24
    out = ref.scene_crops(xyz, xyz, labels, np.array([0, len(xyz)]), ids, None, npoints=64, seed=1)
    h = ref.draw_hash(1, 0)
    assert len(set(out["tries"].tolist())) >= 5 and not out["valid"].all()
    for b in range(len(ids)):
        pts, seg, w, tries, valid = _literal_loop(xyz, labels, np.ones(C, np.float32), 64, _hash_choice(h, b))
        np.testing.assert_array_equal(out["points"][b, :, :3], pts)
        np.testing.assert_array_equal(out["weights"][b], w)
        assert out["tries"][b] == tries and out["valid"][b] == valid


def _late_tries_scene(n=20000, seed=0):
    """A 6 x 6 x 2.5 m box of points labelled only where x < 2.2: a column passes the 70 % test only near that side."""
    rng = np.random.default_rng(seed)
    p = rng.uniform([0, 0, 0], [6, 6, 2.5], (n, 3)).astype(np.float32)
    return p, np.where(p[:, 0] < 2.2, 1 + np.arange(n) % 5, 0).astype(np.int64)


def test_hash_matches_fixed_values():
    assert ref.draw_hash(0, 0) == 0
    for seed, step in [(0, 1), (5, 0), (M64, 3), (123456789, 1 << 40)]:
        assert ref.draw_hash(seed, step) == _mix_int((seed * 0x9E3779B97F4A7C15 + step) & M64)
    h = ref.draw_hash(7, 2)
    for b, t, n in [(0, 0, 1), (3, 9, 400000), (31, 4, 12345)]:
        g = _mix_int((h * 0x9E3779B97F4A7C15 + ((b << 32) | ((1 << 31) + t))) & M64)
        assert ref.centre(h, b, t, n) == ((g >> 32) * n) >> 32
    assert ref.draw_hash(1, 0) == 0xE220A8397B1DCDAF
    assert [ref.centre(0xE220A8397B1DCDAF, 2, t, 100000) for t in range(3)] == [10051, 45562, 73047]


# ---- hand-built columns: centre at (0, 0), so curmin / curmax = -/+ 0.75 in x and y; z range [0, 6.2] ----

def _cell(v, cells, lo, ext):
    return np.float32(lo + (v - 0.5) / cells * ext)


def _voxel_scene(triples, labelled=None):
    """One core point at the centre of each voxel (vx, vy, vz) (vx, vy in 1..31, vz in 1..62), point 0 the column's
    centre (its triple must be (16, 16, vz)), and two points far outside the column that set z to [0, 6.2]."""
    pts = [[_cell(vx, 31, -0.75, 1.5), _cell(vy, 31, -0.75, 1.5), _cell(vz, 62, 0.0, 6.2)] for vx, vy, vz in triples]
    assert pts[0][:2] == [0.0, 0.0]
    pts += [[10.0, 10.0, 0.0], [10.0, 10.0, 6.2]]
    xyz = np.array(pts, np.float32)
    seg = np.ones(len(xyz), np.int64)
    if labelled is not None:
        seg[labelled:len(triples)] = 0
    return xyz, seg


def _triples(k):
    out = [(16, 16, 1)]
    for vz in range(1, 63):
        for vx in range(1, 32):
            for vy in range(1, 32):
                if (vx, vy, vz) != (16, 16, 1):
                    out.append((vx, vy, vz))
                if len(out) == k:
                    return out


def _column(xyz, seg):
    return ref.column(xyz, seg, xyz.min(0), xyz.max(0), 0)


@pytest.mark.parametrize("keys,valid", [(1192, True), (1191, False)])
def test_occupancy_threshold_is_inclusive(keys, valid):
    xyz, seg = _voxel_scene(_triples(keys))
    curchoice, mask, nkeys, isvalid = _column(xyz, seg)
    assert curchoice.sum() == keys and mask.all() and nkeys == keys
    assert isvalid == valid


@pytest.mark.parametrize("labelled,valid", [(1400, True), (1399, False)])
def test_labelled_threshold_is_inclusive(labelled, valid):
    xyz, seg = _voxel_scene(_triples(2000), labelled)
    _, _, nkeys, isvalid = _column(xyz, seg)
    assert nkeys == 2000 and isvalid == valid


def test_colliding_keys_count_once():
    # (vx, vy, vz = 62) and (vx, vy + 1, vz = 0) share the key value vx*1922 + (vy+1)*62: z = 6.2 and z = 0 exactly
    base = _triples(1180)
    xyz, seg = _voxel_scene(base)
    extra = []
    for vx in (3, 9, 20):
        for vy in (4, 5, 6, 7):
            extra.append([_cell(vx, 31, -0.75, 1.5), _cell(vy, 31, -0.75, 1.5), 6.2])        # (vx, vy, 62)
            extra.append([_cell(vx, 31, -0.75, 1.5), _cell(vy + 1, 31, -0.75, 1.5), 0.0])    # (vx, vy + 1, 0)
    xyz = np.concatenate([xyz, np.array(extra, np.float32)])
    seg = np.ones(len(xyz), np.int64)
    triples = set(base) | {(vx, vy, 62) for vx in (3, 9, 20) for vy in (4, 5, 6, 7)} | \
        {(vx, vy + 1, 0) for vx in (3, 9, 20) for vy in (4, 5, 6, 7)}
    keys = {vx * 1922 + vy * 62 + vz for vx, vy, vz in triples}
    assert len(triples) == 1180 + 24 and len(keys) == 1180 + 12
    _, _, nkeys, isvalid = _column(xyz, seg)
    assert nkeys == len(keys) and isvalid  # 1192 distinct values: valid, though 1204 distinct triples


def test_negative_zero_keys_count_once():
    # x = curmin gives vx = 0.0; x in [curmin - 0.01, curmin) gives ceil(-0.004) = -0.0: one key value
    xyz, seg = _voxel_scene(_triples(1191))
    edge = np.array([[-0.75, _cell(4, 31, -0.75, 1.5), _cell(7, 62, 0, 6.2)],
                     [-0.755, _cell(4, 31, -0.75, 1.5), _cell(7, 62, 0, 6.2)]], np.float32)
    xyz = np.concatenate([xyz, edge])
    seg = np.ones(len(xyz), np.int64)
    vx = np.ceil((edge[:, 0].astype(np.float64) + 0.75) / 1.5 * 31.0)
    assert vx[0] == 0.0 and vx[1] == 0.0 and np.signbit(vx[1]) and not np.signbit(vx[0])
    _, mask, nkeys, isvalid = _column(xyz, seg)
    assert mask.sum() == 1193 and nkeys == 1192 and isvalid


def test_zero_z_extent_is_never_valid():
    xyz, seg = _voxel_scene(_triples(3000))
    xyz[:, 2] = 1.25
    _, _, nkeys, isvalid = _column(xyz, seg)
    assert nkeys == 1 and not isvalid  # every key is NaN: np.unique keeps one
    out = ref.scene_crops(xyz, xyz, seg, np.array([0, len(xyz)]), [0], None, npoints=32)
    assert out["tries"][0] == 10 and out["valid"][0] == 0


def test_one_point_scene():
    xyz = np.array([[1.0, 2.0, 3.0]], np.float32)
    out = ref.scene_crops(xyz, xyz * 2, np.array([5]), np.array([0, 1]), [0, 0], LABELWEIGHTS, npoints=16, seed=3)
    assert out["tries"].tolist() == [10, 10] and out["valid"].tolist() == [0, 0] and out["center"].tolist() == [0, 0]
    assert (out["point_index"] == 0).all() and (out["target"] == 5).all()
    np.testing.assert_array_equal(out["weights"], np.full((2, 16), LABELWEIGHTS[5]))
    np.testing.assert_array_equal(out["points"][0, 0], [1, 2, 3, 2, 4, 6])


def test_oracle_out_of_range_scene_ids():
    xyz, rgb, labels = scenes.scannet_room(0, 5000, 3.0)
    out = ref.scene_crops(xyz, rgb, labels, np.array([0, 2000, 5000]), [1, -1, 2, 0], LABELWEIGHTS, npoints=64)
    assert out["tries"][[1, 2]].tolist() == [0, 0] and out["center"][[1, 2]].tolist() == [-1, -1]
    assert (out["point_index"][[1, 2]] == -1).all() and not out["points"][[1, 2]].any()
    assert not out["target"][[1, 2]].any() and not out["weights"][[1, 2]].any()
    assert (out["point_index"][0] >= 2000).all() and (out["point_index"][3] < 2000).all()


def test_label_weights_formula():
    labels = np.array([0, 1, 1, 2, 21, 21, 22, -1])  # 21 = num_classes lands in the last bin; 22 and -1 are dropped
    w = ref.label_weights(labels, 21)
    counts = np.zeros(21, np.float32)
    counts[[0, 1, 2, 20]] = [1, 2, 1, 2]
    want = 1 / np.log(1.2 + counts / np.float32(6))
    assert w.dtype == np.float32
    np.testing.assert_array_equal(w, want.astype(np.float32))


def test_argument_validation_without_gpu():
    from pn2_b200 import _lib
    lib = _lib.load()
    err = lib.pn2_last_error

    def crops(s=1, n=100, c=3, max_count=100, b=4, npoints=64, null=False, lw=False, num_classes=0):
        p = None if null else 16  # never dereferenced: every call below is refused before any launch
        args = [s, n, c, max_count] + [p] * 5 + [b, p, npoints, 0, p, 16 if lw else None, num_classes] + [p] * 7 + [None]
        return lib.pn2_scene_crops(*args)
    assert crops(b=0) == 1 and b"bad dims" in err()
    assert crops(npoints=0) == 1 and b"bad dims" in err()
    assert crops(c=-1) == 1 and b"bad dims" in err()
    assert crops(b=1 << 16, npoints=1 << 15) == 1 and b"2^31" in err()
    assert crops(n=1 << 31, max_count=100) == 1 and b"2^31" in err()
    assert crops(s=0) == 1 and b"s >= 1" in err()
    assert crops(max_count=101) == 1 and b"max_count" in err()
    assert crops(max_count=0) == 1 and b"max_count" in err()
    assert crops(lw=True) == 1 and b"num_classes" in err()
    assert crops(null=True) == 1 and b"null pointer" in err()
    assert lib.pn2_scene_bank_bounds(0, 10, None, None, None, None) == 1 and b"s >= 1" in err()
    assert lib.pn2_scene_bank_bounds(1, 1 << 31, None, None, None, None) == 1 and b"2^31" in err()
    assert lib.pn2_scene_bank_bounds(1, 10, None, None, None, None) == 1 and b"null pointer" in err()


def test_cpu_tensors_are_refused():
    xyz, feats = torch.zeros(16, 3), torch.zeros(16, 3)
    labels, offsets = torch.zeros(16, dtype=torch.int64), torch.tensor([0, 16])
    with pytest.raises(Pn2Error):
        whole_scene.SceneBank(xyz, feats, labels, offsets)
