"""Training crops on the device (csrc/scene_blocks.cu, pn2_b200/whole_scene.py SceneBank) bit-exact against the numpy
restatement of the training loader's loop (oracle/scene_crops_ref.py): all seven outputs on rooms and multi-scene banks,
late tries and the no-valid case, points on the fp64 boundaries of a column, out-of-range scene ids, the step counter,
CUDA-graph capture and replay, the class weights and the bank's validation."""
import numpy as np
import pytest
import torch

from oracle import scene_crops_ref as ref
from pn2_b200 import Pn2Error, scenes, whole_scene

pytestmark = pytest.mark.gpu

C = 21
LABELWEIGHTS = (1.0 + np.arange(C) / 7.0).astype(np.float32) ** 1.5


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _pack(rooms):
    xyz = np.concatenate([r[0] for r in rooms])
    feats = np.concatenate([r[1] for r in rooms])
    labels = np.concatenate([r[2] for r in rooms]).astype(np.int64)
    offsets = np.concatenate([[0], np.cumsum([len(r[0]) for r in rooms])]).astype(np.int64)
    return xyz, feats, labels, offsets


def _bank(dev, packed):
    xyz, feats, labels, offsets = packed
    return whole_scene.SceneBank(_t(xyz, dev), _t(feats, dev), _t(labels, dev), _t(offsets, dev))


def check(bank, packed, ids, labelweights=None, npoints=8192, seed=0, step=None):
    """One bank.crops call (at `step` when given, else at the bank's current step) against the oracle."""
    dev = bank.xyz.device
    if step is not None:
        bank.step.fill_(step)
    step = int(bank.step.item())
    got = bank.crops(_t(np.asarray(ids, np.int32), dev), None if labelweights is None else _t(labelweights, dev), npoints, seed)
    assert int(bank.step.item()) == step + 1
    check_equal(got, ref.scene_crops(*packed, ids, labelweights, npoints, seed, step))
    return got


def check_equal(got, want):
    for k in ("point_index", "points", "target", "weights", "center", "tries", "valid"):
        np.testing.assert_array_equal(getattr(got, k).cpu().numpy(), want[k], err_msg=k)


@pytest.fixture(scope="module")
def rooms_bank(cuda):
    packed = _pack([scenes.scannet_room(20, 3000, 1.2), scenes.scannet_room(21, 100000, 5.0),
                    scenes.scannet_room(22, 250000, 9.5), scenes.scannet_room(23, 400000, 12.0)])
    return _bank(cuda, packed), packed


@pytest.mark.parametrize("npoints", [1024, 8192])
@pytest.mark.parametrize("seed,step", [(0, 0), (7, 5), (2 ** 64 - 1, 1 << 33)])
def test_rooms_match_the_oracle(cuda, rooms_bank, npoints, seed, step):
    bank, packed = rooms_bank
    ids = [3, 1, 0, 2, 1, 1, 3, 0]  # repeated ids draw different columns
    check(bank, packed, ids, LABELWEIGHTS, npoints, seed, step)
    check(bank, packed, ids[:3], None, npoints, seed, step + 1)  # weights = core mask


def test_bounds(cuda, rooms_bank):
    bank, (xyz, _, _, offsets) = rooms_bank
    want = np.stack([np.concatenate([xyz[a:b].min(0), xyz[a:b].max(0)]) for a, b in zip(offsets[:-1], offsets[1:])])
    np.testing.assert_array_equal(bank.bounds.cpu().numpy(), want)
    assert bank.num_scenes == 4 and bank.max_count == 400000


def _late_tries_scene(n, seed):
    rng = np.random.default_rng(seed)
    p = rng.uniform([0, 0, 0], [6, 6, 2.5], (n, 3)).astype(np.float32)
    labels = np.where(p[:, 0] < 2.2, 1 + np.arange(n) % 5, 0).astype(np.int64)
    return p, rng.uniform(-0.5, 0.5, (n, 3)).astype(np.float32), labels


def test_late_tries_and_no_valid_try(cuda):
    packed = _pack([_late_tries_scene(20000, 0), _late_tries_scene(30000, 1)])
    bank = _bank(cuda, packed)
    ids = [0, 1] * 48
    want = ref.scene_crops(*packed, ids, LABELWEIGHTS, 256, 1, 0)
    assert set(range(1, 11)) == set(want["tries"].tolist())
    assert (want["valid"] == 0).any() and ((want["tries"] == 10) & (want["valid"] == 1)).any()
    check(bank, packed, ids, LABELWEIGHTS, 256, seed=1, step=0)


def test_points_on_the_column_boundaries(cuda):
    """The centre of try 0 of crop 0 sits at a chosen point; other points lie on, and one fp32 step either side of,
    the fp64 bounds curmin - 0.2, curmax + 0.2, curmin - 0.01 and curmax + 0.01 in x and y, plus a dense core filler
    so that the try passes."""
    rng = np.random.default_rng(3)
    cx, cy = np.float32(1.2345), np.float32(-0.6789)
    edges = [np.float64(v) for v in (-0.75 - 0.2, 0.75 + 0.2, -0.75 - 0.01, 0.75 + 0.01)]
    xs, ys = [cx], [cy]
    for c, out in ((cx, xs), (cy, ys)):
        for e in edges:
            v = np.float32(np.float64(c) + e)
            out += [np.nextafter(v, np.float32(-np.inf)), v, np.nextafter(v, np.float32(np.inf))]
    gx, gy = np.meshgrid(np.array(xs, np.float32), np.array(ys, np.float32), indexing="ij")
    ring = np.stack([gx.ravel(), gy.ravel(), rng.uniform(0, 2.5, gx.size)], 1)
    filler = np.stack([rng.uniform(cx - 0.7, cx + 0.7, 4000), rng.uniform(cy - 0.7, cy + 0.7, 4000), rng.uniform(0, 2.5, 4000)], 1)
    far = np.array([[cx + 5, cy + 5, 0.0], [cx - 5, cy - 5, 2.5]])
    body = np.concatenate([ring[1:], filler, far]).astype(np.float32)  # ring[0] is the centre itself
    n = len(body) + 1
    for seed in range(100):
        c = ref.centre(ref.draw_hash(seed, 0), 0, 0, n)
        xyz = np.insert(body, c, [cx, cy, 1.0], axis=0).astype(np.float32)
        packed = (xyz, rng.uniform(-0.5, 0.5, (n, 3)).astype(np.float32), np.ones(n, np.int64), np.array([0, n]))
        want = ref.scene_crops(*packed, [0], LABELWEIGHTS, 4096, seed, 0)
        if want["tries"][0] == 1:
            break
    assert want["center"][0] == c and want["valid"][0] == 1
    padded = ref.column(xyz, packed[2], xyz.min(0), xyz.max(0), c)[0]
    ring_in = padded[np.isin(xyz[:, 0], xs) & np.isin(xyz[:, 1], ys)]
    assert 0 < ring_in.sum() < len(ring)  # the ring straddles the padded bound
    bank = _bank(cuda, packed)
    check(bank, packed, [0, 0, 0], LABELWEIGHTS, 4096, seed, 0)


def test_out_of_range_scene_ids(cuda, rooms_bank):
    bank, packed = rooms_bank
    got = check(bank, packed, [1, -1, 4, 0, 2 ** 31 - 1, 3], LABELWEIGHTS, 1024, seed=4, step=9)
    assert got.tries[[1, 2, 4]].tolist() == [0, 0, 0] and got.center[[1, 2, 4]].tolist() == [-1, -1, -1]
    assert (got.point_index[[1, 2, 4]] == -1).all() and not got.points[[1, 2, 4]].any()
    assert not got.target[[1, 2, 4]].any() and not got.weights[[1, 2, 4]].any()


def test_step_counter(cuda, rooms_bank):
    bank, packed = rooms_bank
    ids = _t(np.array([1, 0, 1], np.int32), cuda)
    lw = _t(LABELWEIGHTS, cuda)
    bank.step.zero_()
    first = [bank.crops(ids, lw, 1024, 5) for _ in range(3)]
    assert int(bank.step.item()) == 3
    for k, got in enumerate(first):
        check_equal(got, ref.scene_crops(*packed, [1, 0, 1], LABELWEIGHTS, 1024, 5, k))
    bank.step.zero_()
    for got in first:
        again = bank.crops(ids, lw, 1024, 5)
        for a, b in zip(got, again):
            assert torch.equal(a, b)


def test_graph_capture_and_replay(cuda, rooms_bank):
    """Capture fails on any host synchronisation, so a successful capture shows there is none."""
    bank, packed = rooms_bank
    ids = _t(np.array([2, 3, 1, 3], np.int32), cuda)
    lw = _t(LABELWEIGHTS, cuda)
    side = torch.cuda.Stream(cuda)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        bank.crops(ids, lw, 2048, 9)  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = bank.crops(ids, lw, 2048, 9)
    k = 17
    bank.step.fill_(k)
    for i in range(3):
        graph.replay()
        torch.cuda.synchronize()
        check_equal(static, ref.scene_crops(*packed, [2, 3, 1, 3], LABELWEIGHTS, 2048, 9, k + i))
    assert int(bank.step.item()) == k + 3


def test_label_weights_are_the_loaders(cuda, rooms_bank):
    bank, (_, _, labels, _) = rooms_bank
    w = bank.label_weights(C)
    assert w.dtype == torch.float32 and w.device == cuda
    np.testing.assert_array_equal(w.cpu().numpy(), ref.label_weights(labels, C))  # exact: the formula runs in numpy
    np.testing.assert_array_equal(bank.label_weights(5).cpu().numpy(), ref.label_weights(labels, 5))  # labels >= 5 clamp/drop


def test_bank_validation_and_errors(cuda, rooms_bank):
    xyz, feats, labels = torch.zeros(10, 3, device=cuda), torch.zeros(10, 2, device=cuda), torch.zeros(10, dtype=torch.int64, device=cuda)
    for off in ([0, 10, 10], [1, 10], [0, 9], [0, 6, 4, 10], [0]):
        with pytest.raises(Pn2Error, match="offsets"):
            whole_scene.SceneBank(xyz, feats, labels, torch.tensor(off, device=cuda))
    with pytest.raises(Pn2Error, match="labels"):
        whole_scene.SceneBank(xyz, feats, labels.int(), torch.tensor([0, 10], device=cuda))
    with pytest.raises(Pn2Error, match="offsets"):
        whole_scene.SceneBank(xyz, feats, labels, torch.tensor([0, 10], device=cuda, dtype=torch.int32))
    bank, _ = rooms_bank
    ids = torch.zeros(4, dtype=torch.int32, device=cuda)
    with pytest.raises(Pn2Error, match="bad dims"):
        bank.crops(ids, npoints=0)
    with pytest.raises(Pn2Error, match="bad dims"):
        bank.crops(ids[:0])
    with pytest.raises(Pn2Error, match="2\\^31"):
        bank.crops(torch.zeros(1 << 16, dtype=torch.int32, device=cuda), npoints=1 << 15)
    with pytest.raises(Pn2Error, match="int32"):
        bank.crops(ids.long())
    with pytest.raises(Pn2Error):
        bank.crops(ids.cpu())
