"""numpy restatement of the training crops of pn2_b200/whole_scene.py SceneBank.crops (TEST INFRASTRUCTURE ONLY: tests/
compare the device against it).

The loop is the PointNet++ ScanNet training loader's (ScannetDataset.__getitem__): up to ten random 1.5 m columns over
the scene's whole z range, the first whose 0.2 m padded column is >= 70 % labelled and whose 0.01 m core occupies >= 2 %
of its 31 x 31 x 62 voxel keys is taken (else the tenth), then `npoints` draws with replacement from the padded column.
np.random.choice is replaced by a seeded counter hash:

    h = mix(seed * 0x9E3779B97F4A7C15 + step)
    centre of try t of crop b   = sample_pos(h, b, 2^31 + t, n)
    slot s of crop b            = sample_pos(h, b, s, padded count), a position in the padded set in ascending scene index
"""
import numpy as np

from .whole_scene_ref import _GOLDEN, mix, sample_positions, slot_hash

TRIES = 10
CENTRE_SLOT = 1 << 31


def draw_hash(seed, step):
    """h = mix(seed * 0x9E3779B97F4A7C15 + step) as a Python int"""
    with np.errstate(over="ignore"):
        return int(mix(np.array([seed], dtype=np.uint64) * _GOLDEN + np.uint64(step))[0])


def centre(h, b, t, n):
    """scene index of the centre of try t of crop b in a scene of n points"""
    return int((slot_hash(h, b, [CENTRE_SLOT + t])[0] >> np.uint64(32)) * np.uint64(n) >> np.uint64(32))


def column(point_set, seg, coordmin, coordmax, c):
    """One try of the loader's loop centred on point c -> (curchoice (n,) bool, mask (padded,) bool core of the padded
    points, number of distinct voxel keys, isvalid)."""
    curcenter = point_set[c]
    curmin = curcenter - [0.75, 0.75, 1.5]
    curmax = curcenter + [0.75, 0.75, 1.5]
    curmin[2] = coordmin[2]
    curmax[2] = coordmax[2]
    curchoice = np.sum((point_set >= (curmin - 0.2)) * (point_set <= (curmax + 0.2)), axis=1) == 3
    cur_point_set = point_set[curchoice, :]
    cur_seg = seg[curchoice]
    if len(cur_seg) == 0:
        return curchoice, np.zeros(0, bool), 0, False
    mask = np.sum((cur_point_set >= (curmin - 0.01)) * (cur_point_set <= (curmax + 0.01)), axis=1) == 3
    with np.errstate(invalid="ignore", divide="ignore"):
        vidx = np.ceil((cur_point_set[mask, :] - curmin) / (curmax - curmin) * [31.0, 31.0, 62.0])
    vidx = np.unique(vidx[:, 0] * 31.0 * 62.0 + vidx[:, 1] * 62.0 + vidx[:, 2])
    isvalid = np.sum(cur_seg > 0) / len(cur_seg) >= 0.7 and len(vidx) / 31.0 / 31.0 / 62.0 >= 0.02
    return curchoice, mask, len(vidx), bool(isvalid)


def crop(point_set, seg, npoints, centre_of, slots_of):
    """The loader's loop on one scene with the draws injected: centre_of(t) -> scene index of the centre of try t,
    slots_of(count) -> (npoints,) positions in the padded set.  -> dict index (npoints,) scene indices, core (npoints,)
    bool, center, tries (1..10), valid."""
    coordmax, coordmin = point_set.max(axis=0), point_set.min(axis=0)
    for t in range(TRIES):
        c = centre_of(t)
        curchoice, mask, _, isvalid = column(point_set, seg, coordmin, coordmax, c)
        if isvalid:
            break
    choice = np.asarray(slots_of(int(curchoice.sum())), dtype=np.int64)
    return {"index": np.nonzero(curchoice)[0][choice], "core": mask[choice], "center": c, "tries": t + 1, "valid": isvalid}


def scene_crops(xyz, feats, labels, offsets, scene_ids, labelweights=None, npoints=8192, seed=0, step=0):
    """SceneBank.crops on a packed bank (numpy arrays) -> dict of the seven outputs."""
    h = draw_hash(seed, step)
    rows = np.concatenate([xyz, feats], axis=1).astype(np.float32)
    out = {k: [] for k in ("point_index", "target", "weights", "center", "tries", "valid")}
    for b, sid in enumerate(np.asarray(scene_ids).tolist()):
        if not 0 <= sid < len(offsets) - 1:
            out["point_index"].append(np.full(npoints, -1, np.int64))
            out["target"].append(np.zeros(npoints, np.int64))
            out["weights"].append(np.zeros(npoints, np.float32))
            out["center"].append(-1)
            out["tries"].append(0)
            out["valid"].append(False)
            continue
        lo, hi = int(offsets[sid]), int(offsets[sid + 1])
        n = hi - lo
        r = crop(xyz[lo:hi], labels[lo:hi], npoints, lambda t: centre(h, b, t, n),
                 lambda count: sample_positions(h, b, npoints, count))
        index = lo + r["index"]
        target = labels[index].astype(np.int64)
        w = r["core"].astype(np.float32)
        if labelweights is not None:
            ok = (target >= 0) & (target < len(labelweights))
            w = np.where(ok, labelweights.astype(np.float32)[np.where(ok, target, 0)] * w, np.float32(0)).astype(np.float32)
        out["point_index"].append(index)
        out["target"].append(target)
        out["weights"].append(w)
        out["center"].append(r["center"])
        out["tries"].append(r["tries"])
        out["valid"].append(r["valid"])
    point_index = np.stack(out["point_index"]).astype(np.int32)
    points = np.where((point_index >= 0)[..., None], rows[np.maximum(point_index, 0)], np.float32(0)).astype(np.float32)
    return {"point_index": point_index, "points": points, "target": np.stack(out["target"]), "weights": np.stack(out["weights"]),
            "center": np.array(out["center"], np.int32), "tries": np.array(out["tries"], np.int32),
            "valid": np.array(out["valid"], np.uint8)}


def label_weights(labels, num_classes=21):
    """The loader's class weights in numpy float32."""
    w, _ = np.histogram(labels, range(num_classes + 1))
    w = w.astype(np.float32)
    w = w / np.sum(w)
    return 1 / np.log(1.2 + w)
