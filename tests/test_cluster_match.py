"""LiDAR clusters -> annotated boxes (msc_cluster_match_batch, GeometryEngine.run_cluster_match, ops.cluster_match,
LiDARAgent.process_batch(match_annotations=True), serialize.ext_evidence(cluster_match=...)).

The definition is the scalar C oracle tests/cluster_match_oracle.c; a devkit-style NumPy points_in_box in f64 checks the oracle's
membership, and the kernels must equal the oracle bit for bit."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from tests import cluster_match_oracle as orc
from tests.test_loader_on_disk import _scenes, devkit_shim  # noqa: F401  (a written nuScenes tree and the fixture that loads it)

SENTINEL = 0x5A5A5A5A
# A row's f32 membership may differ from the f64 devkit chain only this close to a face plane of the box (metres).  Measured on the
# samples of test_oracle_membership_against_numpy_f64 (boxes up to 50 m from the sensor): 11,552 of the 49,700 rows planted on faces,
# edges and corners (and one float either side) differ, the farthest 1.9e-6 m from a face plane; none of the 34,700 other rows differs.
FACE_TOL = 1e-5


# ------------------------------------------------------------------------------------------------ NumPy devkit restatement (f64)
def _quat_R(q):
    w, x, y, z = np.asarray(q, np.float64) / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _corners_in_sensor(box, ego_pose, lidar_calib):
    """devkit Box.translate(-t) / rotate(q.inverse) into ego, then into the sensor, and Box.corners()."""
    c, R = np.asarray(box[:3], np.float64), _quat_R(box[6:10])
    for pose in (ego_pose, lidar_calib):
        P = _quat_R(pose[3:7])
        c, R = P.T @ (c - np.asarray(pose[:3])), P.T @ R
    w, l, h = box[3], box[4], box[5]
    xc = l / 2 * np.array([1, 1, 1, 1, -1, -1, -1, -1])
    yc = w / 2 * np.array([1, -1, -1, 1, 1, -1, -1, 1])
    zc = h / 2 * np.array([1, 1, -1, -1, 1, 1, -1, -1])
    return R @ np.stack([xc, yc, zc]) + c[:, None]


def _points_in_box_f64(corners, pts):
    """devkit points_in_box in f64; also each point's distance to the nearest face plane."""
    p1, i, j, k = corners[:, 0], corners[:, 4] - corners[:, 0], corners[:, 1] - corners[:, 0], corners[:, 3] - corners[:, 0]
    v = pts.astype(np.float64) - p1
    iv, jv, kv = v @ i, v @ j, v @ k
    ii, jj, kk = i @ i, j @ j, k @ k
    inside = (0 <= iv) & (iv <= ii) & (0 <= jv) & (jv <= jj) & (0 <= kv) & (kv <= kk)
    dist = np.min(np.stack([np.minimum(np.abs(iv), np.abs(iv - ii)) / np.sqrt(ii), np.minimum(np.abs(jv), np.abs(jv - jj)) / np.sqrt(jj),
                            np.minimum(np.abs(kv), np.abs(kv - kk)) / np.sqrt(kk)]), 0)
    return inside, dist


def _reduce(member, labels, K):
    """The tables of the oracle's contract recomputed from a membership matrix [n, B] with NumPy."""
    n, B = member.shape
    cnt = np.zeros((B, max(K, 1)), np.int64)
    for k in range(K):
        cnt[:, k] = member[labels == k].sum(0)
    cnt = cnt[:, :K]
    box = np.zeros((B, 5), np.int64)
    box[:, 0] = member.sum(0)
    box[:, 1] = member[labels >= 0].sum(0)
    box[:, 2] = (cnt > 0).sum(1)
    box[:, 3] = np.where(cnt.max(1, initial=0) > 0, cnt.argmax(1) if K else -1, -1)   # argmax: the first (smallest) of equal maxima
    box[:, 4] = cnt.max(1, initial=0)
    cl = np.zeros((K, 3), np.int64)
    if K:
        cl[:, 0] = np.where(cnt.max(0, initial=0) > 0, cnt.argmax(0) if B else -1, -1)
        cl[:, 1] = cnt.max(0, initial=0)
        cl[:, 2] = [(member[labels == k].any(1)).sum() for k in range(K)]
    return cl, box


def _face_rows(corners, rng, n_per_face=40):
    """Rows on the faces, edges and corners of a box (f64 -> f32), each also one float either side along every axis."""
    p1, i, j, k = corners[:, 0], corners[:, 4] - corners[:, 0], corners[:, 1] - corners[:, 0], corners[:, 3] - corners[:, 0]
    uvw = rng.uniform(0, 1, (n_per_face * 6, 3))
    for f in range(6):
        uvw[f * n_per_face:(f + 1) * n_per_face, f // 2] = f % 2
    edges = rng.integers(0, 2, (36, 3)).astype(np.float64)
    for ax in range(3):
        edges[ax * 12:(ax + 1) * 12, ax] = rng.uniform(0, 1, 12)
    uvw = np.concatenate([uvw, np.array(np.meshgrid([0, 1], [0, 1], [0, 1])).reshape(3, -1).T, edges])   # faces, corners, edges
    base = (p1 + uvw[:, :1] * i + uvw[:, 1:2] * j + uvw[:, 2:3] * k).astype(np.float32)
    out = [base]
    for ax in range(3):
        for d in (np.inf, -np.inf):
            b = base.copy()
            b[:, ax] = np.nextafter(b[:, ax], np.float32(d))
            out.append(b)
    return np.concatenate(out)


def _rows4(xyz):
    return np.concatenate([np.asarray(xyz, np.float32), np.ones((len(xyz), 1), np.float32)], 1)


# ------------------------------------------------------------------------------------------------ CPU: the oracle
def test_oracle_membership_against_numpy_f64():
    from msc_geom.layout import boxes_from_annotations
    from msc_geom.synthetic import make_sample
    worst, differ, total = 0.0, 0, 0
    for idx, (sweeps, nb) in enumerate(((1, 5), (1, 60), (1, 120))):
        smp = make_sample(40 + idx, n_sweeps=sweeps, n_boxes=nb)
        boxes = boxes_from_annotations(smp["annotations"])
        corners = [_corners_in_sensor(b, smp["ego_pose"], smp["lidar_calib"]) for b in boxes]
        rng = np.random.default_rng(idx)
        bulk = smp["point_cloud"][::3].astype(np.float32)
        rows = np.concatenate([bulk, *[_rows4(_face_rows(c, rng)) for c in corners[:10]]])
        K = 25
        labels = rng.integers(-1, K, len(rows)).astype(np.int32)
        cl, bx, mem = orc.cluster_match(rows, labels, K, boxes, smp["ego_pose"], smp["lidar_calib"], with_membership=True)
        for b, c in enumerate(corners):
            inside, dist = _points_in_box_f64(c, rows[:, :3])
            bad = inside != mem[:, b].astype(bool)
            assert not bad[:len(bulk)].any()
            differ += int(bad.sum())
            total += int(inside.sum())
            if bad.any():
                worst = max(worst, float(dist[bad].max()))
        rc, rb = _reduce(mem.astype(bool), labels, K)
        assert np.array_equal(cl, rc) and np.array_equal(bx, rb)
        assert bx[:, 0].sum() > 0 and (cl[:, 0] >= 0).any()
    assert worst < FACE_TOL and 0 < differ < total, (worst, differ)


def test_oracle_tie_rules():
    ident = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
    box = lambda cx, cy: [cx, cy, 0.0, 2.0, 2.0, 2.0, 1.0, 0.0, 0.0, 0.0]
    # identical duplicate boxes: every count ties, the smaller index wins
    rows = _rows4(np.random.default_rng(0).uniform(-0.9, 0.9, (30, 3)) + [10, 0, 0])
    labels = np.zeros(30, np.int32)
    cl, bx = orc.cluster_match(rows, labels, 1, np.array([box(0, 0), box(10, 0), box(10, 0)]), ident, ident)
    assert cl.tolist() == [[1, 30, 30]] and bx[1].tolist() == bx[2].tolist() == [30, 30, 1, 0, 30] and bx[0].tolist() == [0, 0, 0, -1, 0]
    # equal counts of one cluster in two boxes; equal counts of two clusters in one box; noise counts for rows only
    a = _rows4(np.full((4, 3), [10.0, 0, 0]))
    b = _rows4(np.full((4, 3), [20.0, 0, 0]))
    noise = _rows4(np.full((3, 3), [20.0, 0.5, 0]))
    rows = np.concatenate([b, a, noise, b])
    labels = np.array([1] * 4 + [1] * 4 + [-1] * 3 + [0] * 4, np.int32)
    cl, bx = orc.cluster_match(rows, labels, 2, np.array([box(20, 0), box(10, 0)]), ident, ident)
    assert cl.tolist() == [[0, 4, 4], [0, 4, 8]]
    assert bx.tolist() == [[11, 8, 2, 0, 4], [4, 4, 1, 1, 4]]
    # NaN rows and no boxes
    rows = _rows4(np.full((2, 3), np.nan))
    cl, bx = orc.cluster_match(rows, np.zeros(2, np.int32), 1, np.array([box(0, 0)]), ident, ident)
    assert cl.tolist() == [[-1, 0, 0]] and bx.tolist() == [[0, 0, 0, -1, 0]]
    cl, bx = orc.cluster_match(rows, np.zeros(2, np.int32), 1, np.zeros((0, 10)), ident, ident)
    assert cl.tolist() == [[-1, 0, 0]] and bx.shape == (0, 5)


# ------------------------------------------------------------------------------------------------ CPU: host assembly
class _Fake:
    """Stands in for run_lidar / run_cluster_match results."""

    def __init__(self, v):
        self.v = v

    def to_host(self):
        return self.v


class _FakeEngine:
    def __init__(self, per, matches):
        from msc_geom.layout import GeomParams
        self.params, self.per, self.matches = GeomParams(), per, matches

    def upload(self, hb):
        return hb

    def run_lidar(self, db, **kw):
        return _Fake(self.per)

    def run_cluster_match(self, lr, db):
        return _Fake(self.matches)


def _table(n_points):
    t = np.zeros((len(n_points), 11), np.float32)
    t[:, 10] = n_points
    t[:, 6], t[:, 7] = 5.0 + np.arange(len(n_points)), 1.0
    return t


def _hand_made():
    obj = np.ones((40, 4), np.float32)
    per = [{"counts": np.array([40, 0, 40]), "ground": np.zeros((0, 4), np.float32), "object": obj, "object_off": 0,
            "labels": np.zeros(40, np.int64), "clusters": _table([12, 3, 20]), "cluster_first": np.array([5, 0, 1]), "noise_first": 2},
           {"counts": np.array([5, 0, 5]), "ground": np.zeros((0, 4), np.float32), "object": obj[:5], "object_off": 40,
            "labels": np.zeros(5, np.int64), "clusters": _table([]), "cluster_first": np.zeros(0, np.int64), "noise_first": -1}]
    matches = [{"cluster_match": np.array([[1, 9, 10], [0, 2, 2], [-1, 0, 0]], np.int32),
                "box_match": np.array([[4, 2, 1, 1, 2], [11, 9, 1, 0, 9], [0, 0, 0, -1, 0]], np.int32)},
               {"cluster_match": np.zeros((0, 3), np.int32), "box_match": np.array([[3, 0, 0, -1, 0]], np.int32)}]
    anns = [[_ann((1, 0, 0), (1, 1, 1)), _ann((2, 0, 0), (1, 1, 1), name="human.pedestrian.adult"),
             _ann((3, 0, 0), (1, 1, 1), name="movable_object.barrier")], [_ann((4, 0, 0), (1, 1, 1), name="vehicle.bus")]]
    return per, matches, anns


def test_process_batch_annotation_match_from_a_hand_made_table():
    from msc_geom.lidar_agent import LiDARAgent, set_order
    per, matches, anns = _hand_made()
    agent = LiDARAgent(object(), "m", "LiDARAgent", engine=_FakeEngine(per, matches))
    order = [l for l in set_order(per[0]["cluster_first"], per[0]["noise_first"]) if per[0]["clusters"][l, 10] >= 5]
    assert sorted(order) == [0, 2]
    samples = [{"point_cloud": np.zeros((0, 4), np.float32), "annotations": a} for a in anns]
    plain = agent.process_batch(samples=samples)
    got = agent.process_batch(samples=samples, match_annotations=True)
    assert all("annotation_match" not in r for r in plain)
    for a, b in zip(plain, got):
        b = dict(b)
        b.pop("annotation_match")
        assert json.dumps(a, default=str, sort_keys=True) == json.dumps(b, default=str, sort_keys=True)
    m = got[0]["annotation_match"]
    want_cl = {0: {"num_points": 12, "annotation": "obj_1", "category": "human.pedestrian.adult", "points_in_annotation": 9},
               2: {"num_points": 20, "annotation": None, "category": None, "points_in_annotation": 0}}
    assert [c["index"] for c in m["clusters"]] == list(range(len(order)))
    assert [{k: c[k] for k in ("num_points", "annotation", "category", "points_in_annotation")} for c in m["clusters"]] == [want_cl[l] for l in order]
    best = {l: i for i, l in enumerate(order)}
    assert m["annotations"] == [{"id": "obj_0", "rows": 4, "clusters": 1, "best_cluster": None},     # label 1 has 3 points: not in the order
                                {"id": "obj_1", "rows": 11, "clusters": 1, "best_cluster": best[0]},
                                {"id": "obj_2", "rows": 0, "clusters": 0, "best_cluster": None}]
    assert got[1]["annotation_match"] == {"clusters": [], "annotations": [{"id": "obj_0", "rows": 3, "clusters": 0, "best_cluster": None}]}
    json.dumps(got[0]["annotation_match"])
    # a device batch without annotation dicts: no categories; with them: the same as from samples
    no_cat = agent.process_batch(device_batch=object(), match_annotations=True)[0]["annotation_match"]
    assert [c["category"] for c in no_cat["clusters"]] == [None, None] and no_cat["annotations"] == m["annotations"]
    assert agent.process_batch(device_batch=object(), match_annotations=True, annotations=anns)[0]["annotation_match"] == m


def test_ext_evidence_with_and_without_cluster_match():
    from msc_geom import serialize as S
    anns = [{"category_name": "vehicle.car"}, {"category_name": "vehicle.bus"}]
    args = (anns, np.array([30, 0], np.uint32), np.array([4.0, np.inf], np.float32), np.zeros((2, 3), np.float32), np.ones((2, 2), np.uint8),
            ["CAM_FRONT", "CAM_BACK"])
    plain = S.ext_evidence(*args)
    assert S.ext_evidence(*args, cluster_match=None) == plain
    got = S.ext_evidence(*args, cluster_match=np.array([[25, 20, 2, 1, 12], [3, 0, 0, -1, 0]], np.int32))
    assert got["objects"][0]["lidar_cluster"] == {"rows": 25, "clusters": 2} and "lidar_cluster" not in got["objects"][1]
    for a, b in zip(plain["objects"], got["objects"]):
        b = dict(b)
        b.pop("lidar_cluster", None)
        assert a == b
    json.dumps(got)


def test_refusals_through_ctypes():
    """Every refusal returns MSC_ERR_BAD_ARGUMENT before anything is launched, so no device is needed; n_samples = 0 is a no-op."""
    from msc_geom import _capi
    lib = _capi.load()
    fake = 1 << 20
    need = int(lib.msc_cluster_match_batch_workspace_bytes(2, 3, 100))
    assert need > 0 and need % 256 == 0
    assert lib.msc_cluster_match_batch_workspace_bytes(-1, 3, 100) == 0 and lib.msc_cluster_match_batch_workspace_bytes(2, -3, 100) == 0
    assert lib.msc_cluster_match_batch_workspace_bytes(2, 3, 0x80000000) == 0

    def structs():
        bi = _capi.MscBatchIn(2, 2, 3, 0, *([fake] * 12))
        rows = _capi.MscLidarBatchOut(100, *([fake] * 11))
        out = _capi.MscClusterMatchOut(fake, fake)
        return bi, rows, out

    def call(bi, rows, out, n=2, ws=fake, nbytes=need):
        return lib.msc_cluster_match_batch(C.byref(bi) if bi is not None else None, C.byref(rows) if rows is not None else None, n,
                                           C.byref(out) if out is not None else None, ws, nbytes, None)
    bad = _capi.MSC_ERR_BAD_ARGUMENT
    bi, rows, out = structs()
    assert call(None, rows, out) == bad and call(bi, None, out) == bad and call(bi, rows, None) == bad
    assert call(bi, rows, out, n=1) == bad and call(bi, rows, out, n=3) == bad and call(bi, rows, out, n=-1) == bad
    assert call(bi, rows, out, nbytes=need - 1) == bad and call(bi, rows, out, ws=None) == bad
    assert call(bi, rows, out, ws=fake + 16) == bad  # not 256-byte aligned
    for field in ("sample_box_off", "boxes", "ego_pose", "lidar_calib"):
        bi, rows, out = structs()
        setattr(bi, field, None)
        assert call(bi, rows, out) == bad, field
    for field in ("counts", "object_off", "n_clusters", "object", "labels"):
        bi, rows, out = structs()
        setattr(rows, field, None)
        assert call(bi, rows, out) == bad, field
    for field in ("cluster", "box"):
        bi, rows, out = structs()
        setattr(out, field, None)
        assert call(bi, rows, out) == bad, field
    bi, rows, out = structs()
    bi.n_boxes = -1
    assert call(bi, rows, out) == bad
    bi, rows, out = structs()
    rows.row_capacity = 0x80000000
    assert call(bi, rows, out) == bad
    empty = _capi.MscBatchIn()
    assert call(empty, _capi.MscLidarBatchOut(), _capi.MscClusterMatchOut(), n=0, ws=None, nbytes=0) == 0


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def eng():
    from msc_geom.engine import GeometryEngine
    return GeometryEngine()


def _agent_params():
    from msc_geom.layout import GeomParams
    return GeomParams(bev_res=800)


def _ann(center, size_wlh, yaw=0.0, name="vehicle.car"):
    return {"category_name": name, "translation": list(map(float, center)), "size": list(map(float, size_wlh)),
            "rotation": [float(np.cos(yaw / 2)), 0.0, 0.0, float(np.sin(yaw / 2))]}


def _blob_sample(rng, centres, per_blob, spread, boxes):
    pts = np.concatenate([rng.normal(c, spread, (per_blob, 3)) for c in centres]) if len(centres) else np.zeros((0, 3))
    return {"point_cloud": _rows4(pts), "annotations": boxes}


def _face_sample(rng):
    """Dense clusters whose rows lie exactly on the faces, edges and corners of an axis-aligned and a rotated box (and one float either
    side), plus duplicate and overlapping boxes."""
    ident = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
    anns = [_ann((10, 5, 0), (2, 4, 2)), _ann((-12, 8, 0.5), (2.5, 5, 1.6), yaw=0.5236), _ann((10, 5, 0), (2, 4, 2)),
            _ann((11, 5, 0), (2, 4, 2), name="vehicle.truck")]
    rows = []
    for a in anns[:2]:
        box = np.array(a["translation"] + a["size"] + a["rotation"])
        c = _corners_in_sensor(box, ident, ident)
        rows.append(_face_rows(c, rng, 60))
        lat = np.stack(np.meshgrid(*[np.linspace(0, 1, 9)] * 3), -1).reshape(-1, 3)   # a lattice through the box: one cluster
        p1, i, j, k = c[:, 0], c[:, 4] - c[:, 0], c[:, 1] - c[:, 0], c[:, 3] - c[:, 0]
        rows.append((p1 + lat[:, :1] * i + lat[:, 1:2] * j + lat[:, 2:3] * k).astype(np.float32))
    return {"point_cloud": _rows4(np.concatenate(rows)), "annotations": anns}


def _many_blobs_sample():
    """About 2,000 separated 10-point blobs (one cluster each) under 150 boxes: more (label, box) counters than one work item."""
    rng = np.random.default_rng(8)
    g = np.arange(-40, 40.01, 1.7)
    c = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)
    c = c[(np.hypot(c[:, 0], c[:, 1]) > 3) & (np.hypot(c[:, 0], c[:, 1]) < 47)]
    pts = np.concatenate([np.column_stack([np.full(10, x), np.full(10, y), np.zeros(10)]) + rng.uniform(-0.08, 0.08, (10, 3)) for x, y in c])
    boxes = [_ann((rng.uniform(-40, 40), rng.uniform(-40, 40), 0.0), (rng.uniform(3, 9), rng.uniform(3, 9), 2.0), rng.uniform(-3, 3))
             for _ in range(150)]
    return {"point_cloud": _rows4(pts), "annotations": boxes}, len(c)


def _mixed_samples(golden_dir):
    from msc_geom.nuscenes_loader import create_loader
    from msc_geom.synthetic import make_sample
    rng = np.random.default_rng(21)
    np.random.seed(0)
    samples = [create_loader(None, use_mock=True).get_sample_by_scene_index(0, 0)]
    synth = np.load(os.path.join(golden_dir, "keyframe_synth.npz"))["points"]
    samples.append({"point_cloud": synth, "annotations": [_ann((rng.uniform(-20, 20), rng.uniform(-20, 20), 0), (3, 6, 3), rng.uniform(-3, 3))
                                                          for _ in range(40)]})
    samples.append({"point_cloud": np.load(os.path.join(golden_dir, "keyframe_mock.npz"))["points"], "annotations": []})
    samples += [make_sample(60, n_sweeps=1, n_boxes=0), make_sample(61, n_sweeps=10, n_boxes=5), make_sample(62, n_sweeps=1, n_boxes=60),
                make_sample(63, n_sweeps=10, n_boxes=300)]
    samples.append({"point_cloud": np.zeros((0, 4), np.float32), "annotations": [_ann((5, 5, 0), (2, 2, 2))]})                 # empty keyframe
    samples.append(_blob_sample(rng, [(8, 8, 0)], 7, 0.1, [_ann((8, 8, 0), (2, 2, 2))]))                                         # < min_samples
    samples.append(_blob_sample(rng, [(x, 10.0, 0.0) for x in np.arange(-20, 20, 3.0)], 1, 0.0, [_ann((0, 10, 0), (30, 30, 3))]))  # noise only
    samples.append(_blob_sample(rng, [(6, 6, 0), (6, 9, 0), (-6, -6, 0.5)], 200, 0.3,                                          # overlaps
                                [_ann((6, 7.5, 0), (4, 6, 3)), _ann((6, 7.5, 0), (4, 6, 3)), _ann((6, 6, 0), (2, 2, 2)), _ann((6, 9, 0), (2, 2, 2)),
                                 _ann((-6, -6, 0.5), (3, 3, 3)), _ann((-6, -6, 0.5), (1, 1, 1)), _ann((30, 30, 0), (1, 1, 1))]))
    samples.append(_face_sample(rng))
    weird = rng.normal(0, 10, (3000, 4)).astype(np.float32)
    weird[::37, 0] = np.nan; weird[1::37, 1] = np.inf; weird[2::37, 2] = -np.inf; weird[3::37, 2] = np.nan; weird[4::41, :] = np.nan
    samples.append({"point_cloud": weird, "annotations": [_ann((0, 0, 0), (20, 20, 10)), _ann((5, -5, 0), (8, 8, 8))]})
    many, n_blobs = _many_blobs_sample()
    samples.append(many)
    return samples, n_blobs


def _run(eng, db, sentinel=True):
    """run_lidar + run_cluster_match on `db` with sentinel-filled outputs that end in guard rows; returns (lidar rows, match, guards)."""
    import torch
    from msc_geom.engine import ClusterMatchResult
    lr = eng.run_lidar(db, params=_agent_params())
    m = eng.alloc_cluster_match(lr, db.host)
    big_c = torch.full((lr.row_capacity + 8, 3), SENTINEL, dtype=torch.int32, device=eng.device)
    big_b = torch.full((db.host.n_boxes + 8, 5), SENTINEL, dtype=torch.int32, device=eng.device)
    m = ClusterMatchResult(lr, m.sample_box_off, big_c[:lr.row_capacity], big_b[:db.host.n_boxes], m.workspace)
    eng.run_cluster_match(lr, db, out=m)
    return lr.to_host(), m, (big_c, big_b)


def _check_guards(per, m, guards):
    big_c, big_b = (g.cpu().numpy() for g in guards)
    written = np.zeros(big_c.shape[0], bool)
    for r in per:
        written[r["object_off"]:r["object_off"] + len(r["clusters"])] = True
    assert (big_c[~written] == SENTINEL).all()
    assert (big_b[-8:] == SENTINEL).all() and not (big_b[:-8] == SENTINEL).all(1).any()


def _assert_tables_equal(a, b, what=""):
    for k in ("cluster_match", "box_match"):
        assert a[k].shape == b[k].shape and np.array_equal(a[k], b[k]), (what, k)


@pytest.mark.gpu
def test_mixed_batch_is_bit_exact_to_the_oracle(eng, golden_dir):
    from msc_geom.layout import pack_batch
    samples, n_blobs = _mixed_samples(golden_dir)
    hb = pack_batch(samples)
    db = eng.upload(hb)
    launches = eng.kernel_launches
    per, m, guards = _run(eng, db)
    assert eng.kernel_launches - launches == 15 + 3
    got = m.to_host()
    assert len(got) == len(samples)
    _check_guards(per, m, guards)
    want = orc.batch(hb, per)
    for s, (g, (cl, bx)) in enumerate(zip(got, want)):
        assert g["cluster_match"].shape == cl.shape and np.array_equal(g["cluster_match"], cl), s
        assert g["box_match"].shape == bx.shape and np.array_equal(g["box_match"], bx), s
    assert len(per[-1]["clusters"]) >= n_blobs - 5 > 1900                              # the many-blobs sample spans many label tiles
    assert hb.max_boxes_per_sample == 300 and sum((g["cluster_match"][:, 0] >= 0).sum() for g in got) > 100
    face = got[-3]
    assert face["box_match"][0, 3] == face["box_match"][2, 3] >= 0 and face["box_match"][0, 0] == face["box_match"][2, 0]   # duplicates
    assert all(len(g["cluster_match"]) == 0 for g in (got[7], got[8], got[9]))             # empty, < min_samples, noise only
    assert got[9]["box_match"][0, 0] > 0 and got[9]["box_match"][0, 1] == 0


@pytest.mark.gpu
def test_batch_equals_single_samples_permutations_and_tiles(eng, golden_dir):
    from msc_geom import ops
    from msc_geom.layout import pack_batch
    samples, _ = _mixed_samples(golden_dir)
    samples = samples[:-1]
    hb = pack_batch(samples)
    _, m, _ = _run(eng, eng.upload(hb))
    base = m.to_host()
    for s, smp in enumerate(samples):
        one = ops.cluster_match(eng, smp, params=_agent_params())
        _assert_tables_equal(one, base[s], s)
    perm = np.random.default_rng(4).permutation(len(samples))
    _, mp, _ = _run(eng, eng.upload(pack_batch([samples[i] for i in perm])))
    for j, g in enumerate(mp.to_host()):
        _assert_tables_equal(g, base[perm[j]], (j, perm[j]))
    n = 3 * len(samples) - 2
    per, mt, guards = _run(eng, eng.upload_tiled(hb, 3, n))
    _check_guards(per, mt, guards)
    tiled = mt.to_host()
    assert len(tiled) == n
    for j, g in enumerate(tiled):
        _assert_tables_equal(g, base[j % len(samples)], j)


@pytest.mark.gpu
def test_config3_scale(eng):
    from msc_geom.layout import pack_batch
    from msc_geom.synthetic import make_sample
    hb = pack_batch([make_sample(i, n_sweeps=10, n_boxes=60) for i in range(37)])
    db = eng.upload_tiled(hb, 16, 592)
    per, m, guards = _run(eng, db)
    _check_guards(per, m, guards)
    got = m.to_host()
    assert len(got) == 592
    for s in range(0, 592, 37):
        cl, bx = orc.cluster_match(per[s]["object"], per[s]["labels"], len(per[s]["clusters"]), db.host.boxes[s * 60:(s + 1) * 60],
                                   db.host.ego_pose[s], db.host.lidar_calib[s])
        assert np.array_equal(got[s]["cluster_match"], cl) and np.array_equal(got[s]["box_match"], bx), s
    for s in range(37, 592):
        _assert_tables_equal(got[s], got[s % 37], s)
    assert sum(int((g["cluster_match"][:, 0] >= 0).sum()) for g in got[:37]) > 37


def _host_assembly(agent, per, matches, anns):
    from msc_geom.lidar_agent import annotation_match, set_order
    out = []
    for r, mm, a in zip(per, matches, anns):
        order = ([l for l in set_order(r["cluster_first"], r["noise_first"]) if int(r["clusters"][l, 10]) >= 5]
                 if len(r["object"]) >= agent.dbscan_min_samples else [])
        out.append(annotation_match(order, r["clusters"], mm["cluster_match"], mm["box_match"], a))
    return out


@pytest.mark.gpu
def test_agent_annotation_match(eng, golden_dir):
    from msc_geom.layout import pack_batch
    from msc_geom.lidar_agent import LiDARAgent
    from msc_geom.synthetic import make_sample
    samples = [make_sample(70 + i, n_sweeps=1 + 9 * (i % 2), n_boxes=(0, 5, 60, 120)[i]) for i in range(4)]
    agent = LiDARAgent(object(), "m", "LiDARAgent", engine=eng)
    got = agent.process_batch(samples, match_annotations=True)
    plain = agent.process_batch(samples)
    db = eng.upload(pack_batch(samples))
    lr = eng.run_lidar(db, params=agent._params())
    per, matches = lr.to_host(), eng.run_cluster_match(lr, db).to_host()
    want = _host_assembly(agent, per, matches, [s["annotations"] for s in samples])
    assert [g["annotation_match"] for g in got] == want
    assert sum(c["annotation"] is not None for w in want for c in w["clusters"]) > 3
    assert all(c["category"] is not None for w in want for c in w["clusters"] if c["annotation"] is not None)
    for a, b in zip(got, plain):
        a = dict(a)
        a.pop("annotation_match")
        assert json.dumps(a, default=str, sort_keys=True) == json.dumps(b, default=str, sort_keys=True)
        assert "annotation_match" not in b


@pytest.mark.gpu
def test_lazy_loader_batch(eng, tmp_path, devkit_shim):
    from msc_geom import io as mio
    from msc_geom.lidar_agent import LiDARAgent
    scenes = _scenes()
    mio.write_nuscenes_tree(str(tmp_path), scenes)
    eager = devkit_shim.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=3)
    lazy = devkit_shim.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=3, lazy_sweeps=True)
    toks = [t for sc in eager.get_scene_list() for t in eager.scene_sample_tokens(sc["token"])]
    ea = [eager.load_sample(t) for t in toks]
    lz = [lazy.load_sample(t) for t in toks]
    agent = LiDARAgent(object(), "m", "LiDARAgent", engine=eng)
    anns = [s["annotations"] for s in lz]
    got = agent.process_batch(device_batch=eng.upload(mio.stage_batch(lz)), match_annotations=True, annotations=anns)
    want = agent.process_batch(ea, match_annotations=True)
    assert [g["annotation_match"] for g in got] == [w["annotation_match"] for w in want]
    bare = agent.process_batch(device_batch=eng.upload(mio.stage_batch(lz)), match_annotations=True)
    for g, b in zip(got, bare):
        assert g["annotation_match"]["annotations"] == b["annotation_match"]["annotations"]
        assert all(c["category"] is None for c in b["annotation_match"]["clusters"])


@pytest.mark.gpu
def test_lidar_status_and_refusals(eng):
    import torch
    from msc_geom import _capi
    from msc_geom.layout import pack_batch
    from msc_geom.synthetic import make_sample
    hb = pack_batch([make_sample(80, n_sweeps=1, n_boxes=10), make_sample(81, n_sweeps=1, n_boxes=4)])
    db = eng.upload(hb)
    from msc_geom.engine import make_params
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    # a row capacity below the keyframe rows sets msc_lidar_batch's status: the match must not be returned
    small = eng.alloc_lidar(hb)
    small.row_capacity -= 1
    mp = make_params(_agent_params())
    need = int(eng.lib.msc_lidar_batch_workspace_bytes(C.byref(mp), C.c_double(0.5), 2, small.row_capacity))
    lws = torch.empty(need, dtype=torch.uint8, device=eng.device)
    assert eng.lib.msc_lidar_batch(C.byref(mp), C.c_double(0.5), 10, C.byref(db.struct()), C.byref(small.struct()), lws.data_ptr(), need,
                                   stream) == 0
    m = eng.run_cluster_match(small, db)
    with pytest.raises(_capi.MscError, match="status"):
        m.to_host()
    # refusals with real buffers
    lr = eng.run_lidar(db)
    m = eng.alloc_cluster_match(lr, hb)
    bi, rows, bo = db.struct(), lr.struct(), m.struct()
    need = int(eng.lib.msc_cluster_match_batch_workspace_bytes(2, hb.n_boxes, lr.row_capacity))
    ws = m.workspace.data_ptr()
    bad = _capi.MSC_ERR_BAD_ARGUMENT
    call = lambda *a: eng.lib.msc_cluster_match_batch(*a)
    assert call(C.byref(bi), C.byref(rows), 2, C.byref(bo), ws, need - 1, stream) == bad
    assert call(C.byref(bi), C.byref(rows), 1, C.byref(bo), ws, need, stream) == bad
    assert call(C.byref(bi), C.byref(rows), -2, C.byref(bo), ws, need, stream) == bad
    assert call(C.byref(bi), C.byref(rows), 2, None, ws, need, stream) == bad
    assert call(C.byref(bi), C.byref(rows), 2, C.byref(_capi.MscClusterMatchOut(bo.cluster, None)), ws, need, stream) == bad
    assert call(C.byref(bi), C.byref(rows), 2, C.byref(bo), None, need, stream) == bad
    assert call(C.byref(bi), C.byref(rows), 2, C.byref(bo), ws, need, stream) == 0
    assert len(m.to_host()) == 2
    with pytest.raises(_capi.MscError):
        eng.run_cluster_match(lr, eng.upload(pack_batch([make_sample(80, n_sweeps=1, n_boxes=10)])))
    empty = eng.upload(pack_batch([]))
    assert eng.run_cluster_match(eng.run_lidar(empty), empty).to_host() == []
