"""The batched keyframe evidence (msc_lidar_batch, GeometryEngine.run_lidar, LiDARAgent.process_batch): per sample identical to the
single-keyframe path (ops.keyframe_filter_split -> ops.dbscan -> ops.cluster_aabb, LiDARAgent.process) on the sample's keyframe."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from msc_geom.lidar_agent import set_order
from tests.test_loader_on_disk import _scenes, devkit_shim  # noqa: F401  (a written nuScenes tree and the fixture that loads it)


# ------------------------------------------------------------------------------------------------ CPU: the set-iteration order
def _set_iteration(labels):
    uniq = set(labels)
    uniq.discard(-1)
    return [int(l) for l in uniq]


def test_set_order_iterates_like_set_of_labels():
    """DBSCAN-style dense labels 0..k-1 (numbered in any order) and sparse label values, where the set order is not always ascending."""
    rng = np.random.default_rng(7)
    not_ascending = 0
    for trial in range(3000):
        n = int(rng.integers(1, 400))
        raw = rng.integers(-1, int(rng.integers(1, 80)), n)
        if trial % 2:
            ids = np.unique(raw[raw >= 0])
            relabel = dict(zip(ids.tolist(), rng.permutation(len(ids)).tolist()))
            labels = np.array([relabel.get(int(v), -1) for v in raw], np.int64)
            first = [int(np.flatnonzero(labels == c)[0]) for c in range(len(ids))]
        else:
            labels = np.where(raw >= 0, raw * int(rng.integers(1, 40)) + int(rng.integers(0, 1000)), -1).astype(np.int64)
            first = {int(c): int(np.flatnonzero(labels == c)[0]) for c in np.unique(labels[labels >= 0])}
        noise = int(np.flatnonzero(labels == -1)[0]) if (labels == -1).any() else -1
        want = _set_iteration(labels)
        assert set_order(first, noise) == want, labels.tolist()
        not_ascending += want != sorted(want)
    assert not_ascending > 0  # the trap the helper exists for


def test_set_order_empty_and_noise_only():
    assert set_order([], -1) == [] and set_order([], 0) == []
    assert set_order([3], 0) == [0]


# ------------------------------------------------------------------------------------------------ GPU
def _engine():
    from msc_geom.engine import GeometryEngine
    return GeometryEngine()


@pytest.fixture(scope="module")
def eng():
    return _engine()


def _agent_params():
    from msc_geom.layout import GeomParams
    return GeomParams(bev_res=800)


def _keyframe(sample):
    if sample.get("lidar_sweeps"):
        return sample["lidar_sweeps"][0]["points_raw"][:, :4]
    return np.asarray(sample["point_cloud"], np.float32)


def _reference(eng, pc, eps=0.5, min_samples=10):
    from msc_geom import ops
    kept, ground, obj = ops.keyframe_filter_split(eng, pc, _agent_params())
    labels = ops.dbscan(eng, obj[:, :3], eps, min_samples) if len(obj) else np.zeros(0, np.int64)
    k = int(labels.max()) + 1 if labels.size else 0
    table = ops.cluster_aabb(eng, obj, labels.astype(np.int32), k)
    first = np.array([np.flatnonzero(labels == c)[0] for c in range(k)], np.int64)
    noise = int(np.flatnonzero(labels == -1)[0]) if (labels == -1).any() else -1
    return {"counts": (len(kept), len(ground), len(obj)), "ground": ground, "object": obj, "labels": labels, "clusters": table,
            "cluster_first": first, "noise_first": noise}


def _assert_same(got, ref, what=""):
    assert tuple(int(v) for v in got["counts"]) == ref["counts"], what
    for k in ("ground", "object", "labels", "clusters", "cluster_first"):
        assert got[k].shape[0] == ref[k].shape[0] and np.array_equal(got[k], ref[k]), (what, k)
    assert got["noise_first"] == ref["noise_first"], what


def _insert_sample_without_sweeps(hb, j):
    """hb with an extra sample at index j that owns no sweep (and no boxes)."""
    from msc_geom.layout import HostBatch
    ins = lambda a: np.insert(a, j, a[j] if j < len(a) else a[-1], axis=0)
    return HostBatch(hb.n_samples + 1, hb.points, np.insert(hb.sample_sweep_off, j, hb.sample_sweep_off[j]).astype(np.int32), hb.sweep_start,
                     hb.sweep_count, hb.sweep_pose, hb.sweep_time_lag, np.insert(hb.sample_box_off, j, hb.sample_box_off[j]).astype(np.int32),
                     hb.boxes, ins(hb.ego_pose), ins(hb.lidar_calib), ins(hb.cam_ego_pose), ins(hb.cam_calib), ins(hb.cam_K), hb.n_cams,
                     hb.max_boxes_per_sample)


def _edge_clouds():
    rng = np.random.default_rng(11)
    few = np.concatenate([rng.uniform(-20, 20, (40, 4)) * [1, 1, 0, 1] + [0, 0, -2.0, 0],      # ground
                          rng.normal(0, 0.1, (7, 4)) + [8, 8, 0, 0]]).astype(np.float32)         # 7 object rows (< min_samples)
    ground_only = (rng.uniform(-30, 30, (500, 4)) * [1, 1, 0, 1] + [0, 0, -2.5, 0]).astype(np.float32)
    weird = rng.normal(0, 10, (3000, 4)).astype(np.float32)
    weird[::37, 0] = np.nan; weird[1::37, 1] = np.inf; weird[2::37, 2] = -np.inf; weird[3::37, 2] = np.nan; weird[4::41, :] = np.nan
    weird[5::43, 2] = np.float32(-1.4)
    return {"few_objects": few, "all_ground": ground_only, "nan_inf": weird}


def _mixed_samples(golden_dir):
    from msc_geom.nuscenes_loader import create_loader
    from msc_geom.synthetic import make_sample
    samples = [{"point_cloud": np.load(os.path.join(golden_dir, f"keyframe_{n}.npz"))["points"]} for n in ("mock", "edge", "synth", "empty", "flatobj")]
    np.random.seed(0)
    samples.append(create_loader(None, use_mock=True).get_sample_by_scene_index(0, 0))
    samples += [make_sample(3, n_sweeps=1, n_boxes=5), make_sample(4, n_sweeps=10, n_boxes=5)]
    samples.append({"point_cloud": np.zeros((0, 4), np.float32)})
    samples += [{"point_cloud": v} for v in _edge_clouds().values()]
    return samples


@pytest.mark.gpu
def test_batch_equals_the_per_sample_path(eng, golden_dir):
    from msc_geom.layout import pack_batch
    samples = _mixed_samples(golden_dir)
    hb = _insert_sample_without_sweeps(pack_batch(samples), 4)
    got = eng.run_lidar(eng.upload(hb), params=_agent_params()).to_host()
    assert len(got) == len(samples) + 1
    empty = got.pop(4)
    assert tuple(empty["counts"]) == (0, 0, 0) and len(empty["labels"]) == 0 and len(empty["clusters"]) == 0 and empty["noise_first"] == -1
    for i, (s, g) in enumerate(zip(samples, got)):
        _assert_same(g, _reference(eng, _keyframe(s)), i)
    assert sum(len(g["clusters"]) for g in got) > 10  # the batch does cluster something
    for i, name in enumerate(("mock", "edge", "synth", "empty", "flatobj")):  # the reference goldens, through the batch path
        gold = np.load(os.path.join(golden_dir, f"keyframe_{name}.npz"))
        assert int(got[i]["counts"][0]) == len(gold["kept"])
        assert np.array_equal(got[i]["ground"], gold["ground"]) and np.array_equal(got[i]["object"], gold["object"])


@pytest.mark.gpu
def test_clusters_synth_golden_is_reproduced(eng, golden_dir):
    from msc_geom.layout import pack_batch
    from msc_geom.lidar_agent import LiDARAgent
    g = np.load(os.path.join(golden_dir, "clusters_synth.npz"))
    other = {"point_cloud": np.load(os.path.join(golden_dir, "keyframe_synth.npz"))["points"]}
    got = eng.run_lidar(eng.upload(pack_batch([other, {"point_cloud": g["object"]}, other])), params=_agent_params()).to_host()[1]
    assert np.array_equal(got["object"], g["object"]) and np.array_equal(got["labels"], g["labels"])
    order = [l for l in set_order(got["cluster_first"], got["noise_first"]) if got["clusters"][l, 10] >= 5]
    labels = g["labels"]
    assert order == [int(l) for l in set(labels.tolist()) if l != -1 and (labels == l).sum() >= 5]
    meta = LiDARAgent._metadata_of(got["clusters"], order)
    assert len(meta) == len(g["num_points"])
    for i, m in enumerate(meta):
        assert np.array_equal(m["center"], g["center"][i]) and np.array_equal(m["dimensions"], g["dimensions"][i])
        assert m["distance"] == g["distance"][i] and m["num_points"] == g["num_points"][i] and m["direction"] == str(g["direction"][i])


@pytest.mark.gpu
def test_process_batch_on_the_mock_sample_matches_reference(eng, golden_json):
    from msc_geom.lidar_agent import LiDARAgent
    from msc_geom.nuscenes_loader import create_loader
    np.random.seed(0)
    sample = create_loader(None, use_mock=True).get_sample_by_scene_index(0, 0)
    agent = LiDARAgent(object(), "m", "LiDARAgent", engine=eng, llm=lambda *a, **k: "STUB",
                       cluster_classifier=lambda images, mosaic, batch: [{"category": "car", "confidence": 0.9} for _ in batch])
    out = agent.process_batch([sample])[0]
    ref = golden_json["process_mock"]
    assert out["bev_metadata"] == ref["bev_metadata"] and out["structured_report"] == ref["structured_report"]
    assert out["observations"] == ref["observations"] and out["agent"] == "LiDARAgent" and out["modality"] == "lidar"
    sf = dict(out["semantic_features"]); near = sf.pop("nearest_object")
    rf = dict(ref["semantic_features"]); rd = rf.pop("nearest_object_distance")
    assert sf == rf and ((near is None and rd is None) or float(near.distance) == rd)
    assert json.loads(json.dumps(out["detected_objects"])) == ref["detected_objects"]


class _Recorder:
    def __init__(self):
        self.calls, self.llm_calls = [], []

    def classifier(self, images, mosaic, meta):
        self.calls.append((images, mosaic, meta))
        cats = ("car", "truck", "unknown", "pedestrian", "bus")
        return [{"category": cats[m["index"] % 5], "confidence": 0.2 + 0.1 * (m["index"] % 8)} for m in meta]

    def llm(self, messages, **kw):
        self.llm_calls.append((messages, kw.get("bev_semantic")))
        return "seen %d" % len(self.llm_calls)


def _json_form(d):
    from msc_geom.lidar_agent import LiDARAgent
    d = dict(d)
    sf = dict(d["semantic_features"])
    near = sf.pop("nearest_object")
    sf["nearest"] = None if near is None else LiDARAgent._object_to_dict(near)
    d["semantic_features"] = sf
    return json.loads(json.dumps(d, default=float))


def _assert_calls_equal(a, b):
    assert len(a) == len(b)
    for (ia, ma, da), (ib, mb, db) in zip(a, b):
        assert len(ia) == len(ib) and all(np.array_equal(x, y) for x, y in zip(ia, ib)) and np.array_equal(ma, mb)
        assert json.loads(json.dumps(da, default=lambda v: np.asarray(v).tolist())) == json.loads(json.dumps(db, default=lambda v: np.asarray(v).tolist()))


@pytest.mark.gpu
def test_process_batch_equals_process(eng, golden_dir):
    from msc_geom.lidar_agent import LiDARAgent
    samples = _mixed_samples(golden_dir)
    contexts = [None if i % 2 else {"camera": "sample %d" % i} for i in range(len(samples))]
    ra, rb = _Recorder(), _Recorder()
    a = LiDARAgent(object(), "m", "LiDARAgent", engine=eng, llm=ra.llm, cluster_classifier=ra.classifier)
    b = LiDARAgent(object(), "m", "LiDARAgent", engine=eng, llm=rb.llm, cluster_classifier=rb.classifier)
    want = [a.process(_keyframe(s), c) for s, c in zip(samples, contexts)]
    got = b.process_batch(samples, contexts=contexts)
    assert [_json_form(x) for x in got] == [_json_form(x) for x in want]
    assert len(ra.calls) > 2
    _assert_calls_equal(rb.calls, ra.calls)
    assert len(ra.llm_calls) == len(rb.llm_calls) == len(samples)
    for (ma, sa), (mb, sb) in zip(ra.llm_calls, rb.llm_calls):
        assert ma == mb and np.array_equal(sa, sb)
    # without injected callables: no images, no BEV, the same dicts
    plain = LiDARAgent(object(), "m", "LiDARAgent", engine=eng)
    assert [_json_form(x) for x in plain.process_batch(samples)] == [_json_form(plain.process(_keyframe(s))) for s in samples]
    # eps / min_samples are the agent's
    a.dbscan_eps, a.dbscan_min_samples, b.dbscan_eps, b.dbscan_min_samples = 0.3, 4, 0.3, 4
    ra.calls.clear(); rb.calls.clear()
    want = [a.process(_keyframe(s)) for s in samples[:8]]
    assert [_json_form(x) for x in b.process_batch(samples[:8])] == [_json_form(x) for x in want]
    _assert_calls_equal(rb.calls, ra.calls)


@pytest.mark.gpu
@pytest.mark.parametrize("eps,min_samples", [(0.5, 10), (0.3, 4)])
def test_labels_equal_sklearn(eng, eps, min_samples):
    from sklearn.cluster import DBSCAN
    from msc_geom.layout import pack_batch
    from msc_geom.synthetic import make_sample
    rng = np.random.default_rng(5)
    blobs = np.concatenate([rng.normal(c, s, (m, 3)) for c, s, m in [((3, 0, 0), 0.3, 400), ((5.2, 0, 0), 0.35, 300), ((10, 5, 1), 0.15, 60),
                                                                      ((-8, -8, 0), 1.5, 800), ((4, -9, 0.5), 0.05, 12)]])
    blob_pc = np.concatenate([blobs, np.ones((len(blobs), 1))], 1).astype(np.float32)
    samples = [make_sample(i, n_sweeps=1, n_boxes=5) for i in range(3)] + [{"point_cloud": blob_pc}]
    got = eng.run_lidar(eng.upload(pack_batch(samples)), params=_agent_params(), eps=eps, min_samples=min_samples).to_host()
    checked = 0
    for g in got:
        obj = g["object"][:, :3].astype(np.float64)
        if len(obj) >= 12:
            assert np.array_equal(g["labels"], DBSCAN(eps=eps, min_samples=min_samples).fit(obj).labels_)
            checked += 1
    assert checked == len(samples)


@pytest.mark.gpu
def test_samples_are_isolated(eng, golden_dir):
    from msc_geom.layout import pack_batch
    p = _agent_params()
    synth = np.load(os.path.join(golden_dir, "keyframe_synth.npz"))["points"]
    alone = eng.run_lidar(eng.upload(pack_batch([{"point_cloud": synth}])), params=p).to_host()[0]
    two = eng.run_lidar(eng.upload(pack_batch([{"point_cloud": synth}, {"point_cloud": synth}])), params=p).to_host()
    for g in two:
        _assert_same(g, _as_ref(alone))
    # a second sample whose points lie within eps of the first's: each alone, never merged
    rng = np.random.default_rng(3)
    a = np.concatenate([rng.normal([6, 6, 0], 0.3, (300, 3)), np.ones((300, 1))], 1).astype(np.float32)
    b = a.copy(); b[:, 0] += 0.2
    both = eng.run_lidar(eng.upload(pack_batch([{"point_cloud": a}, {"point_cloud": b}])), params=p).to_host()
    for pc, g in zip((a, b), both):
        _assert_same(g, _reference(eng, pc))
        assert len(g["clusters"]) >= 1 and g["clusters"][:, 10].sum() <= len(pc)
    # permuting the samples permutes the results
    samples = _mixed_samples(golden_dir)
    base = eng.run_lidar(eng.upload(pack_batch(samples)), params=p).to_host()
    perm = np.random.default_rng(1).permutation(len(samples))
    shuffled = eng.run_lidar(eng.upload(pack_batch([samples[i] for i in perm])), params=p).to_host()
    for j, i in enumerate(perm):
        _assert_same(shuffled[j], _as_ref(base[i]), (j, i))
    # device-tiled copies give identical results
    hb = pack_batch(samples)
    tiled = eng.run_lidar(eng.upload_tiled(hb, 3, 3 * len(samples) - 2), params=p).to_host()
    assert len(tiled) == 3 * len(samples) - 2
    for j, g in enumerate(tiled):
        _assert_same(g, _as_ref(base[j % len(samples)]), j)


def _as_ref(g):
    return {"counts": tuple(int(v) for v in g["counts"]), **{k: g[k] for k in ("ground", "object", "labels", "clusters", "cluster_first")},
            "noise_first": g["noise_first"]}


def _serpentine(n, step=0.04):
    """n points spaced `step` apart along a path that stays inside the keyframe gate: 70 m rows joined by 2 m rungs."""
    pts, x, y, d = [], -35.0, -30.0, 1.0
    while len(pts) < n:
        pts.append((x, y))
        if (d > 0 and x + step > 35.0) or (d < 0 and x - step < -35.0):
            for _ in range(50):
                y += step
                pts.append((x, y))
            d = -d
        else:
            x += d * step
    xy = np.array(pts[:n])
    return np.stack([xy[:, 0], xy[:, 1] + 0.01 * np.sin(np.arange(n)), np.zeros(n), np.ones(n)], 1).astype(np.float32)


@pytest.mark.gpu
def test_worst_case_merges_in_one_sweep(eng, golden_dir):
    from msc_geom.layout import pack_batch
    chain = _serpentine(6000)
    lattice = np.stack(np.meshgrid(np.arange(12) * 0.5 + 5, np.arange(12) * 0.5 + 5, np.arange(3) * 0.5), -1).reshape(-1, 3)
    lattice = np.concatenate([lattice, np.ones((len(lattice), 1))], 1).astype(np.float32)     # distances exactly eps
    synth = {"point_cloud": np.load(os.path.join(golden_dir, "keyframe_synth.npz"))["points"]}
    clouds = [chain, chain[::-1].copy(), lattice]
    got = eng.run_lidar(eng.upload(pack_batch([synth, {"point_cloud": chain}, synth, {"point_cloud": chain[::-1].copy()},
                                               {"point_cloud": lattice}, synth])), params=_agent_params()).to_host()   # status clear, or it raises
    for pc, g in zip(clouds, (got[1], got[3], got[4])):
        assert len(g["object"]) == len(pc)
        _assert_same(g, _reference(eng, pc))
    for g in (got[1], got[3]):
        assert g["labels"].max() == 0 and (g["labels"] == 0).all() and len(g["clusters"]) == 1


@pytest.mark.gpu
def test_config3_scale(eng):
    from msc_geom.layout import pack_batch
    from msc_geom.synthetic import make_sample
    samples = [make_sample(i, n_sweeps=10, n_boxes=60) for i in range(37)]
    db = eng.upload_tiled(pack_batch(samples), 16, 592)
    got = eng.run_lidar(db, params=_agent_params()).to_host()
    assert len(got) == 592
    for i in (0, 1, 36, 37, 300, 591):
        _assert_same(got[i], _reference(eng, _keyframe(samples[i % 37])), i)
    for i in range(37, 592):
        assert np.array_equal(got[i]["labels"], got[i % 37]["labels"]) and np.array_equal(got[i]["clusters"], got[i % 37]["clusters"])


@pytest.mark.gpu
def test_lazy_loader_batch(eng, tmp_path, devkit_shim):
    from msc_geom import io as mio
    from msc_geom.lidar_agent import LiDARAgent
    scenes = _scenes()
    mio.write_nuscenes_tree(str(tmp_path), scenes)
    eager = devkit_shim.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=3)
    lazy = devkit_shim.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=3, lazy_sweeps=True)
    toks = [t for sc in eager.get_scene_list() for t in eager.scene_sample_tokens(sc["token"])]
    lz = [lazy.load_sample(t) for t in toks]
    assert all(s["point_cloud"] is None for s in lz)
    rec_a, rec_b = _Recorder(), _Recorder()
    a = LiDARAgent(object(), "m", "LiDARAgent", engine=eng, llm=rec_a.llm, cluster_classifier=rec_a.classifier)
    b = LiDARAgent(object(), "m", "LiDARAgent", engine=eng, llm=rec_b.llm, cluster_classifier=rec_b.classifier)
    want = [a.process(eager.load_sample(t)["point_cloud"]) for t in toks]
    got = b.process_batch(device_batch=eng.upload(mio.stage_batch(lz)))
    assert [_json_form(x) for x in got] == [_json_form(x) for x in want]
    _assert_calls_equal(rec_b.calls, rec_a.calls)


@pytest.mark.gpu
def test_refusals_and_empty_batch(eng):
    import torch
    from msc_geom import _capi
    from msc_geom.engine import make_params
    from msc_geom.layout import pack_batch
    hb = pack_batch([{"point_cloud": np.random.default_rng(0).normal(0, 5, (500, 4)).astype(np.float32)}])
    db = eng.upload(hb)
    for eps, ms in ((0.0, 10), (-1.0, 10), (float("nan"), 10), (0.5, 0), (0.5, -3)):
        with pytest.raises(_capi.MscError) as e:
            eng.run_lidar(db, eps=eps, min_samples=ms)
        assert e.value.status == _capi.MSC_ERR_BAD_ARGUMENT
    out = eng.alloc_lidar(hb)
    mp = make_params(_agent_params())
    need = int(eng.lib.msc_lidar_batch_workspace_bytes(C.byref(mp), C.c_double(0.5), 1, out.row_capacity))
    assert need > 0 and int(eng.lib.msc_lidar_batch_workspace_bytes(C.byref(mp), C.c_double(0.0), 1, out.row_capacity)) == 0
    ws = torch.empty(need, dtype=torch.uint8, device=eng.device)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    bi, bo = db.struct(), out.struct()
    assert eng.lib.msc_lidar_batch(C.byref(mp), C.c_double(0.5), 10, C.byref(bi), C.byref(bo), ws.data_ptr(), need - 1, stream) == _capi.MSC_ERR_BAD_ARGUMENT
    assert eng.lib.msc_lidar_batch(C.byref(mp), C.c_double(0.5), 10, C.byref(bi), None, ws.data_ptr(), need, stream) == _capi.MSC_ERR_BAD_ARGUMENT
    nulled = _capi.MscLidarBatchOut.from_buffer_copy(bo)
    nulled.labels = None
    assert eng.lib.msc_lidar_batch(C.byref(mp), C.c_double(0.5), 10, C.byref(bi), C.byref(nulled), ws.data_ptr(), need, stream) == _capi.MSC_ERR_BAD_ARGUMENT
    assert eng.lib.msc_lidar_batch(C.byref(mp), C.c_double(0.5), 10, C.byref(bi), C.byref(bo), ws.data_ptr(), need, stream) == 0
    # n_samples = 0: a successful no-op, whatever the buffers
    empty_in = _capi.MscBatchIn()
    assert eng.lib.msc_lidar_batch(C.byref(mp), C.c_double(0.5), 10, C.byref(empty_in), C.byref(_capi.MscLidarBatchOut()), None, 0, stream) == 0
    res = eng.run_lidar(eng.upload(pack_batch([])))
    assert res.to_host() == []
    # a row capacity below the keyframe rows is reported through the status word
    small = eng.alloc_lidar(hb)
    small.row_capacity = out.row_capacity - 1
    need = int(eng.lib.msc_lidar_batch_workspace_bytes(C.byref(mp), C.c_double(0.5), 1, small.row_capacity))
    ws = torch.empty(need, dtype=torch.uint8, device=eng.device)
    assert eng.lib.msc_lidar_batch(C.byref(mp), C.c_double(0.5), 10, C.byref(bi), C.byref(small.struct()), ws.data_ptr(), need, stream) == 0
    with pytest.raises(_capi.MscError, match="row_capacity"):
        small.to_host()
