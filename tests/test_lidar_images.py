"""The LiDAR agent's images batched on the device (msc_keyframe_bev_batch / GeometryEngine.run_lidar_bev, msc_cluster_views_batch /
GeometryEngine.run_cluster_views): every byte equals the per-sample path (finish_bev_layers over ops.keyframe_bev_layers,
finish_cluster_view over ops.cluster_views), which the reference goldens pin."""
import ctypes as C
import os

import numpy as np
import pytest

from msc_geom import _capi
from msc_geom.lidar_agent import bev_stamp, cluster_view_stamp, density_table, finish_bev_layers, finish_cluster_view, set_order

BEV_GEOMETRIES = ((800, 50), (801, 50), (64, 50), (640, 37.5))


def apply_stamp(img, stamp):
    out = np.ascontiguousarray(img).copy()
    flat = out.reshape(-1, 3)
    px, col = stamp[:, 0].astype(np.int64), stamp[:, 1]
    flat[px, 0], flat[px, 1], flat[px, 2] = col & 255, (col >> 8) & 255, (col >> 16) & 255
    return out


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("res,bev_range", BEV_GEOMETRIES)
def test_bev_stamp_equals_the_drawn_overlays(res, bev_range):
    rng = np.random.default_rng(res)
    stamp = bev_stamp(res, bev_range)
    assert stamp.shape[0] > 0 and stamp[:, 0].max() < res * res
    if (res, bev_range) == (800, 50):
        assert stamp.shape[0] == 6199
    for _ in range(3):
        sem = rng.integers(0, 256, (res, res, 3), dtype=np.uint8)
        count = rng.integers(0, 5, (res, res)).astype(np.uint32)
        want = finish_bev_layers(count, np.zeros((res, res), np.float32), sem.copy(), res, bev_range)["semantic"]
        assert np.array_equal(apply_stamp(sem[::-1], stamp), want)


def test_cluster_view_stamp_equals_the_drawn_axes_and_titles():
    rng = np.random.default_rng(4)
    stamp = cluster_view_stamp()
    assert stamp.shape[0] == 1147
    for _ in range(3):
        img = rng.integers(0, 256, (512, 512, 3), dtype=np.uint8)
        assert np.array_equal(apply_stamp(img, stamp), finish_cluster_view(img.copy()))


def test_density_from_a_longer_table_equals_finish_bev_layers():
    """What the device computes -- lut[c] / lut[cmax] * 255 in float32, truncated, from one table longer than any count -- against
    finish_bev_layers' density (flipped), on random count grids, including an all-zero one."""
    rng = np.random.default_rng(9)
    lut = density_table(60000)
    for hi in (0, 1, 2, 7, 300, 50000):
        count = rng.integers(0, hi + 1, (96, 96)).astype(np.uint32)
        want = finish_bev_layers(count, np.zeros((96, 96), np.float32), np.zeros((96, 96, 3), np.uint8), 96, 50)["density"]
        cmax = int(count.max())
        got = np.zeros_like(want) if cmax == 0 else (lut[count] / lut[cmax] * np.float32(255)).astype(np.uint8)
        assert lut.dtype == np.float32 and np.array_equal(got[::-1], want), hi
    assert np.array_equal(density_table(10), lut[:11])


def test_argument_refusals_without_a_device():
    """Bad arguments are refused with MSC_ERR_BAD_ARGUMENT before anything is launched (without a device a launch fails otherwise)."""
    from msc_geom.engine import make_params
    from msc_geom.layout import GeomParams
    lib = _capi.load()
    p = 1 << 20  # a 256-byte aligned address that is never dereferenced
    need = int(lib.msc_keyframe_bev_batch_workspace_bytes(64, 2))
    assert need >= 8 * 64 * 64 * 2 and lib.msc_keyframe_bev_batch_workspace_bytes(0, 2) == 0
    rows = _capi.MscLidarBatchOut(100, p, p, p, p, p, p, p, p, p, p, p)

    def bev(res=64, first=0, n=2, S=3, rows_=rows, lut=p, lut_len=10, sem=p, height=p, dens=p, status=p, ws=p, ws_bytes=need):
        mp = make_params(GeomParams(bev_res=res, bev_range=50.0))
        return lib.msc_keyframe_bev_batch(C.byref(mp), C.byref(rows_) if rows_ is not None else None, S, first, n, lut, lut_len, p, 4, sem,
                                          height, dens, status, ws, ws_bytes, None)

    nulled = _capi.MscLidarBatchOut.from_buffer_copy(rows)
    nulled.ground_off = None
    for kw in ({"res": 0}, {"res": -5}, {"res": 8193}, {"first": -1}, {"n": -1}, {"first": 2, "n": 2}, {"rows_": None}, {"rows_": nulled},
               {"lut": None}, {"lut_len": 0}, {"sem": None}, {"height": None}, {"dens": None}, {"status": None}, {"ws": None},
               {"ws_bytes": need - 1}):
        assert bev(**kw) == _capi.MSC_ERR_BAD_ARGUMENT, kw
    assert bev(n=0, sem=None, height=None, dens=None, status=None, ws=None, ws_bytes=0) == 0

    vneed = int(lib.msc_cluster_views_batch_workspace_bytes(2, 100))
    assert vneed >= 2 * (1 << 20) + 2 * 400 and lib.msc_cluster_views_batch_workspace_bytes(2, 1 << 24) == 0

    def views(v=((0, 10, 0), (10, 30, 1)), n=None, maxp=100, rows_=p, labels=p, out=p, status=p, ws=p, ws_bytes=vneed):
        a = np.ascontiguousarray(np.array(v, np.int32).reshape(-1, 3))
        return lib.msc_cluster_views_batch(rows_, labels, a.ctypes.data, len(a) if n is None else n, maxp, p, 8, out, status, ws, ws_bytes, None)

    for kw in ({"v": ((0, 10, 0), (10, 10, 1))}, {"v": ((0, 10, 0), (12, 10, 1))}, {"v": ((-1, 10, 0), (10, 30, 1))}, {"n": -1},
               {"maxp": -1}, {"maxp": 1 << 24}, {"rows_": None}, {"labels": None}, {"out": None}, {"status": None}, {"ws": None},
               {"ws_bytes": vneed - 1}):
        assert views(**kw) == _capi.MSC_ERR_BAD_ARGUMENT, kw
    assert views(v=(), n=0, rows_=None, labels=None, out=None, status=None, ws=None, ws_bytes=0) == 0


# ------------------------------------------------------------------------------------------------ GPU
def _params():
    from msc_geom.layout import GeomParams
    return GeomParams(bev_res=800)


def _keyframe(sample):
    if sample.get("lidar_sweeps"):
        return sample["lidar_sweeps"][0]["points_raw"][:, :4]
    return np.asarray(sample["point_cloud"], np.float32)


def _golden_samples(golden_dir):
    return [{"point_cloud": np.load(os.path.join(golden_dir, f"keyframe_{n}.npz"))["points"]} for n in ("mock", "edge", "synth", "empty", "flatobj")]


def _mixed_samples(golden_dir):
    """Golden and synthetic keyframes, a sample without sweeps, samples with no ground, no object or neither, and a cell with 40,000
    returns."""
    from msc_geom.synthetic import make_sample
    rng = np.random.default_rng(21)
    ground_only = (rng.uniform(-30, 30, (500, 4)) * [1, 1, 0, 1] + [0, 0, -2.5, 0]).astype(np.float32)
    object_only = (rng.uniform(-40, 40, (800, 4)) * [1, 1, 0.5, 1] + [0, 0, 0.5, 0]).astype(np.float32)
    pile = np.concatenate([np.tile(np.float32([[7.01, -3.02, 0.4, 1.0]]), (40000, 1)), rng.normal(0, 8, (2000, 4))]).astype(np.float32)
    pile[:40000, 2] += np.linspace(0, 1, 40000, dtype=np.float32)
    return (_golden_samples(golden_dir) + [make_sample(3, n_sweeps=1, n_boxes=5), {"point_cloud": ground_only}, {"point_cloud": object_only},
                                           {"point_cloud": np.zeros((0, 4), np.float32)}, {"point_cloud": pile}, make_sample(4, n_sweeps=3, n_boxes=5)])


def _batch(eng, samples, without_sweeps=()):
    from msc_geom.layout import pack_batch
    from tests.test_lidar_batch import _insert_sample_without_sweeps
    hb = pack_batch(samples)
    for j in without_sweeps:
        hb = _insert_sample_without_sweeps(hb, j)
    return eng.run_lidar(eng.upload(hb), params=_params())


def _per_sample_bev(eng, pc, res, bev_range):
    from msc_geom import ops
    from msc_geom.layout import GeomParams
    _, ground, obj = ops.keyframe_filter_split(eng, pc, GeomParams(bev_res=800))
    return finish_bev_layers(*ops.keyframe_bev_layers(eng, ground, obj, res, float(bev_range)), res, bev_range)


def _assert_bev_equal(got, want, what):
    for k in ("semantic", "height", "density"):
        assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k]), (what, k, int((got[k] != want[k]).sum()))


@pytest.mark.gpu
def test_bev_equals_the_reference_goldens(engine, golden_dir):
    lr = _batch(engine, _golden_samples(golden_dir))
    got = engine.run_lidar_bev(lr, 800, 50.0).to_host()
    for i, name in enumerate(("mock", "edge", "synth", "empty", "flatobj")):
        g = np.load(os.path.join(golden_dir, f"keyframe_{name}.npz"))
        _assert_bev_equal(got[i], {k: g[k] for k in ("semantic", "height", "density")}, name)


@pytest.mark.gpu
@pytest.mark.parametrize("res,bev_range", [(800, 50), (513, 30.0)])
def test_bev_equals_the_per_sample_path(engine, golden_dir, res, bev_range):
    samples = _mixed_samples(golden_dir)
    lr = _batch(engine, samples, without_sweeps=(2,))
    keyframes = [_keyframe(s) for s in samples]
    keyframes.insert(2, np.zeros((0, 4), np.float32))
    want = [_per_sample_bev(engine, pc, res, bev_range) for pc in keyframes]
    got = engine.run_lidar_bev(lr, res, bev_range).to_host()
    assert len(got) == len(want) == lr.n_samples
    for i, (g, w) in enumerate(zip(got, want)):
        _assert_bev_equal(g, w, i)
    assert int(want[-2]["density"].max()) == 255 and lr.sample_rows >= 42000


@pytest.mark.gpu
def test_bev_windows_chunks_and_sentinels(engine, golden_dir, monkeypatch):
    import torch
    from msc_geom import engine as engine_mod
    from msc_geom.engine import make_params
    from msc_geom.layout import GeomParams
    samples = _mixed_samples(golden_dir)
    lr = _batch(engine, samples)
    res, rng = 160, 50.0
    want = [_per_sample_bev(engine, _keyframe(s), res, rng) for s in samples]
    per = int(engine.lib.msc_keyframe_bev_batch_workspace_bytes(res, 1))
    monkeypatch.setattr(engine_mod, "BEV_WORKSPACE_PER_CALL", 3 * per)  # calls of 3 samples
    S = lr.n_samples
    for first, n in ((0, S), (1, S - 1), (2, 5), (S - 1, 1), (4, 0)):
        launches = engine.kernel_launches
        got = engine.run_lidar_bev(lr, res, rng, first=first, n=n).to_host()
        assert engine.kernel_launches - launches == 3 * ((n + 2) // 3)
        assert len(got) == n
        for i, g in enumerate(got):
            _assert_bev_equal(g, want[first + i], (first, n, i))
    with pytest.raises(_capi.MscError):
        engine.run_lidar_bev(lr, res, rng, first=S - 1, n=2)
    # C level: sentinel-filled buffers one sample wider on each side; only the window is written, and a repeat gives the same bytes
    first, n = 3, 4
    sem = torch.full((n + 2, res, res, 3), 0xA5, dtype=torch.uint8, device=engine.device)
    hgt = torch.full((n + 2, res, res), -7.0, dtype=torch.float32, device=engine.device)
    den = torch.full((n + 2, res, res), 0x5A, dtype=torch.uint8, device=engine.device)
    status = torch.zeros(1, dtype=torch.int32, device=engine.device)
    need = int(engine.lib.msc_keyframe_bev_batch_workspace_bytes(res, n))
    ws = torch.empty(need, dtype=torch.uint8, device=engine.device)
    lut = torch.from_numpy(density_table(lr.sample_rows)).to(engine.device)
    stamp = torch.from_numpy(bev_stamp(res, rng).view(np.int32)).to(engine.device)
    mp, rows = make_params(GeomParams(bev_res=res, bev_range=rng)), lr.struct()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    outs = []
    for _ in range(2):
        rc = engine.lib.msc_keyframe_bev_batch(C.byref(mp), C.byref(rows), S, first, n, lut.data_ptr(), lut.numel(), stamp.data_ptr(), stamp.shape[0],
                                               sem[1].data_ptr(), hgt[1].data_ptr(), den[1].data_ptr(), status.data_ptr(), ws.data_ptr(), need, stream)
        assert rc == 0
        outs.append((sem.cpu().numpy(), hgt.cpu().numpy(), den.cpu().numpy()))
    assert int(status.item()) == 0
    for (s_, h_, d_) in outs:
        for j in (0, n + 1):
            assert (s_[j] == 0xA5).all() and (h_[j] == -7.0).all() and (d_[j] == 0x5A).all()
        for i in range(n):
            _assert_bev_equal({"semantic": s_[1 + i], "height": h_[1 + i], "density": d_[1 + i]}, want[first + i], i)
    assert all(np.array_equal(a, b) for a, b in zip(outs[0], outs[1]))


@pytest.mark.gpu
def test_bev_table_one_entry_short_raises(engine, golden_dir):
    import torch
    from msc_geom import ops
    from msc_geom.layout import GeomParams
    samples = _mixed_samples(golden_dir)
    lr = _batch(engine, samples)
    counts = []
    for s in samples:
        _, ground, obj = ops.keyframe_filter_split(engine, _keyframe(s), GeomParams(bev_res=800))
        counts.append(int(ops.keyframe_bev_layers(engine, ground, obj, 800, 50.0)[0].max()))
    cmax = max(counts)
    engine._bev_lut = torch.from_numpy(density_table(cmax - 1)).to(engine.device)  # one entry short of the largest count
    lr.sample_rows = cmax - 1
    try:
        with pytest.raises(_capi.MscError, match="density table"):
            engine.run_lidar_bev(lr, 800, 50.0).to_host()
        lr.sample_rows = cmax
        engine._bev_lut = None
        assert len(engine.run_lidar_bev(lr, 800, 50.0).to_host(("density",))) == lr.n_samples
    finally:
        engine._bev_lut = None


@pytest.mark.gpu
def test_cluster_views_equal_the_reference_goldens(engine, golden_dir):
    import torch
    g = np.load(os.path.join(golden_dir, "cluster_views.npz"))
    n = int(g["n"])
    pts = [g[f"pts_{i}"] for i in range(n)]
    rows = np.concatenate([np.zeros((3, 4), np.float32)] + pts)  # three leading rows outside every view
    off = np.cumsum([3] + [len(p) for p in pts])
    views = [(int(off[i]), int(off[i + 1]), 0) for i in range(n)]
    t_rows = torch.from_numpy(rows).to(engine.device)
    t_labels = torch.zeros(len(rows), dtype=torch.int32, device=engine.device)
    got = engine.run_cluster_views(t_rows, t_labels, views).to_host()
    for i in range(n):
        assert np.array_equal(got[i], g[f"img_{i}"]), i
    with pytest.raises(_capi.MscError, match="max_view_points"):
        engine.run_cluster_views(t_rows, t_labels, views, max_view_points=len(pts[3]) - 1).to_host()
    assert np.array_equal(engine.run_cluster_views(t_rows, t_labels, views, max_view_points=len(pts[3])).to_host(), got)


@pytest.mark.gpu
@pytest.mark.parametrize("eps,min_samples", [(0.5, 10), (0.7, 2)])
def test_cluster_views_equal_the_per_sample_path(engine, golden_dir, monkeypatch, eps, min_samples):
    """Views of a run_lidar batch in set_order order, across call boundaries, against agent._cluster_visualizations per sample; the
    chain of 6,000 points is one cluster larger than a CTA's worth of rows, min_samples = 2 gives many tiny clusters."""
    from msc_geom import engine as engine_mod
    from msc_geom.layout import pack_batch
    from msc_geom.lidar_agent import LiDARAgent
    from tests.test_lidar_batch import _serpentine
    samples = _golden_samples(golden_dir)[:3] + [{"point_cloud": _serpentine(6000)}] + _mixed_samples(golden_dir)[5:7]
    lr = engine.run_lidar(engine.upload(pack_batch(samples)), params=_params(), eps=eps, min_samples=min_samples)
    per = lr.to_host()
    agent = LiDARAgent(object(), "m", "LiDARAgent", engine=engine)
    views, want = [], []
    for r in per:
        if len(r["object"]) < min_samples:
            continue
        order = [l for l in set_order(r["cluster_first"], r["noise_first"]) if int(r["clusters"][l, 10]) >= 5]
        views += [(r["object_off"], r["object_off"] + len(r["object"]), l) for l in order]
        want += agent._cluster_visualizations(r["object"], r["labels"].astype(np.int32), order)
    assert len(views) > 12 and max(int(r["clusters"][:, 10].max()) for r in per if len(r["clusters"])) >= 6000
    per_view = int(engine.lib.msc_cluster_views_batch_workspace_bytes(1, 20000))
    monkeypatch.setattr(engine_mod, "CLUSTER_VIEWS_WORKSPACE_PER_CALL", 5 * per_view)  # calls of at most 5 views
    got = engine.run_cluster_views(lr.object, lr.labels, views).to_host()
    assert len(got) == len(want)
    bad = [i for i in range(len(want)) if not np.array_equal(got[i], want[i])]
    assert not bad, bad[:10]


@pytest.mark.gpu
def test_process_batch_images_across_chunks(engine, golden_dir, monkeypatch):
    """process_batch with cluster images drawn a few at a time: the classifier's images and mosaics are still process's."""
    from msc_geom import lidar_agent
    from msc_geom.lidar_agent import LiDARAgent
    from tests.test_lidar_batch import _Recorder, _assert_calls_equal, _json_form
    monkeypatch.setattr(lidar_agent, "CLUSTER_IMAGES_PER_CALL", 7)
    samples = _golden_samples(golden_dir) + _mixed_samples(golden_dir)[5:7]
    ra, rb = _Recorder(), _Recorder()
    a = LiDARAgent(object(), "m", "LiDARAgent", engine=engine, llm=ra.llm, cluster_classifier=ra.classifier)
    b = LiDARAgent(object(), "m", "LiDARAgent", engine=engine, llm=rb.llm, cluster_classifier=rb.classifier)
    want = [a.process(_keyframe(s)) for s in samples]
    got = b.process_batch(samples)
    assert [_json_form(x) for x in got] == [_json_form(x) for x in want]
    _assert_calls_equal(rb.calls, ra.calls)
    assert len(ra.calls) > 2
    for (ma, sa), (mb, sb) in zip(ra.llm_calls, rb.llm_calls):
        assert ma == mb and np.array_equal(sa, sb)
