"""GPU parity tests: every CUDA entry point of the C-ABI against the oracle and the reference-generated goldens.
Bar: bit-exact for integer / byte / index outputs and for order-independent floats; float tolerances are written
where an order- or library-dependent float is compared."""
import ctypes as C
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from msc_geom import _capi, ops
from msc_geom.layout import GeomParams, HostBatch, boxes_from_annotations, pack_batch, tile_batch
from msc_geom.synthetic import edge_case_cloud, make_sample
from tests import oracle_bridge as OB

IDENT7 = np.array([0, 0, 0, 1, 0, 0, 0.0])


DEFAULT_CONFIGS = _capi.FUSED_CONFIGS  # 10: stream4.cu (default), 7: fused_stream.cu (the TMA-ring generation)


def check_fused(eng, samples, params=None, config=None, n_cams=6):
    """Run the fused path and compare every output with the oracle; config=None checks every shape in DEFAULT_CONFIGS."""
    if config is None:
        for cfg in DEFAULT_CONFIGS:
            res = check_fused(eng, samples, params=params, config=cfg, n_cams=n_cams)
        _capi.set_option("config", _capi.DEFAULT_FUSED_CONFIG)
        return res
    p = params or GeomParams()
    _capi.set_option("config", config)
    hb = pack_batch(samples, n_cams=n_cams)
    out = eng.run_fused(eng.upload(hb), params=p)
    import torch
    torch.cuda.synchronize()
    got = out.to_host()
    for i in range(hb.n_samples):
        ref = OB.oracle_fused(hb, i, p)
        b0, b1 = hb.sample_box_off[i], hb.sample_box_off[i + 1]
        for k in ("box_count", "box_nearest", "box_centroid", "proj_visible", "proj_extent"):
            assert np.array_equal(got[k][b0:b1], ref[k], equal_nan=True), (config, i, k)
        for k in ("bev_count", "bev_isum_q", "bev_height"):
            assert np.array_equal(got[k][i], ref[k]), (config, i, k, int((got[k][i] != ref[k]).sum()))
        assert np.array_equal(got["stats"][i][:13], ref["stats"][:13]), (config, i, got["stats"][i], ref["stats"])
        # size-independent invariants
        st = got["stats"][i]
        assert st[3] + st[4] == st[2] and int(got["bev_count"][i].sum()) == st[2] and st[1] <= st[0]
    return hb, got


@pytest.mark.parametrize("config", [10, 7])
def test_fused_config3_shape(engine, config):
    check_fused(engine, [make_sample(i, n_sweeps=10, n_boxes=60) for i in range(2)], config=config)
    if config == 10:  # the standard configuration takes the compile-time-constant instantiation of stream4.cu; the generic one must agree
        assert _capi.get_option("last_standard") == 1
        try:
            _capi.set_option("standard", 0)
            check_fused(engine, [make_sample(i, n_sweeps=10, n_boxes=60) for i in range(2)], config=config)
            assert _capi.get_option("last_standard") == 0
            check_fused(engine, [make_sample(5, n_sweeps=3, n_boxes=130)], config=config)       # more boxes than the standard capacity
            _capi.set_option("standard", 1)
            check_fused(engine, [make_sample(5, n_sweeps=3, n_boxes=130)], config=config)
            assert _capi.get_option("last_standard") == 0
            check_fused(engine, [make_sample(6, n_sweeps=3, n_boxes=128)], config=config)       # exactly the standard capacity
            assert _capi.get_option("last_standard") == 1
        finally:
            _capi.set_option("standard", 1)


def test_fused_mini_boxes_and_mixed_sweeps(engine):
    check_fused(engine, [make_sample(20 + i, n_sweeps=1 + 3 * (i % 3), n_boxes="mini") for i in range(4)])


def test_fused_ragged_and_empty_inputs(engine):
    a = make_sample(30, n_sweeps=4, n_boxes=7)
    sw = a["lidar_sweeps"]
    sw[0]["points_raw"] = sw[0]["points_raw"][:1001]          # not a multiple of 4 or 64
    sw[1]["points_raw"] = sw[1]["points_raw"][:0]             # empty sweep
    sw[2]["points_raw"] = sw[2]["points_raw"][:63]            # shorter than one warp tile
    sw[3]["points_raw"] = sw[3]["points_raw"][:64 * 32 + 1]   # one point into the next round of warp tiles
    b = make_sample(31, n_sweeps=2, n_boxes=0)                # no boxes
    c = make_sample(32, n_sweeps=1, n_boxes=3)
    c["lidar_sweeps"] = [dict(c["lidar_sweeps"][0], points_raw=c["lidar_sweeps"][0]["points_raw"][:0])]  # no points at all
    d = {"point_cloud": np.random.default_rng(5).normal(0, 12, (5000, 4)).astype(np.float32), "annotations": []}  # plain reference-style sample
    for cfg in DEFAULT_CONFIGS:
        check_fused(engine, [a, b, c, d], config=cfg)
    check_fused(engine, [d])                    # a batch without a single box
    check_fused(engine, [c])                    # ... and one without a single point


def test_fused_edge_queue_counter_spill(engine):
    """stream4.cu keeps the exact wedge tests' per-camera counts in eight 8-bit counters per lane and spills them before the 255th
    queue drain of a sample part.  A 30-sweep sample classified on 4 m cull cells (most cells are crossed by an image-column ray)
    with a 16-cell window sends well over 255 x 32 points per warp through the edge queue."""
    s = make_sample(47, n_sweeps=30, n_boxes=12)
    try:
        _capi.set_option("cull_shift", 3)
        _capi.set_option("window", 16)
        for ppt, grid in ((2, 1), (4, 3)):  # (few CTAs: ~590 / ~390 drains per warp and sample part)
            _capi.set_option("ppt", ppt)
            _capi.set_option("grid", grid)
            check_fused(engine, [s], config=10)
    finally:
        for k, v in (("ppt", _capi.DEFAULT_FUSED_PPT), ("grid", 0), ("window", 0), ("cull_shift", -1), ("config", _capi.DEFAULT_FUSED_CONFIG)):
            _capi.set_option(k, v)


def test_fused_crowded_cell_and_max_boxes(engine):
    s = make_sample(40, n_sweeps=2, n_boxes=60)
    base = s["annotations"][0]
    for k in range(9):  # nine boxes stacked on one spot: more than four ids per cull cell -> test-every-box path
        a = dict(s["annotations"][1 + k])
        a["translation"] = [base["translation"][0] + 0.05 * k, base["translation"][1], base["translation"][2]]
        a["rotation"] = base["rotation"]
        a["size"] = base["size"]
        s["annotations"][1 + k] = a
    hb, got = check_fused(engine, [s])
    assert got["box_count"][:10].min() > 0
    big = make_sample(41, n_sweeps=1, n_boxes=255)
    check_fused(engine, [big])


def test_fused_under_declared_max_boxes_sets_the_flag(engine):
    """A caller that under-declares max_boxes_per_sample: the boxes the kernel has room for are exact (fused_stream.cu: the declared
    number; stream4.cu sizes its tables for at least 128 boxes), the overflow bit of stats[13] is set for a sample with more,
    everything that does not depend on boxes is unaffected -- in both kernels."""
    import dataclasses
    import torch
    s = [make_sample(45, n_sweeps=2, n_boxes=140), make_sample(46, n_sweeps=1, n_boxes=4)]
    hb = pack_batch(s)
    p = GeomParams()
    cut = dataclasses.replace(hb, max_boxes_per_sample=5)
    for cfg in DEFAULT_CONFIGS:
        room = 128 if cfg == 10 else 5
        _capi.set_option("config", cfg)
        out = engine.run_fused(engine.upload(cut), params=p); torch.cuda.synchronize()
        got = out.to_host()
        for i in range(2):
            ref = OB.oracle_fused(hb, i, p)
            b0 = hb.sample_box_off[i]
            n_ok = min(room, hb.sample_box_off[i + 1] - b0)
            for k in ("box_count", "box_nearest", "box_centroid"):
                assert np.array_equal(got[k][b0:b0 + n_ok], ref[k][:n_ok]), (cfg, i, k)
            for k in ("proj_visible", "proj_extent"):
                assert np.array_equal(got[k][b0:hb.sample_box_off[i + 1]], ref[k]), (cfg, i, k)
            assert np.array_equal(got["bev_count"][i], ref["bev_count"]) and np.array_equal(got["stats"][i][:13], ref["stats"][:13])
            assert bool(got["stats"][i][13] >> 31) == (i == 0), (cfg, i, got["stats"][i][13])
    _capi.set_option("config", _capi.DEFAULT_FUSED_CONFIG)


def test_fused_fov_filter_and_weird_values(engine):
    s = make_sample(50, n_sweeps=3, n_boxes=30)
    raw = s["lidar_sweeps"][1]["points_raw"]
    raw[::7, 3] = -5.0          # negative intensity clamps to 0
    raw[1::7, 3] = 300.25       # clamps to 65535 / 256
    raw[2::7, 3] = np.nan
    raw[3::11, 0] = np.nan      # NaN coordinates fail every compare
    raw[5::13, 2] = np.inf
    raw[6::17, 3] = 17.123
    check_fused(engine, [s])
    check_fused(engine, [s], params=GeomParams(fov_keep_mask=0b000001))
    check_fused(engine, [s], params=GeomParams(fov_keep_mask=0b101000))


def test_fused_threshold_points_identity_pose(engine):
    """Points exactly on every strict threshold (lidar_agent.py:106-110, :128) and BEV cell edge, through an identity sweep."""
    pc = edge_case_cloud()
    rng = np.random.default_rng(3)
    extra = np.stack([np.float32(v) for v in (49.999996, -49.999996, 1.0000001, 7.4999995)]).astype(np.float32)
    pts = np.concatenate([pc, np.stack([rng.choice(extra, 500), rng.choice(extra, 500), rng.uniform(-3, 5, 500).astype(np.float32),
                                        rng.uniform(0, 255, 500).astype(np.float32)], 1)])
    anns = []
    for cx, cy in [(10.0, 0.0), (-7.0, 3.0), (3.0, -7.0)]:  # axis-aligned boxes whose faces pass through many of the grid-aligned points
        anns.append({"category_name": "vehicle.car", "translation": [cx, cy, 0.0], "size": [2.0, 4.0, 2.0], "rotation": [1.0, 0.0, 0.0, 0.0]})
    sample = {"point_cloud": pts, "annotations": anns, "ego_pose": IDENT7, "lidar_calib": IDENT7}
    hb, got = check_fused(engine, [sample], n_cams=6)
    assert got["box_count"].sum() > 0


def test_fused_other_grid_and_exact_division_path(engine):
    """A divisor that is not on the Markstein whitelist takes the IEEE-division instantiation."""
    s = [make_sample(60 + i, n_sweeps=2, n_boxes=25) for i in range(2)]
    check_fused(engine, s, params=GeomParams(range_max=40.0, bev_range=45.0, bev_res=150))
    assert _capi.get_option("last_fastdiv") == 0
    check_fused(engine, s, params=GeomParams(range_max=30.0, bev_range=32.0, bev_res=128, z_max=3.0, ground_z=-1.0, remove_close_radius=2.5))
    check_fused(engine, s)
    assert _capi.get_option("last_fastdiv") == 1
    # a grid smaller than the fine edge-class table of the streaming kernel: the table then covers every cell, clipped edge cells included
    check_fused(engine, s, params=GeomParams(range_max=9.5, bev_range=10.0, bev_res=40))
    check_fused(engine, s, params=GeomParams(range_max=24.0, bev_range=16.0, bev_res=48))   # range beyond the grid: points clip into edge cells
    # cell sizes just above a power-of-two fraction of 2 m (0.512 m, 0.256 m): the automatic cull grid is capped at 64 x 64 cells so that
    # its tables fit beside 32 warp blocks (a 100 x 100 grid of 1.024 m cells would not)
    check_fused(engine, s, params=GeomParams(range_max=50.0, bev_range=51.2, bev_res=200))
    check_fused(engine, s, params=GeomParams(range_max=50.0, bev_range=51.2, bev_res=400))
    check_fused(engine, s, params=GeomParams(range_max=50.0, bev_range=100.0, bev_res=400))


def test_fused_many_sweeps_and_camera_counts(engine):
    """More sweeps than the kernel caches in shared memory (64): the sweep table and poses fall back to global memory.
    Also 0 and 8 cameras."""
    from msc_geom.geometry import ref_from_sweep
    base = make_sample(95, n_sweeps=10, n_boxes=12)
    sw = []
    for k in range(70):
        src = base["lidar_sweeps"][k % 10]
        M = src["ref_from_sensor"].copy()
        M[:, 3] += 0.01 * k                         # every sweep gets its own transform
        sw.append(dict(src, points_raw=src["points_raw"][k * 97: k * 97 + 700 + 13 * k], ref_from_sensor=M))
    many = dict(base, lidar_sweeps=sw)
    for cfg in DEFAULT_CONFIGS:
        check_fused(engine, [many, make_sample(96, n_sweeps=2, n_boxes=5)], config=cfg)
    s0 = make_sample(97, n_sweeps=2, n_boxes=9)
    s0["cameras"] = []
    check_fused(engine, [s0], params=GeomParams(n_cams=0), n_cams=0)
    s8 = make_sample(98, n_sweeps=2, n_boxes=9)
    s8["cameras"] = s8["cameras"] + [dict(s8["cameras"][1], channel="CAM_X1"), dict(s8["cameras"][4], channel="CAM_X2")]
    check_fused(engine, [s8], params=GeomParams(n_cams=8), n_cams=8)


def test_fused_fov_counts_off_and_small_window(engine):
    s = [make_sample(70, n_sweeps=2, n_boxes=20)]
    _capi.set_option("fov", 0)
    try:
        p = GeomParams()
        hb = pack_batch(s)
        import torch
        got = engine.run_fused(engine.upload(hb), params=p); torch.cuda.synchronize(); got = got.to_host()
        ref = OB.oracle_fused(hb, 0, p)
        assert np.array_equal(got["stats"][0][:5], ref["stats"][:5]) and (got["stats"][0][5:13] == 0).all()
        assert np.array_equal(got["bev_count"][0], ref["bev_count"]) and np.array_equal(got["box_count"], ref["box_count"])
    finally:
        _capi.set_option("fov", 1)
    for w in (2, 40, 0):  # almost everything through the 64-bit global reductions, then the default window
        _capi.set_option("window", w)
        check_fused(engine, s)
    _capi.set_option("window", 0)


def test_fused_static_partition_over_ctas(engine):
    """stream4.cu partitions a batch statically in warp tiles: CTA b of G owns global tiles [b T / G, (b + 1) T / G), so samples
    straddle CTA boundaries and merge their parts with integer reductions (the last ticket finalises).  Results must not depend on
    G -- forced grids from one CTA to more CTAs than tiles, the automatic one, one keyframe, empty samples at either end."""
    s = [make_sample(80 + i, n_sweeps=1 + 4 * (i % 3), n_boxes=15 + 40 * i) for i in range(3)]
    s.append({"point_cloud": np.random.default_rng(6).normal(0, 12, (3000, 4)).astype(np.float32), "annotations": []})
    empty = make_sample(32, n_sweeps=1, n_boxes=3)
    empty["lidar_sweeps"] = [dict(empty["lidar_sweeps"][0], points_raw=empty["lidar_sweeps"][0]["points_raw"][:0])]
    try:
        for ppt in (4, 2):  # both launch shapes: 512 threads x 4 points per lane, 1024 x 2
            _capi.set_option("ppt", ppt)
            for grid in (1, 2, 3, 7, 37, 148, 0):
                _capi.set_option("grid", grid)
                check_fused(engine, s, config=10)
                assert _capi.get_option("last_config") == 10 and _capi.get_option("threads") == (512 if ppt == 4 else 1024)
                assert _capi.get_option("last_grid") == grid or grid == 0
        check_fused(engine, [make_sample(90, n_sweeps=1, n_boxes=60)], config=10)   # BASELINE config 2: one keyframe
        assert _capi.get_option("last_grid") > 1
        for grid in (1, 5, 148):
            _capi.set_option("grid", grid)
            check_fused(engine, [empty, s[0], empty, empty, s[3], empty], config=10)
            check_fused(engine, [empty, empty], config=10)
        tiny = make_sample(91, n_sweeps=1, n_boxes=19)                    # fewer warp tiles (87) than CTAs: most CTAs own nothing,
        tiny["lidar_sweeps"][0]["points_raw"] = tiny["lidar_sweeps"][0]["points_raw"][:11029]   # every tile is a part of its own
        for grid in (148, 100, 87, 86):
            _capi.set_option("grid", grid)
            check_fused(engine, [tiny], config=10)
        _capi.set_option("window", 20)                                    # most cells through the global reductions, partitioned as well
        _capi.set_option("grid", 11)
        check_fused(engine, s, config=10)
    finally:
        _capi.set_option("grid", 0)
        _capi.set_option("ppt", _capi.DEFAULT_FUSED_PPT)
        _capi.set_option("window", 0)
        _capi.set_option("config", _capi.DEFAULT_FUSED_CONFIG)


def test_fused_stream4_random_shapes_and_options(engine):
    """stream4.cu against the oracle on random batch shapes crossed with random launch options: points per lane (1024 x 2 / 512 x 4),
    grid (how samples straddle CTAs), window size, cull-cell size, the compile-time-constant instantiation on / off, grid geometry."""
    rng = np.random.default_rng(2024)
    try:
        for trial in range(8):
            n = int(rng.integers(1, 5))
            s = [make_sample(int(rng.integers(300, 400)), n_sweeps=int(rng.integers(1, 6)), n_boxes=int(rng.integers(0, 90))) for _ in range(n)]
            for smp in s:  # ragged sweeps: lengths that leave partial warp tiles of either shape
                for sw in smp["lidar_sweeps"]:
                    sw["points_raw"] = sw["points_raw"][: int(rng.integers(1, 34720))]
            params = None
            if trial % 3 == 2:
                params = GeomParams(range_max=float(rng.choice([30.0, 40.0, 50.0])), bev_range=float(rng.choice([32.0, 51.2, 60.0])),
                                    bev_res=int(rng.choice([64, 128, 256])), z_max=3.0, ground_z=-1.2)
            ppt, grid, window, cull_shift = int(rng.choice([2, 4])), int(rng.choice([0, 1, 3, 29, 148])), int(rng.choice([0, 0, 16, 60])), int(rng.choice([-1, -1, 1, 3]))
            if cull_shift == 1 and (ppt == 2 or (params is not None and params.bev_res > 200)):
                cull_shift = 2  # (cull cells of two BEV cells: the id and count tables of a 200 x 200 grid do not fit beside 32 warp blocks)
            for k, v in (("ppt", ppt), ("grid", grid), ("window", window), ("cull_shift", cull_shift)):
                _capi.set_option(k, v)
            _capi.set_option("standard", int(rng.integers(0, 2)))
            check_fused(engine, s, params=params, config=10)
    finally:
        for k, v in (("ppt", _capi.DEFAULT_FUSED_PPT), ("grid", 0), ("window", 0), ("cull_shift", -1), ("standard", 1), ("config", _capi.DEFAULT_FUSED_CONFIG)):
            _capi.set_option(k, v)


@pytest.mark.parametrize("config", [10, 7])
def test_fused_full_size_batch_properties(engine, config):
    """BASELINE config-3 batch at the benchmark's size (592 samples, 205.5 M points): size-independent properties, replica
    equality (bit-reproducibility under different scheduling), idempotence, and the oracle on sampled samples."""
    import torch
    p = GeomParams()
    _capi.set_option("config", config)
    uniq = [make_sample(100 + i, n_sweeps=10, n_boxes=60) for i in range(8)]
    hb_u = pack_batch(uniq)
    hb = tile_batch(hb_u, 74)
    assert hb.n_samples == 592
    db = engine.upload(hb)
    out = engine.run_fused(db, params=p); torch.cuda.synchronize()
    got = out.to_host(with_bev=False)
    cnt = out.bev_ci[..., 0]
    st = got["stats"]
    assert (st[:, 0] == 347200).all() and (st[:, 3] + st[:, 4] == st[:, 2]).all()
    assert torch.equal(cnt.sum(dim=(1, 2)).cpu(), torch.from_numpy(st[:, 2].astype(np.int64)).to(torch.int64))
    nb = hb_u.n_boxes
    for k in ("box_count", "box_nearest", "box_centroid", "proj_visible", "proj_extent"):
        a = got[k].reshape((74, nb) + got[k].shape[1:])
        assert (a == a[0:1]).all(), k                       # every replica bit-identical
    assert (st.reshape(74, 8, 16) == st.reshape(74, 8, 16)[0:1]).all()
    assert torch.equal(out.bev_ci[:8], out.bev_ci[8 * 73: 8 * 74]) and torch.equal(out.bev_height[:8], out.bev_height[8 * 37: 8 * 38])
    out2 = engine.run_fused(db, params=p); torch.cuda.synchronize()   # idempotent: outputs are fully rewritten
    assert torch.equal(out.bev_ci, out2.bev_ci) and torch.equal(out.box_centroid, out2.box_centroid)
    for i in (3, 6):
        ref = OB.oracle_fused(hb_u, i, p)
        b0, b1 = hb_u.sample_box_off[i], hb_u.sample_box_off[i + 1]
        assert np.array_equal(got["box_count"][b0:b1], ref["box_count"]) and np.array_equal(got["box_centroid"][b0:b1], ref["box_centroid"])
        assert np.array_equal(out.bev_ci[i, ..., 0].cpu().numpy().view(np.uint32), ref["bev_count"])
        assert np.array_equal(out.bev_height[i].cpu().numpy(), ref["bev_height"])


# ------------------------------------------------------------------------------------------------ keyframe path vs the reference
@pytest.mark.parametrize("name", ["mock", "edge", "synth", "empty", "flatobj"])
def test_keyframe_filter_split_and_bev_match_reference(engine, golden_dir, name):
    from msc_geom.lidar_agent import LiDARAgent
    g = np.load(os.path.join(golden_dir, f"keyframe_{name}.npz"))
    agent = LiDARAgent(object(), "m", "n", engine=engine)
    kept = agent._preprocess_point_cloud(g["points"])
    ground, obj = agent._segment_ground(kept)
    assert np.array_equal(kept, g["kept"]) and np.array_equal(ground, g["ground"]) and np.array_equal(obj, g["object"])
    bev = agent._generate_multi_layer_bev(ground, obj)
    for k in ("semantic", "height", "density"):
        assert bev[k].dtype == g[k].dtype and np.array_equal(bev[k], g[k]), (name, k)


def test_segment_ground_alone_keeps_every_row(engine):
    """_segment_ground on an arbitrary array (lidar_agent.py:128-130): no gate, NaN z goes to `object` like pc[~mask]."""
    from msc_geom.lidar_agent import LiDARAgent
    rng = np.random.default_rng(9)
    pc = rng.normal(0, 40, (5000, 4)).astype(np.float32)
    pc[::50, 2] = np.nan; pc[1::50, 0] = np.inf; pc[2::50, 2] = -1.4; pc[3::50, 2] = np.float32(-1.4000001)
    agent = LiDARAgent(object(), "m", "n", engine=engine)
    for thr in (-1.4, 0.25):
        ground, obj = agent._segment_ground(pc, thr)
        m = pc[:, 2] < thr
        assert np.array_equal(ground, pc[m], equal_nan=True) and np.array_equal(obj, pc[~m], equal_nan=True)


def test_keyframe_strided_devkit_view(engine, golden_dir):
    g = np.load(os.path.join(golden_dir, "keyframe_synth.npz"))
    raw = np.zeros((g["points"].shape[0], 5), np.float32)
    raw[:, :4] = g["points"]; raw[:, 4] = 7.0
    view = raw[:, :4]                                  # 20-byte pitch, like nuscenes_loader.py:152-155
    rows, pitch = ops._raw_rows(view)
    assert pitch == 5 and rows.__array_interface__["data"][0] == raw.__array_interface__["data"][0]  # no host repack
    kept, ground, obj = ops.keyframe_filter_split(engine, view, GeomParams(bev_res=800))
    assert np.array_equal(kept, g["kept"]) and np.array_equal(obj, g["object"])


def test_lidar_agent_process_matches_reference(engine, golden_dir, golden_json):
    from msc_geom.lidar_agent import LiDARAgent
    from msc_geom.nuscenes_loader import create_loader
    np.random.seed(0)
    sample = create_loader(None, use_mock=True).get_sample_by_scene_index(0, 0)
    agent = LiDARAgent(object(), "m", "LiDARAgent", engine=engine, llm=lambda *a, **k: "STUB",
                       cluster_classifier=lambda images, mosaic, batch: [{"category": "car", "confidence": 0.9} for _ in batch])
    out = agent.process(sample["point_cloud"])
    ref = golden_json["process_mock"]
    assert out["bev_metadata"] == ref["bev_metadata"] and out["structured_report"] == ref["structured_report"]
    assert out["observations"] == ref["observations"] and out["agent"] == "LiDARAgent" and out["modality"] == "lidar"
    sf = dict(out["semantic_features"]); near = sf.pop("nearest_object")
    rf = dict(ref["semantic_features"]); rd = rf.pop("nearest_object_distance")
    assert sf == rf and ((near is None and rd is None) or float(near.distance) == rd)
    assert json.loads(json.dumps(out["detected_objects"])) == ref["detected_objects"]


def test_detect_objects_hands_cluster_images_to_the_classifier(engine, golden_dir):
    """lidar_agent.py:198-224: the classifier gets, per batch of ten, the clusters' 4-view images (here rastered in ONE launch for all
    clusters) and their metadata; the images equal the per-cluster method's and the mosaic is the reference's batch sheet."""
    from msc_geom.lidar_agent import LiDARAgent, cluster_mosaic
    g = np.load(os.path.join(golden_dir, "clusters_synth.npz"))
    seen = []

    def classifier(images, mosaic, meta):
        seen.append((images, mosaic, meta))
        return [{"category": "car", "confidence": 0.9} for _ in meta]
    agent = LiDARAgent(object(), "m", "n", engine=engine, cluster_classifier=classifier)
    objs = agent._detect_objects_3d(g["object"])
    n = len(g["num_points"])
    assert len(objs) == n and sum(len(b[2]) for b in seen) == n and all(len(b[0]) == len(b[2]) <= 10 for b in seen)
    assert [m["index"] for b in seen for m in b[2]] == list(range(n))
    labels = g["labels"]
    order = [int(l) for l in set(labels.tolist()) if l != -1 and (labels == l).sum() >= 5]
    first = agent._generate_cluster_visualization(g["object"][labels == order[0]])
    assert seen[0][0][0].shape == (512, 512, 3) and np.array_equal(seen[0][0][0], first)
    assert np.array_equal(seen[0][1], cluster_mosaic(seen[0][0]))


def test_scenegraph_process_returns_the_reference_keys(engine, golden_dir):
    from msc_geom.scenegraph_agent import SceneGraphAgent
    gold = json.load(open(os.path.join(golden_dir, "agent_golden.json")))
    anns = gold["scenegraph_fallback"]["annotations"]
    agent = SceneGraphAgent(object(), "m", "SceneGraphAgent", engine=engine)
    out, ref = agent.process(anns), gold["scenegraph_fallback"]["result"]
    assert {k: out[k] for k in ref} == ref                               # agent, modality, scene_graph (local fallback), observations
    assert [o["id"] for o in out["evidence"]["objects"]] == ["obj_0", "obj_1"]   # additive key: the GPU-computed table
    full = gold["scenegraph_llm"]["result"]
    prompts = []
    agent.scene_graph_fn = lambda prompt: (prompts.append(prompt), full["scene_graph"])[1]   # the injected LLM half
    out2 = agent.process(anns)
    assert {k: out2[k] for k in full} == full and prompts[0] == agent.scene_graph_prompt(anns)

    def failing(prompt):
        raise RuntimeError("LLM down")
    agent.scene_graph_fn = failing
    assert agent.process(anns)["scene_graph"] == ref["scene_graph"]      # the reference's except-branch (:378-421)


def test_cluster_metadata_matches_reference(engine, golden_dir):
    from msc_geom.lidar_agent import LiDARAgent
    g = np.load(os.path.join(golden_dir, "clusters_synth.npz"))
    agent = LiDARAgent(object(), "m", "n", engine=engine)
    labels = g["labels"]
    order = [int(l) for l in set(labels.tolist()) if l != -1 and (labels == l).sum() >= 5]
    meta = agent._cluster_metadata(g["object"], labels, order)
    assert len(meta) == len(g["num_points"])
    for i, m in enumerate(meta):
        assert np.array_equal(m["center"], g["center"][i]) and np.array_equal(m["dimensions"], g["dimensions"][i])
        assert m["distance"] == g["distance"][i] and m["num_points"] == g["num_points"][i] and m["direction"] == str(g["direction"][i])


def test_dbscan_rejects_non_finite_and_merges_long_chains(engine):
    """NaN / inf input raises like scikit-learn's check_array; a long chain of core points (the worst case for hooking) is one cluster."""
    from sklearn.cluster import DBSCAN
    X = np.random.default_rng(1).normal(0, 1, (50, 3))
    X[7, 1] = np.nan
    with pytest.raises(ValueError):
        ops.dbscan(engine, X)
    X[7, 1] = np.inf
    with pytest.raises(ValueError):
        ops.dbscan(engine, X)
    t = np.arange(6000, dtype=np.float64) * 0.04            # a 240 m line, every point a core point, one component
    chain = np.stack([t, 0.01 * np.sin(t), np.zeros_like(t)], 1)
    got = ops.dbscan(engine, chain, 0.5, 10)
    assert np.array_equal(got, DBSCAN(eps=0.5, min_samples=10).fit(chain).labels_) and got.max() == 0


def _dbscan_cases():
    rng = np.random.default_rng(4)
    blobs = np.concatenate([rng.normal(c, s, (m, 3)) for c, s, m in [((0, 0, 0), 0.3, 400), ((2.2, 0, 0), 0.35, 300), ((10, 5, 1), 0.15, 60),
                                                                      ((-6, -6, 0), 1.5, 800), ((4, -9, 0.5), 0.05, 12)]]).astype(np.float32)
    lattice = np.stack(np.meshgrid(np.arange(12) * 0.5, np.arange(12) * 0.5, np.arange(3) * 0.5), -1).reshape(-1, 3).astype(np.float32)  # distances exactly eps
    dup = np.repeat(rng.uniform(-3, 3, (40, 3)).astype(np.float32), 11, 0)                                                              # exact duplicates
    sparse = rng.uniform(-40, 40, (3000, 3)).astype(np.float32)                                                                        # all noise
    return {"blobs": blobs, "lattice": lattice, "duplicates": dup, "noise": sparse, "tiny": blobs[:7]}


@pytest.mark.parametrize("case", ["blobs", "lattice", "duplicates", "noise", "tiny", "synth_k1", "synth_k10"])
def test_dbscan_labels_equal_sklearn(engine, case):
    """SURVEY.md section 8(f) rank 2: device DBSCAN must reproduce sklearn.cluster.DBSCAN(eps=0.5, min_samples=10) label for label
    (the reference's call, lidar_agent.py:148-153), on the [EXT]-aggregated object points too."""
    from sklearn.cluster import DBSCAN
    if case.startswith("synth"):
        s = make_sample(7, n_sweeps=1 if case.endswith("k1") else 10)
        xyzi, _ = ops.aggregate_sweeps(engine, [(sw["points_raw"], sw["ref_from_sensor"], sw["time_lag"]) for sw in s["lidar_sweeps"]])
        _, _, obj = ops.keyframe_filter_split(engine, xyzi, GeomParams(bev_res=800))
        X = obj[:, :3]
        if case.endswith("k10"):
            X = X[np.abs(X[:, 0]) < 25]          # keep the CPU side of the comparison to a few seconds
    else:
        X = _dbscan_cases()[case]
    ref = DBSCAN(eps=0.5, min_samples=10).fit(X).labels_
    got = ops.dbscan(engine, X, 0.5, 10)
    assert got.dtype == ref.dtype and np.array_equal(got, ref), (case, int((got != ref).sum()), int(ref.max()) + 1)
    if case == "blobs":
        assert ref.max() >= 2 and (ref == -1).any()
        ref2 = DBSCAN(eps=0.3, min_samples=4).fit(X).labels_
        assert np.array_equal(ops.dbscan(engine, X, 0.3, 4), ref2)
        pc4 = np.concatenate([X, np.ones((len(X), 1), np.float32)], 1)   # (N,4) rows, like object_points[:, :3] of an (N,4) cloud
        assert np.array_equal(ops.dbscan(engine, pc4[:, :3], 0.5, 10), ref)


def test_cluster_views_match_reference(engine, golden_dir):
    """Cluster 4-view raster (lidar_agent.py:241-356) and mosaic (:366-386): exact uint8 equality with the reference's images."""
    from msc_geom.lidar_agent import LiDARAgent, cluster_mosaic
    g = np.load(os.path.join(golden_dir, "cluster_views.npz"))
    agent = LiDARAgent(object(), "m", "n", engine=engine)
    n = int(g["n"])
    singles = [agent._generate_cluster_visualization(g[f"pts_{i}"]) for i in range(n)]
    for i in range(n):
        assert singles[i].dtype == np.uint8 and np.array_equal(singles[i], g[f"img_{i}"]), i
    # all clusters of one cloud in a single launch
    pts = np.concatenate([g[f"pts_{i}"] for i in range(n)])
    labels = np.concatenate([np.full(len(g[f"pts_{i}"]), i) for i in range(n)])
    perm = np.random.default_rng(0).permutation(len(pts))          # interleave clusters; order inside a cluster must survive
    perm = perm[np.argsort(labels[perm] * 0, kind="stable")]
    inv = np.argsort(perm, kind="stable")
    keep_order = np.argsort(np.stack([labels, np.arange(len(pts))], 1)[:, 0], kind="stable")
    batch = agent._cluster_visualizations(pts, labels, list(range(n)))
    for i in range(n):
        assert np.array_equal(batch[i], g[f"img_{i}"]), i
    assert np.array_equal(cluster_mosaic(singles[:5]), g["mosaic"])


@pytest.mark.parametrize("case", ["mock", "docs_scene_1", "docs_scene_2", "docs_scene_3", "edge"])
def test_scenegraph_agent_matches_reference(engine, golden_json, case):
    from msc_geom.scenegraph_agent import SceneGraphAgent
    g = golden_json["annotations"][case]
    agent = SceneGraphAgent(object(), "m", "SceneGraphAgent", engine=engine)
    objs = agent._parse_annotations(g["annotations"])
    assert len(objs) == len(g["parsed"])
    for a, b in zip(objs, g["parsed"]):
        for k in ("id", "category", "direction", "state", "visibility", "attributes", "position"):
            assert a[k] == b[k], (k, a, b)
        # the reference squares with libm pow (1 ulp from the exact product for some inputs): 1e-5 relative is the bar, 2 ulp is what we hold
        assert abs(float(a["distance"]) - b["distance"]) <= 2 * np.spacing(b["distance"]) or (np.isnan(a["distance"]) and np.isnan(b["distance"]))
    assert {k: [o["id"] for o in v] for k, v in agent._categorize_objects(objs).items()} == g["categorized"]
    assert {k: [o["id"] for o in v] for k, v in agent._build_spatial_zones(objs).items()} == g["zones"]
    if g["describe"] is not None:
        rc = agent.region_counts(g["annotations"])
        for name in ("front", "back", "left", "right"):
            assert f"- {name.capitalize()} region: {rc[name]} objects" in g["describe"]


def test_cloud_stats_match_reference(engine, golden_dir, golden_json):
    pts = np.load(os.path.join(golden_dir, "keyframe_mock.npz"))["points"]
    mn, mx, mean = ops.cloud_stats(engine, pts)
    assert np.array_equal(mn, pts[:, :3].min(0)) and np.array_equal(mx, pts[:, :3].max(0))
    text = golden_json["describe_point_cloud_mock"]
    assert f"X range: [{mn[0]:.1f}, {mx[0]:.1f}] m" in text and f"Z range: [{mn[2]:.1f}, {mx[2]:.1f}] m" in text
    assert f"Average distance from ego: {mean:.1f} m" in text
    assert abs(mean - OB.oracle_cloud_stats(pts)[1] / len(pts)) <= 1e-12 * mean  # f64 accumulation, order differs


# ------------------------------------------------------------------------------------------------ [EXT] tables vs the oracle
def test_aggregate_sweeps_bit_exact(engine):
    s = make_sample(80, n_sweeps=5)
    s["lidar_sweeps"][2]["points_raw"] = s["lidar_sweeps"][2]["points_raw"][:777]
    hb = pack_batch([s])
    ref_xyzi, ref_t = OB.oracle_aggregate(hb, 0)
    xyzi, t = ops.aggregate_sweeps(engine, [(sw["points_raw"], sw["ref_from_sensor"], sw["time_lag"]) for sw in s["lidar_sweeps"]])
    assert np.array_equal(xyzi, ref_xyzi) and np.array_equal(t, ref_t)


def test_projection_and_relations_match_oracle(engine):
    from msc_geom.camera_agent import projection_evidence
    from msc_geom.scenegraph_agent import SceneGraphAgent
    s = make_sample(81, n_sweeps=1, n_boxes=200)
    boxes = boxes_from_annotations(s["annotations"])
    pose = np.stack([c["ego_pose"] for c in s["cameras"]]); cal = np.stack([c["calib"] for c in s["cameras"]])
    K = np.stack([c["intrinsic"].reshape(9) for c in s["cameras"]])
    vis, ext = ops.project_boxes(engine, boxes, pose, cal, K)
    rv, re = OB.oracle_project(boxes, pose, cal, K)
    assert np.array_equal(vis, rv) and np.array_equal(ext, re) and vis.sum() > 10
    ev = projection_evidence(engine, s)
    assert sum(v["visible_objects"] for v in ev.values()) == int(vis.sum())
    agent = SceneGraphAgent(object(), "m", "n", engine=engine)
    for ego in (None, s["ego_pose"]):
        rel = agent.relations(s["annotations"], ego)
        ref = OB.oracle_relations(OB.oracle_footprints(boxes, ego))
        assert np.array_equal(rel["rect"], OB.oracle_footprints(boxes, ego))
        assert np.array_equal(rel["dist"], ref["dist"]) and np.array_equal(rel["category"], ref["category"]) and np.array_equal(rel["overlap"], ref["overlap"])
        # bearing goes through atan2 (CUDA vs glibc differ in the last ulps): 1e-5 relative, as north_star states
        assert np.allclose(rel["bearing"], ref["bearing"], rtol=1e-5, atol=1e-4)
    assert rel["overlap"].sum() > 200  # diagonal + some genuinely overlapping footprints


def test_upload_tiled_equals_host_tiling(engine):
    import torch
    from msc_geom.layout import truncate_batch
    hb_u = pack_batch([make_sample(130 + i, n_sweeps=2, n_boxes=4 + i) for i in range(3)])
    for reps, keep in ((3, None), (3, 7), (1, 2)):
        want = tile_batch(hb_u, reps)
        if keep is not None:
            want = truncate_batch(want, keep)
        got = engine.upload_tiled(hb_u, reps, keep)
        assert got.host.n_samples == want.n_samples and got.host.n_points == want.n_points
        for k in ("sample_sweep_off", "sweep_start", "sweep_count", "sweep_pose", "sample_box_off", "boxes", "cam_K"):
            assert np.array_equal(got.tensors[k].cpu().numpy().view(getattr(want, k).dtype).reshape(getattr(want, k).shape), getattr(want, k)), k
        assert np.array_equal(got.tensors["points"].cpu().numpy(), want.points, equal_nan=True)
        a = engine.run_fused(got); torch.cuda.synchronize(); a = a.to_host()
        b = engine.run_fused(engine.upload(want)); torch.cuda.synchronize(); b = b.to_host()
        for k in ("box_count", "bev_count", "stats", "box_centroid"):
            assert np.array_equal(a[k], b[k]), k


def test_batched_relation_tables_match_oracle(engine):
    import torch
    samples = [make_sample(120 + i, n_sweeps=1, n_boxes=nb) for i, nb in enumerate([7, 0, 200, 33])]
    hb = pack_batch(samples)
    db = engine.upload(hb)
    rel, pair_off = engine.alloc_relations(hb)
    engine.run_relations(db, rel); torch.cuda.synchronize()
    for i, s in enumerate(samples):
        n = len(s["annotations"])
        if n == 0:
            continue
        ref = OB.oracle_relations(OB.oracle_footprints(boxes_from_annotations(s["annotations"]), None))
        sl = slice(int(pair_off[i]), int(pair_off[i]) + n * n)
        assert np.array_equal(rel["dist"][sl].cpu().numpy().reshape(n, n), ref["dist"])
        assert np.array_equal(rel["category"][sl].cpu().numpy().reshape(n, n), ref["category"])
        assert np.array_equal(rel["overlap"][sl].cpu().numpy().reshape(n, n), ref["overlap"])
        assert np.allclose(rel["bearing"][sl].cpu().numpy().reshape(n, n), ref["bearing"], rtol=1e-5, atol=1e-4)


def test_patch_reference_style_classes(engine, golden_dir):
    """integration.patch_reference() on stand-ins shaped like the reference classes (same attribute names)."""
    from msc_geom import integration

    class RefLidar:  # attributes of lidar_agent.py:40-49
        def __init__(self):
            self.bev_resolution, self.bev_range, self.dbscan_eps, self.dbscan_min_samples = 800, 50, 0.5, 10

    class RefScene:
        def __init__(self):
            self.spatial_zones = {}

    integration.patch_reference(RefLidar, RefScene, engine)
    g = np.load(os.path.join(golden_dir, "keyframe_mock.npz"))
    a = RefLidar()
    kept = a._preprocess_point_cloud(g["points"])
    ground, obj = a._segment_ground(kept)
    assert np.array_equal(kept, g["kept"]) and np.array_equal(a._generate_multi_layer_bev(ground, obj)["semantic"], g["semantic"])
    sg = RefScene()
    sg.spatial_zones = {z: None for z in ("front_close", "front_medium", "front_far", "left_close", "left_medium", "right_close", "right_medium",
                                          "back_close", "back_medium")}
    objs = sg._parse_annotations([{"category_name": "vehicle.car", "translation": [10.0, 2.0, 0.5], "velocity": [3.0, 0.5]}])
    assert objs[0]["direction"] == "right" and float(objs[0]["distance"]) == 10.198039027185569
    assert [o["id"] for o in sg._build_spatial_zones(objs)["right_medium"]] == ["obj_0"]


def test_staged_files_batch_runs_from_pinned_memory(engine, tmp_path):
    """SURVEY 8(f) rank 3: sweeps read from .pcd.bin files straight into a pinned batch buffer give the same evidence."""
    import torch
    from msc_geom import io as mio
    samples = [make_sample(110 + i, n_sweeps=2, n_boxes=6) for i in range(2)]
    fsamples = []
    for i, s in enumerate(samples):
        fs = dict(s); fs["lidar_sweeps"] = []
        for k, sw in enumerate(s["lidar_sweeps"]):
            path = str(tmp_path / f"s{i}_{k}.pcd.bin"); mio.write_pcd_bin(path, sw["points_raw"])
            fs["lidar_sweeps"].append({"path": path, "ref_from_sensor": sw["ref_from_sensor"], "time_lag": sw["time_lag"]})
        fsamples.append(fs)
    hb = mio.stage_batch(fsamples, threads=4)
    assert hb._pinned_holder is not None and hb._pinned_holder.is_pinned()
    a = engine.run_fused(engine.upload(hb, non_blocking=True)); torch.cuda.synchronize(); a = a.to_host()
    b = engine.run_fused(engine.upload(pack_batch(samples))); torch.cuda.synchronize(); b = b.to_host()
    for k in ("box_count", "box_centroid", "bev_count", "bev_isum_q", "bev_height", "stats", "proj_extent"):
        assert np.array_equal(a[k], b[k]), k


def test_bad_arguments_raise(engine):
    from msc_geom.engine import make_params
    s = make_sample(90, n_sweeps=1, n_boxes=4)
    hb = pack_batch([s])
    with pytest.raises(_capi.MscError):
        engine.run_fused(engine.upload(hb), params=GeomParams(range_max=80.0))      # fixed-point centroid range
    with pytest.raises(_capi.MscError):
        engine.run_fused(engine.upload(hb), params=GeomParams(bev_res=201))          # odd grid
    with pytest.raises(_capi.MscError):
        engine.run_fused(engine.upload(hb), params=GeomParams(n_cams=4))             # batch packed for 6 cameras


# ------------------------------------------------------------------------------------------------ camera images (on-disk step)
def _jpeg_bytes(img, **kw):
    import io
    from PIL import Image
    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", **kw)
    return b.getvalue()


@pytest.mark.gpu
def test_jpeg_decode_equals_pil_bit_for_bit(engine):
    """NuScenesLoader._load_camera is np.array(Image.open(path)) (nuscenes_loader.py:136-144): the device reconstruction (integer IDCT,
    fancy chroma upsampling, fixed-point colour conversion) after the host Huffman decode must equal libjpeg-turbo's output exactly --
    every subsampling PIL writes, odd sizes (partial MCUs, one-column chroma planes), optimised Huffman tables, restart intervals,
    grayscale, and a nuScenes-sized frame."""
    import io
    from PIL import Image
    from msc_geom import ops
    rng = np.random.default_rng(11)

    def scene(h, w):  # smooth structure + texture + hard edges, so that every coefficient band and the clamps are exercised
        yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
        base = np.stack([127 + 120 * np.sin(xx / 17.0 + yy / 29.0), 127 + 120 * np.cos(xx / 7.0), 255 * ((xx // 13 + yy // 11) % 2)], -1)
        return np.clip(base + rng.normal(0, 25, (h, w, 3)), 0, 255).astype(np.uint8)
    cases = []
    for (h, w) in ((16, 16), (17, 33), (1, 1), (2, 3), (3, 2), (8, 5), (9, 4), (31, 64), (240, 321)):
        img = scene(h, w)
        for sub in (0, 1, 2):
            for q in (35, 90, 100):
                cases.append(_jpeg_bytes(img, quality=q, subsampling=sub))
        cases.append(_jpeg_bytes(img, quality=75, subsampling=2, optimize=True))
        cases.append(_jpeg_bytes(img[..., 0].copy(), quality=80))  # grayscale
    big = scene(900, 1600)
    cases.append(_jpeg_bytes(big, quality=90, subsampling=2))
    cases.append(_jpeg_bytes(rng.integers(0, 256, (64, 96, 3), dtype=np.uint8), quality=95, subsampling=2))  # noise: large coefficients, clamping
    try:
        cases.append(_jpeg_bytes(big[:200, :301], quality=85, subsampling=2, restart_marker_blocks=7))
        cases.append(_jpeg_bytes(big[:100, :200], quality=85, subsampling=1, restart_marker_rows=1))
    except TypeError:
        pass
    got = ops.decode_jpeg_batch(engine, cases, threads=4)
    for i, (g, data) in enumerate(zip(got, cases)):
        ref = np.array(Image.open(io.BytesIO(data)))
        assert g.shape == ref.shape and g.dtype == np.uint8, (i, g.shape, ref.shape)
        assert np.array_equal(g, ref), (i, ref.shape, int((g != ref).sum()), int(np.abs(g.astype(int) - ref.astype(int)).max()))
    # unsupported flavours are refused, not mis-decoded
    with pytest.raises(_capi.MscError):
        ops.decode_jpeg(engine, _jpeg_bytes(big[:64, :64], progressive=True))
    with pytest.raises(_capi.MscError):
        ops.decode_jpeg(engine, b"not a jpeg at all")


@pytest.mark.gpu
def test_loader_camera_frames_through_the_device_decoder(engine, tmp_path):
    """The loader mirror with an engine attached decodes the camera JPEGs of a written nuScenes tree on the device: same arrays as its
    PIL path (the reference's np.array(Image.open(...)))."""
    import importlib
    import sys
    shim = os.path.join(os.path.dirname(os.path.abspath(__file__)), "devkit_shim")
    sys.path.insert(0, shim)
    try:
        import msc_geom.nuscenes_loader as nl
        nl = importlib.reload(nl)
        from msc_geom import io as mio
        rng = np.random.default_rng(3)
        scenes = []
        for si in range(1):
            sc = []
            for k in range(2):
                s = make_sample(700 + 10 * si + k, n_sweeps=1, n_boxes=3)
                s["images"] = [np.clip(rng.normal(128, 40, (90, 160, 3)), 0, 255).astype(np.uint8) for _ in s["cameras"]]
                s["scene_name"], s["scene_description"] = f"scene-{si:04d}", "jpeg"
                sc.append(s)
            scenes.append(sc)
        mio.write_nuscenes_tree(str(tmp_path), scenes)
        a = nl.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=1)
        b = nl.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=1, engine=engine)
        for tok in a.scene_sample_tokens(a.get_scene_list()[0]["token"]):
            ia, ib = a.load_sample(tok)["images"], b.load_sample(tok)["images"]
            assert len(ia) == len(ib) == 6 and all(x.shape == (90, 160, 3) and np.array_equal(x, y) for x, y in zip(ia, ib))
    finally:
        sys.path.remove(shim)
        for m in [m for m in sys.modules if m == "nuscenes" or m.startswith("nuscenes.")]:
            del sys.modules[m]
        import msc_geom.nuscenes_loader as nl2
        importlib.reload(nl2)
