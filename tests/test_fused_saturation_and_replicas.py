"""The fused path at counter saturation and through its replica stores.

Every check here covers all 16 stats words (stats[13]: bit 0 = a cell count of the shared-memory window reached 65536, bit 31 = more
boxes than the kernel had room for; 14 and 15 are zero).  Crowded-cell samples put 70,000 rows into one BEV cell, so the Q8 intensity
sum of that cell passes 2^32 (70,000 x 65,280) and the box accumulators and centroid carry words take 70,000 members.  They are compared
with the C oracle and with a plain NumPy int64 / float64 evaluation, over the launch shapes, grids (how a sample is split over CTAs),
window sizes and both kernels.  msc_fused_evidence_batch_replicated is checked on one device: its replica arenas must hold the local
tables byte for byte and nothing outside them."""
import dataclasses

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from msc_geom import _capi
from msc_geom.layout import GeomParams, pack_batch
from msc_geom.synthetic import make_sample
from tests import oracle_bridge as OB

IDENT7 = np.array([0, 0, 0, 1, 0, 0, 0.0])
N_CROWD = 70_000
NEAR, FAR = (3.0, 2.0), (40.0, 5.0)   # lower corners of BEV cells (106, 104) and (180, 110) of the default 200-cell, 0.5 m grid
SENTINEL = 0xA5
MSC_ERR_BAD_ARGUMENT = -1   # include/msc_geom.h
OPTION_DEFAULTS = (("ppt", _capi.DEFAULT_FUSED_PPT), ("grid", 0), ("window", 0), ("standard", 1), ("config", _capi.DEFAULT_FUSED_CONFIG))


def restore_options():
    for k, v in OPTION_DEFAULTS:
        _capi.set_option(k, v)


# ------------------------------------------------------------------------------------------------ comparisons
def check_stats(st, ref_stats, ref_count, n_boxes, declared_boxes, p):
    """All 16 stats words of one sample after a call: [:13] equal the oracle's; [13] bit 0 iff an oracle cell count inside the
    window of the call is >= 65536, whatever the partition; bit 31 iff the sample holds more boxes than the kernel had room for
    (stream4.cu sizes its tables for at least 128, fused_stream.cu for the declared maximum); [14] and [15] are zero."""
    assert np.array_equal(st[:13], ref_stats[:13]), (st, ref_stats)
    w = _capi.get_option("last_window")
    lo = (p.bev_res - w) // 2                    # stream4.cu s4_layout / fused_stream.cu stream_layout
    crowded = w > 0 and int(ref_count[lo:lo + w, lo:lo + w].max()) >= 65536
    room = max(declared_boxes, 128) if _capi.get_option("last_config") == 10 else max(declared_boxes, 1)
    want = (1 if crowded else 0) | ((1 << 31) if n_boxes > room else 0)
    assert int(st[13]) == want, ("stats[13]", hex(int(st[13])), hex(want), "window", w)
    assert st[14] == 0 and st[15] == 0, st


def check_against_oracle(hb, got, refs, p, declared_boxes):
    """Every output of every sample against the oracle (`refs[i]` = OB.oracle_fused(hb, i, p)); box entries beyond the kernel's room
    are not compared (their contents are unspecified)."""
    room = max(declared_boxes, 128) if _capi.get_option("last_config") == 10 else max(declared_boxes, 1)
    for i, ref in enumerate(refs):
        b0, b1 = int(hb.sample_box_off[i]), int(hb.sample_box_off[i + 1])
        n_ok = min(room, b1 - b0)
        for k in ("box_count", "box_nearest", "box_centroid"):
            assert np.array_equal(got[k][b0:b0 + n_ok], ref[k][:n_ok]), (i, k)
        for k in ("proj_visible", "proj_extent"):
            assert np.array_equal(got[k][b0:b1], ref[k]), (i, k)
        for k in ("bev_count", "bev_isum_q", "bev_height"):
            assert np.array_equal(got[k][i], ref[k]), (i, k, int((got[k][i] != ref[k]).sum()))
        check_stats(got["stats"][i], ref["stats"], ref["bev_count"], b1 - b0, declared_boxes, p)


def numpy_reference(pts, boxes, p):
    """Plain evaluation of one identity-pose sample (its sweep transform is exact): the filters of lidar_agent.py:106-110 and the BEV
    cell of :547-552 in float32, per-cell count / max height / Q8 intensity sum in int64 (the sum then taken mod 2^32), axis-aligned box
    membership and centroids in float64."""
    f = np.float32
    x, y, z, inten = (np.ascontiguousarray(pts[:, k], np.float32) for k in range(4))
    rc = f(p.remove_close_radius)
    close = (np.abs(x) < rc) & (np.abs(y) < rc)
    s2 = x * x + y * y
    d = np.sqrt(s2)
    keep = ~close & (d > f(p.range_min)) & (d < f(p.range_max)) & (z < f(p.z_max)) & (z > f(p.z_min))
    r, res = f(p.bev_range), p.bev_res

    def cell(c):
        return np.clip(np.trunc((c + r) / (f(2.0) * r) * f(res)), 0, res - 1).astype(np.int64)
    lin = cell(y) * res + cell(x)
    q = np.clip(np.rint(inten * f(1 << p.intensity_shift)), 0, 65535).astype(np.int64)
    count = np.zeros(res * res, np.int64)
    isum = np.zeros(res * res, np.int64)
    height = np.zeros(res * res, np.float32)
    np.add.at(count, lin[keep], 1)
    np.add.at(isum, lin[keep], q[keep])
    up = keep & (z > 0)
    np.maximum.at(height, lin[up], z[up])
    n = len(x)
    stats = np.array([n, n - int(close.sum()), int(keep.sum()), int((keep & (z < f(p.ground_z))).sum())], np.int64)
    xyz = np.stack([x, y, z], 1).astype(np.float64)
    box_count, box_nearest, box_centroid = [], [], []
    for b in boxes:
        assert np.array_equal(b[6:10], [1, 0, 0, 0]), "axis-aligned boxes only"
        half = np.array([b[4], b[3], b[5]]) / 2.0          # size is (w, l, h): l along x, w along y
        dist = np.abs(xyz - b[:3]) - half
        near_face = (dist <= 1e-3).all(1) & (np.abs(dist) < 1e-3).any(1) & keep
        assert not near_face.any(), "test data: a point within 1 mm of a box face"
        m = keep & (dist <= 0).all(1)
        box_count.append(int(m.sum()))
        box_nearest.append(np.sqrt(s2[m].min()) if m.any() else np.float32(np.inf))
        box_centroid.append(xyz[m].mean(0) if m.any() else np.zeros(3))
    return {"bev_count": count.reshape(res, res), "bev_isum_q": (isum & 0xFFFFFFFF).reshape(res, res), "bev_isum_full": isum.reshape(res, res),
            "bev_height": height.reshape(res, res), "stats": stats, "box_count": np.array(box_count), "box_nearest": np.array(box_nearest, np.float32),
            "box_centroid": np.array(box_centroid).reshape(-1, 3)}


def check_against_numpy(got, ref, i=0, b0=0):
    for k in ("bev_count", "bev_isum_q", "bev_height"):
        assert np.array_equal(got[k][i].astype(ref[k].dtype), ref[k]), (k, int((got[k][i].astype(ref[k].dtype) != ref[k]).sum()))
    st = got["stats"][i].astype(np.int64)
    assert np.array_equal(st[:4], ref["stats"]) and st[4] == ref["stats"][2] - ref["stats"][3], (st[:5], ref["stats"])
    nb = len(ref["box_count"])
    assert np.array_equal(got["box_count"][b0:b0 + nb].astype(np.int64), ref["box_count"])
    assert np.array_equal(got["box_nearest"][b0:b0 + nb], ref["box_nearest"])
    err = np.abs(got["box_centroid"][b0:b0 + nb].astype(np.float64) - ref["box_centroid"])
    assert (err <= 2.0 ** -17).all(), err.max()        # fixed-point sums at 2^-17 m, then one f32 rounding


# ------------------------------------------------------------------------------------------------ samples
def crowd(rng, corner, n, jitter):
    """n rows in the 0.5 m cell with lower corner `corner`: exactly at (corner + 0.1, z 0.5, intensity 255), or spread inside it (away
    from its edges), with heights in the box (0.1 .. 0.9) or under it (ground, -2.5 .. -1.5) and intensities of 230 .. 260 (Q8
    clamps at 65535; the cell's sum still passes 2^32)."""
    pts = np.empty((n, 4), np.float32)
    if not jitter:
        pts[:] = (corner[0] + 0.1, corner[1] + 0.1, 0.5, 255.0)
        return pts
    pts[:, 0] = corner[0] + rng.uniform(0.02, 0.48, n)
    pts[:, 1] = corner[1] + rng.uniform(0.02, 0.48, n)
    pts[:, 2] = np.where(rng.random(n) < 0.8, rng.uniform(0.1, 0.9, n), rng.uniform(-2.5, -1.5, n))
    pts[:, 3] = rng.uniform(230.0, 260.0, n)
    return pts


def background(rng, n):
    """A cloud over the whole grid and beyond (some rows fail the range, height and remove_close gates), none near the crowded cells."""
    pts = np.stack([rng.uniform(-58, 58, n), rng.uniform(-58, 58, n), rng.uniform(-3.5, 5.5, n), rng.uniform(0, 255, n)], 1)
    pts[: n // 50, :2] = rng.uniform(-1.2, 1.2, (n // 50, 2))
    away = np.ones(n, bool)
    for cx, cy in (NEAR, FAR):
        away &= ~((np.abs(pts[:, 0] - cx - 0.25) < 1.5) & (np.abs(pts[:, 1] - cy - 0.25) < 1.5))
    return pts[away].astype(np.float32)


def crowded_sample(kind, seed=17):
    rng = np.random.default_rng(seed)
    if kind == "near":
        pts = crowd(rng, NEAR, N_CROWD, False)
    elif kind == "far":
        pts = crowd(rng, FAR, N_CROWD, False)
    elif kind == "jittered":
        pts = np.concatenate([crowd(rng, NEAR, N_CROWD, True), crowd(rng, FAR, N_CROWD, True)])
    else:  # "cloud": both crowded cells shuffled into a background cloud
        pts = np.concatenate([crowd(rng, NEAR, N_CROWD, True), crowd(rng, FAR, N_CROWD, True), background(rng, 30_000)])
        pts = pts[rng.permutation(len(pts))]
    # an axis-aligned 1 m box around each crowded cell: same-address box atomics, centroid carry words at 70k members
    anns = [{"category_name": "vehicle.car", "translation": [cx + 0.25, cy + 0.25, 0.5], "size": [1.0, 1.0, 1.0], "rotation": [1.0, 0.0, 0.0, 0.0]}
            for cx, cy in (NEAR, FAR)]
    return {"point_cloud": pts, "annotations": anns, "ego_pose": IDENT7, "lidar_calib": IDENT7}


def run(engine, db, p):
    """One call into result tables pre-filled with the sentinel and BEV layers pre-filled with garbage (the kernels write every
    table entry and zero-fill the layers themselves)."""
    out = engine.alloc_result(db.host, p)
    out.table_arena.fill_(SENTINEL)
    out.bev_ci.fill_(-1)
    out.bev_height.fill_(7.0)
    engine.run_fused(db, out, params=p)
    torch.cuda.synchronize()
    return out


# ------------------------------------------------------------------------------------------------ crowded cells
@pytest.mark.parametrize("kind", ["near", "far", "jittered", "cloud"])
def test_fused_crowded_cell_saturation(engine, kind):
    """70,000 rows in one cell near the sensor (inside every default window) and / or one periphery cell: the cell's Q8 intensity sum
    wraps mod 2^32 in the window's u32 words, the periphery's 64-bit reductions and a straddling part's 64-bit merge alike, and
    stats[13] bit 0 is set for a window cell whether the sample runs on one CTA or is split over many."""
    s = crowded_sample(kind)
    p = GeomParams()
    hb = pack_batch([s])
    db = engine.upload(hb)
    refs = [OB.oracle_fused(hb, 0, p)]
    npref = numpy_reference(s["point_cloud"], hb.boxes, p)
    assert np.array_equal(refs[0]["bev_count"], npref["bev_count"]) and np.array_equal(refs[0]["bev_isum_q"], npref["bev_isum_q"])
    assert npref["bev_count"].max() >= N_CROWD and npref["bev_isum_full"].max() >= 2 ** 32 and npref["box_count"].max() >= 50_000
    try:
        for ppt in (2, 4):
            for grid in (1, 2, 3, 7, 37, 148, 0):
                for window in (0, 16, 2):    # (window 2 leaves no window at all on a 200-cell grid: win_lo must be even)
                    for std in (1, 0):
                        for k, v in (("config", 10), ("ppt", ppt), ("grid", grid), ("window", window), ("standard", std)):
                            _capi.set_option(k, v)
                        got = run(engine, db, p).to_host()
                        ctx = dict(ppt=ppt, grid=grid, window=window, standard=std, last_window=_capi.get_option("last_window"))
                        assert _capi.get_option("last_config") == 10 and (grid == 0 or _capi.get_option("last_grid") == grid), ctx
                        if window == 16:
                            assert _capi.get_option("last_window") == 16, ctx
                        try:
                            check_against_oracle(hb, got, refs, p, hb.max_boxes_per_sample)
                            check_against_numpy(got, npref)
                        except AssertionError as e:
                            raise AssertionError(f"{ctx}: {e}") from e
        _capi.set_option("grid", 0)
        _capi.set_option("ppt", _capi.DEFAULT_FUSED_PPT)
        for window in (0, 16, 2):
            _capi.set_option("config", 7)
            _capi.set_option("window", window)
            got = run(engine, db, p).to_host()
            assert _capi.get_option("last_config") == 7
            check_against_oracle(hb, got, refs, p, hb.max_boxes_per_sample)
            check_against_numpy(got, npref)
    finally:
        restore_options()


# ------------------------------------------------------------------------------------------------ replicas on one device
def replica_batch(n_cams):
    """A ragged batch: empty samples at both ends, ordinary samples that a small grid splits over CTAs, one with 140 boxes (more than
    any layout has room for once the declared maximum is cut to 5: stats[13] bit 31) and the crowded near cell (bit 0)."""
    def cams(s):
        if n_cams == 0:
            s["cameras"] = []
        elif n_cams == 8:
            s["cameras"] = s["cameras"] + [dict(s["cameras"][1], channel="CAM_X1"), dict(s["cameras"][4], channel="CAM_X2")]
        return s
    def empty():
        s = make_sample(32, n_sweeps=1, n_boxes=3)
        s["lidar_sweeps"] = [dict(s["lidar_sweeps"][0], points_raw=s["lidar_sweeps"][0]["points_raw"][:0])]
        return s
    samples = [cams(empty()), cams(make_sample(210, n_sweeps=3, n_boxes=20)), cams(make_sample(211, n_sweeps=1, n_boxes=140)),
               crowded_sample("near"), cams(make_sample(212, n_sweeps=2, n_boxes=0)), cams(empty())]
    hb = pack_batch(samples, n_cams=n_cams)
    return dataclasses.replace(hb, max_boxes_per_sample=5)


def split_samples(hb, grid):
    """The samples of hb that the static partition of stream4.cu (CTA b of G owns warp tiles [b T / G, (b + 1) T / G), 128-row tiles
    per sweep) splits over CTAs."""
    tiles = (hb.sweep_count.astype(np.int64) + 127) // 128
    per_sample = np.array([tiles[hb.sample_sweep_off[i]:hb.sample_sweep_off[i + 1]].sum() for i in range(hb.n_samples)])
    off = np.concatenate([[0], np.cumsum(per_sample)])
    T = int(off[-1])
    return {i for b in range(1, grid) for i in range(hb.n_samples) if off[i] < b * T // grid < off[i + 1]}


def sentinel_arena(n, device):
    return torch.full((n,), SENTINEL, dtype=torch.uint8, device=device)


def table_mask(engine, hb, n_cams):
    """Bytes of an arena that the six tables occupy (the gaps between them are alignment padding)."""
    lay, size = engine.table_layout(hb.n_samples, hb.n_boxes, n_cams)
    m = np.zeros(size, bool)
    for o, n in lay.values():
        m[o:o + n] = True
    return torch.from_numpy(m), size


@pytest.mark.parametrize("n_cams", [6, 0, 8])
def test_fused_replicated_tables_on_one_device(engine, n_cams):
    """msc_fused_evidence_batch_replicated with 1, 3 and 8 replica arenas (local tensors here; peers' memory in a multi-GPU job): every
    replica holds the local tables byte for byte, the local tables equal a plain call's, every output equals the oracle, and no byte of
    a replica arena outside the tables (alignment gaps, the padded tail) is touched."""
    p = GeomParams(n_cams=n_cams)
    hb = replica_batch(n_cams)
    db = engine.upload(hb)
    refs = [OB.oracle_fused(hb, i, p) for i in range(hb.n_samples)]
    mask, size = table_mask(engine, hb, n_cams)
    mask = mask.to(engine.device)
    try:
        _capi.set_option("config", 10)
        for grid in (3, 0):
            _capi.set_option("grid", grid)
            assert grid == 0 or 3 in split_samples(hb, grid)   # the crowded sample is merged from parts
            plain = engine.alloc_result(hb, p, arena=sentinel_arena(size, engine.device))
            engine.run_fused(db, plain, params=p)
            torch.cuda.synchronize()
            check_against_oracle(hb, plain.to_host(), refs, p, hb.max_boxes_per_sample)
            assert (plain.table_arena[~mask] == SENTINEL).all()
            for n_rep in (1, 3, 8):
                local = engine.alloc_result(hb, p, arena=sentinel_arena(size, engine.device))
                arenas = [sentinel_arena(size + 256 * (r + 1) + 13, engine.device) for r in range(n_rep)]   # padded beyond the layout
                engine.run_fused(db, local, params=p, replicas=engine.replica_structs(hb, arenas, p))
                torch.cuda.synchronize()
                got = local.to_host()
                check_against_oracle(hb, got, refs, p, hb.max_boxes_per_sample)
                assert torch.equal(local.table_arena, plain.table_arena), (grid, n_rep)
                for r, a in enumerate(arenas):
                    assert torch.equal(a[:size], local.table_arena), (grid, n_rep, r)
                    assert (a[size:] == SENTINEL).all(), (grid, n_rep, r, "tail")
        assert got["stats"][3][13] & 1 and got["stats"][2][13] >> 31 and not any(got["stats"][i][13] for i in (0, 1, 4, 5))
    finally:
        restore_options()


def test_fused_replicated_refusals(engine):
    """Replicated result tables are refused -- before anything is launched or written -- with fov_keep_mask != 0 (fused_stream.cu
    only), with config 7 forced, and with more than MSC_MAX_REPLICAS replicas."""
    p = GeomParams()
    hb = pack_batch([make_sample(220, n_sweeps=1, n_boxes=6)])
    db = engine.upload(hb)
    _, size = engine.table_layout(hb.n_samples, hb.n_boxes, p.n_cams)
    arenas = [sentinel_arena(size, engine.device) for _ in range(9)]
    try:
        with pytest.raises(_capi.MscError) as e:
            engine.run_fused(db, params=GeomParams(fov_keep_mask=0b1), replicas=engine.replica_structs(hb, arenas[:2], p))
        assert e.value.status == MSC_ERR_BAD_ARGUMENT
        _capi.set_option("config", 7)
        with pytest.raises(_capi.MscError) as e:
            engine.run_fused(db, params=p, replicas=engine.replica_structs(hb, arenas[:2], p))
        assert e.value.status == MSC_ERR_BAD_ARGUMENT
        _capi.set_option("config", 10)
        with pytest.raises(_capi.MscError) as e:   # (run_fused hands the count straight to the C-ABI)
            engine.run_fused(db, params=p, replicas=engine.replica_structs(hb, arenas, p))
        assert e.value.status == MSC_ERR_BAD_ARGUMENT
        torch.cuda.synchronize()
        assert all((a == SENTINEL).all() for a in arenas)
        engine.run_fused(db, params=p, replicas=engine.replica_structs(hb, arenas[:8], p))   # eight is the limit
        torch.cuda.synchronize()
        assert all(torch.equal(a, arenas[0]) for a in arenas[1:8]) and (arenas[8] == SENTINEL).all()
    finally:
        restore_options()
