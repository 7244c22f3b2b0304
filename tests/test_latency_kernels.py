"""Keyframe, aggregation, table and DBSCAN kernels at the sizes and edges where they can go wrong.

Each kernel is held against two references: the C oracle (tests/oracle_bridge.py), bit for bit wherever the repository
defines the arithmetic exactly, and a plain NumPy / Python restatement of the reference's expressions written here, which
does not use the oracle, so a defect that the oracle and a kernel share is caught as well.  Every input is seeded.

What the sizes reach: filter/split and aggregation above 1,048,576 rows (and spans) run the carry loop of kf_scan_kernel
over two or more chunks; cloud stats above 303,104 rows repeat the grid-stride loop; relation tables at n = 1, 15, 17, 33
and batches with max_boxes = 200 or 17 leave partial 16x16 tiles; DBSCAN at n <= 11 is where scikit-learn brute-forces."""
import math

import numpy as np
import pytest

from msc_geom import _capi, ops
from msc_geom.geometry import sqrt_thresholds
from msc_geom.layout import GeomParams, pack_batch
from msc_geom.synthetic import make_sample
from tests import oracle_bridge as OB

pytestmark = pytest.mark.gpu

f32 = np.float32


def _up(v):
    return np.nextafter(f32(v), f32(np.inf))


def _dn(v):
    return np.nextafter(f32(v), f32(-np.inf))


def _same_f32(a, b):
    """Bit-identical float32 arrays, except that any NaN equals any NaN (device and host NaN payloads differ)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def _same_f64(a, b):
    a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a.view(np.uint64)[~na], b.view(np.uint64)[~nb])


# ------------------------------------------------------------------------------------------------ keyframe filter / split
_FS_SIZES = [1, 31, 1023, 1024, 1025, 1 << 20, (1 << 20) + 1, 2_500_000]
_FS_CLOUDS = {}


def _pair_with_square_sum(t):
    """float32 (x, y) whose float32 x*x + y*y is exactly t, or None."""
    x = f32(np.sqrt(float(t) * 0.6))
    for _ in range(64):
        a = x * x
        rem = float(t) - float(a)
        if rem > 0:
            y = f32(np.sqrt(rem))
            for _k in range(8):
                for yy in (y, _dn(y), _up(y)):
                    if a + yy * yy == t:
                        return x, yy
                y = _dn(y)
        x = _up(x)
    return None


def _filter_edge_rows(p):
    """Rows on, and one float either side of, every threshold of lidar_agent.py:106-110 and :128, plus NaN / inf rows."""
    rows = []
    for r in (p.range_min, p.range_max):            # on an axis float32 sqrt(x*x) == |x|
        for v in (_dn(r), f32(r), _up(r)):
            for sx, sy in ((1, 0), (-1, 0), (0, 1), (0, -1)):
                rows.append((sx * v, sy * v, 0.5, 1.0))
    s_lo, s_hi = sqrt_thresholds(p.range_min, p.range_max)   # off the axes: x*x + y*y on the squared limits
    found = 0
    for s in (s_lo, s_hi):
        for t in (_dn(s), f32(s), _up(s)):
            xy = _pair_with_square_sum(t)
            if xy is not None:
                found += 1
                rows.append((xy[0], xy[1], 0.5, 2.0))
                rows.append((-xy[1], xy[0], 0.5, 2.0))
    assert found >= 4
    for z in (p.z_min, p.z_max, p.ground_z):
        for v in (_dn(z), f32(z), _up(z)):
            rows.append((10.0, 3.0, v, 3.0))
    nan, inf = np.nan, np.inf
    rows += [(nan, 5, 0, 4), (5, nan, 0, 4), (5, 5, nan, 4), (inf, 5, 0, 4), (-inf, 5, 0, 4), (5, -inf, 0, 4), (5, 5, inf, 4),
             (5, 5, -inf, 4), (nan, nan, nan, nan), (5, 5, -2.0, nan), (-0.0, 5, -0.0, 4)]
    return np.array(rows, np.float32)


def _filter_cloud(pitch):
    """2.5 M rows with `pitch` floats per row (4 contiguous, 5 the devkit's 20-byte view, 8); edge rows at the start, across
    the 1024-row block edge, across the 1024-block chunk edge of the scan and scattered."""
    if pitch in _FS_CLOUDS:
        return _FS_CLOUDS[pitch]
    rng = np.random.default_rng(100 + pitch)
    n = _FS_SIZES[-1]
    raw = np.full((n, pitch), 7.0, np.float32)
    raw[:, 0:2] = rng.uniform(-60, 60, (n, 2))
    raw[:, 2] = rng.uniform(-4, 6, n)
    raw[:, 3] = rng.uniform(0, 255, n)
    edges = _filter_edge_rows(GeomParams())
    k = len(edges)
    for at in (0, 1024 - k // 2, (1 << 20) - k // 2 - 3, n - k):
        raw[at:at + k, :4] = edges
    idx = rng.choice(n, 20000, replace=False)
    raw[idx, :4] = edges[rng.integers(0, k, idx.size)]
    raw[1 << 20, :4] = (10.0, 3.0, 0.5, 9.0)      # the only row of block 1024 when n = 1,048,577: an object row
    _FS_CLOUDS[pitch] = raw
    return raw


def _np_filter_split(pc, p, split_only):
    """lidar_agent.py:103-132 as boolean masks: float32 sqrt(x**2 + y**2), strict compares (float32 thresholds, NEP 50)."""
    x, y, z = pc[:, 0], pc[:, 1], pc[:, 2]
    if split_only:
        keep = np.ones(len(pc), bool)
    else:
        with np.errstate(invalid="ignore", over="ignore"):
            d = np.sqrt(x ** 2 + y ** 2)
        keep = (d > f32(p.range_min)) & (d < f32(p.range_max)) & (z < f32(p.z_max)) & (z > f32(p.z_min))
    low = z < f32(p.ground_z)
    return keep, keep & low, keep & ~low


@pytest.mark.parametrize("split_only", [False, True], ids=["filter", "split_only"])
@pytest.mark.parametrize("pitch", [4, 5, 8])
def test_keyframe_filter_split_sizes_pitches_thresholds(engine, pitch, split_only):
    p = GeomParams(bev_res=800)
    raw = _filter_cloud(pitch)
    for n in _FS_SIZES:
        view = raw[:n, :4]
        assert ops._raw_rows(view)[1] == (pitch if n > 1 else 4)   # NumPy calls a one-row view contiguous
        kept, ground, obj = ops.keyframe_filter_split(engine, view, p, split_only=split_only)
        pc = np.ascontiguousarray(view)
        mk, mg, mo = _np_filter_split(pc, p, split_only)
        assert _same_f32(kept, pc[mk]) and _same_f32(ground, pc[mg]) and _same_f32(obj, pc[mo]), (n, pitch, split_only)
        if not split_only:
            ki, gi, oi = OB.oracle_keyframe_filter_split(view, p)
            assert np.array_equal(np.flatnonzero(mk), ki) and np.array_equal(np.flatnonzero(mg), gi) and np.array_equal(np.flatnonzero(mo), oi)
        if n >= 1024:
            assert 0 < mg.sum() < mk.sum() and mo.sum() > 0


# ------------------------------------------------------------------------------------------------ keyframe BEV
def _np_bev(ground, obj, res, r=50.0):
    """lidar_agent.py:539-597 before the overlays, in the reference's order: float32 pixel maths, count and 0-initialised
    height over vstack([ground, object]), ground colour, then objects coloured in array order (the last one in a cell wins)."""
    def pix(c):
        return np.clip(((c + f32(r)) / f32(2 * r) * f32(res)).astype(np.int64), 0, res - 1)
    allp = np.vstack([ground[:, :4], obj[:, :4]]).astype(np.float32)
    count = np.zeros((res, res), np.int64)
    height = np.zeros((res, res), np.float32)
    if len(allp):
        x, y = pix(allp[:, 0]), pix(allp[:, 1])
        np.add.at(count, (y, x), 1)
        np.maximum.at(height, (y, x), allp[:, 2])
    sem = np.zeros((res, res, 3), np.uint8)
    if len(ground):
        sem[pix(ground[:, 1]), pix(ground[:, 0])] = (80, 80, 120)
    if len(obj):
        h = obj[:, 2].astype(np.float32)
        if h.max() > h.min():
            hn = (h - h.min()) / (h.max() - h.min())
            lo = hn < 0.5
            g = np.where(lo, f32(255) * (f32(1) - hn * f32(2)), f32(255) * (f32(1) - (hn - f32(0.5)) * f32(2))).astype(np.int64)
        else:
            g = np.full(len(h), int(255 * (1 - (0.5 - 0.5) * 2)), np.int64)
        cell = pix(obj[:, 1]) * res + pix(obj[:, 0])
        last = np.full(res * res, -1, np.int64)
        np.maximum.at(last, cell, np.arange(len(obj)))
        hit = np.flatnonzero(last >= 0)
        flat = sem.reshape(-1, 3)
        flat[hit, 0] = 0
        flat[hit, 1] = g[last[hit]]
        flat[hit, 2] = 255
    return count, height, sem


def _bev_cases(res):
    rng = np.random.default_rng(500 + res)
    r = 50.0
    k = np.unique(np.concatenate([np.arange(0, min(res, 40) + 1), np.linspace(0, res, 25).astype(np.int64), [res - 1, res]]))
    edge = (k.astype(np.float64) * (2 * r) / res - r).astype(np.float32)          # cell edges, rounded to float32
    edge = np.unique(np.concatenate([edge, _up(edge), _dn(edge), [f32(-r), f32(r), _dn(-r), _up(r), _dn(r), _up(-r)]]))
    g = np.zeros((3000 + 2 * edge.size, 4), np.float32)
    g[:3000, :2] = rng.uniform(-55, 55, (3000, 2))
    g[3000:3000 + edge.size, 0] = edge
    g[3000:3000 + edge.size, 1] = rng.choice(edge, edge.size)
    g[3000 + edge.size:, 1] = edge
    g[3000 + edge.size:, 0] = rng.choice(edge, edge.size)
    g[:, 2] = rng.uniform(-3, -1.41, len(g))
    o = np.zeros((3000 + 2 * edge.size, 4), np.float32)
    o[:, :2] = g[rng.permutation(len(g)), :2]
    o[:3000, :2] = rng.uniform(-55, 55, (3000, 2))
    o[:, 2] = rng.uniform(-1.4, 5, len(o))
    o[:, 3] = rng.uniform(0, 100, len(o))
    # points sharing cells, drawn in increasing, decreasing and shuffled height order: the last one in the array colours
    share = []
    for j, order in enumerate(("inc", "dec", "shuf")):
        z = np.linspace(-1.0, 4.5, 7).astype(np.float32)
        z = z if order == "inc" else z[::-1] if order == "dec" else z[rng.permutation(7)]
        xy = rng.uniform(-40, 40, 2).astype(np.float32)
        share.append(np.column_stack([np.repeat(xy[None], 7, 0), z, np.full(7, j, np.float32)]))
    o = np.vstack([o[: len(o) // 2], *share, o[len(o) // 2:]]).astype(np.float32)
    cases = {"mixed": (g, o), "empty_ground": (g[:0], o), "empty_object": (g, o[:0]), "both_empty": (g[:0], o[:0])}
    flat = o.copy(); flat[:, 2] = 1.25
    cases["flat_object_z"] = (g, flat)                                  # hmax == hmin: every object cell is green 255
    neg = o.copy(); neg[:, 2] = -np.abs(neg[:, 2]) - 0.5
    cases["negative_z"] = (g, neg)                                      # the height layer stays 0
    if res in (2, 800):
        c = np.zeros((70000, 4), np.float32)                            # one cell with 70,000 points (beyond 16-bit counts)
        c[:, 0] = 3.0 + rng.uniform(0.25, 0.75, 70000) * (100.0 / res)          # the middle half of one cell
        c[:, 1] = -7.0 + rng.uniform(0.25, 0.75, 70000) * (100.0 / res)
        c[:, 2] = rng.uniform(-1.4, 4.0, 70000)
        cases["crowded_cell"] = (g[:100], np.vstack([o[:500], c, o[500:1000]]))
    return cases


@pytest.mark.parametrize("res", [1, 2, 199, 200, 800, 801], ids=lambda v: f"res{v}")
def test_keyframe_bev_grid_sizes_edges_and_winners(engine, res):
    for name, (ground, obj) in _bev_cases(res).items():
        count, height, sem = ops.keyframe_bev_layers(engine, ground, obj, res=res)
        pts = np.vstack([ground[:, :4], obj[:, :4]]).astype(np.float32) if len(ground) + len(obj) else np.zeros((1, 4), np.float32)
        rc, rh, rs = OB.oracle_keyframe_bev(pts, np.arange(len(ground)), len(ground) + np.arange(len(obj)), 50.0, res)
        nc, nh, ns = _np_bev(ground, obj, res)
        assert np.array_equal(count, rc) and np.array_equal(count.astype(np.int64), nc), (res, name)
        assert _same_f32(height, rh) and _same_f32(height, nh), (res, name)
        assert np.array_equal(sem, rs) and np.array_equal(sem, ns), (res, name, int((sem != ns).any(-1).sum()))
        assert int(count.sum()) == len(ground) + len(obj)
        if name == "crowded_cell":
            assert count.max() >= 70000
        if name == "negative_z":
            assert not height.any()
        if name == "flat_object_z":
            assert set(np.unique(sem[..., 1])) <= {0, 80, 255} and (sem[..., 1] == 255).any()


# ------------------------------------------------------------------------------------------------ multi-sweep aggregation
def _sweep_rows(rng, n, rc):
    raw = np.zeros((n, 5), np.float32)
    raw[:, :3] = rng.uniform(-40, 40, (n, 3))
    raw[:, 2] *= 0.1
    raw[:, 3] = rng.uniform(0, 255, n)
    raw[:, 4] = rng.integers(0, 32, n)
    special = np.array([(rc, 0.5), (-rc, 0.2), (0.3, rc), (0.3, -rc), (rc, rc), (-rc, -rc), (_dn(rc), 0.5), (_up(rc), 0.5),
                        (0.5, _dn(rc)), (0.5, _up(-rc)), (0.0, 0.0), (-0.0, 0.5), (np.nan, 0.5), (0.5, np.nan), (np.nan, np.nan)],
                       np.float32)
    if n:
        at = rng.choice(n, min(n, 3 * len(special)), replace=False)
        raw[at, :2] = special[np.arange(at.size) % len(special)]
        raw[at[: at.size // 4], 2] = np.nan
    return raw


def _pose(rng):
    a = rng.uniform(-np.pi, np.pi)
    M = np.zeros((3, 4))
    M[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    M[2, 2] = 1.0
    M[:, 3] = rng.uniform(-20, 20, 3)
    M[:2, 2] = rng.uniform(-0.01, 0.01, 2)
    return M


def _np_aggregate(sweeps, rc):
    """devkit from_file_multisweep (App. A.1): drop |x| < r and |y| < r (NaN kept), transform in float64, cast to float32."""
    out, lag = [], []
    for raw, M, tl in sweeps:
        keep = ~((np.abs(raw[:, 0]) < f32(rc)) & (np.abs(raw[:, 1]) < f32(rc)))
        p = raw[keep].astype(np.float64)
        xyz = (p[:, :3] @ M[:, :3].T + M[:, 3]).astype(np.float32)
        out.append(np.column_stack([xyz, raw[keep, 3]]).astype(np.float32))
        lag.append(np.full(len(p), tl, np.float32))
    return np.vstack(out), np.concatenate(lag)


_AGG_CASES = {
    "empty_ends_and_middle": ([0, 1, 1023, 0, 4097, 34719, 3, 0], 1.0),
    "ragged_other_radius": ([5, 0, 1025, 77, 2, 0, 1], 2.5),
    "single_row": ([1], 1.0),
    "span_above_2_20": ([34720] * 13 + [0] + [34720] * 16 + [33001, 34720], 1.0),   # 31 sweeps: 1,076,320-row span
}


@pytest.mark.parametrize("case", list(_AGG_CASES))
def test_aggregate_sweeps_empty_sweeps_radius_edges_nan_and_long_spans(engine, case):
    lengths, rc = _AGG_CASES[case]
    rng = np.random.default_rng(700 + list(_AGG_CASES).index(case))
    sweeps = [(_sweep_rows(rng, n, rc), _pose(rng), float(np.float32(0.05 * k))) for k, n in enumerate(lengths)]
    xyzi, tl = ops.aggregate_sweeps(engine, sweeps, remove_close_radius=rc)
    s = make_sample(90, n_sweeps=1, n_boxes=0)
    s["lidar_sweeps"] = [{"points_raw": raw, "ref_from_sensor": M, "time_lag": lag} for raw, M, lag in sweeps]
    ref_xyzi, ref_t = OB.oracle_aggregate(pack_batch([s]), 0, rc)
    assert _same_f32(xyzi, ref_xyzi) and np.array_equal(tl, ref_t), case
    np_xyzi, np_t = _np_aggregate(sweeps, rc)
    assert xyzi.shape == np_xyzi.shape and np.array_equal(tl, np_t)
    assert _same_f32(xyzi[:, 3], np_xyzi[:, 3]) and np.array_equal(np.isnan(xyzi), np.isnan(np_xyzi))
    fin = ~np.isnan(np_xyzi[:, :3])
    diff = np.abs(xyzi[:, :3][fin].astype(np.float64) - np_xyzi[:, :3][fin])
    assert (diff <= np.spacing(np.abs(np_xyzi[:, :3][fin]))).all()          # within 1 ulp of float32
    if case == "span_above_2_20":
        assert len(lengths) * max(lengths) > (1 << 20)


# ------------------------------------------------------------------------------------------------ cloud statistics
@pytest.mark.parametrize("pitch", [4, 5])
@pytest.mark.parametrize("n", [1, 303_104, 303_105, 2_000_000])
def test_cloud_stats_sizes_pitches(engine, n, pitch):
    rng = np.random.default_rng(n + pitch)
    raw = np.full((n, pitch), 3.0, np.float32)
    raw[:, :2] = rng.uniform(-80, 80, (n, 2))
    raw[:, 2] = rng.uniform(-5, 10, n)
    if n > 1:
        raw[n - 1, :3] = (-999.0, 999.0, -999.0)   # extremes in the last row: only the grid-stride loop reaches it above 303,104
        raw[n // 2, :3] = (998.0, -998.0, 997.0)
    view = raw[:, :4]
    assert ops._raw_rows(view)[1] == (pitch if n > 1 else 4)
    mn, mx, mean = ops.cloud_stats(engine, view)
    x = np.ascontiguousarray(view[:, :3])
    assert _same_f32(mn, x.min(0)) and _same_f32(mx, x.max(0)), (n, pitch)
    omm, osum = OB.oracle_cloud_stats(view)
    assert _same_f32(mn, omm[:3]) and _same_f32(mx, omm[3:])
    radial = np.sqrt(x[:, 0] * x[:, 0] + x[:, 1] * x[:, 1]).astype(np.float64)   # float32 sqrt(x*x + y*y), summed exactly
    exact = math.fsum(radial.tolist()) / n
    assert abs(mean - exact) <= 1e-12 * exact and abs(osum / n - exact) <= 1e-12 * exact


def test_cloud_stats_signed_zero_extremes_are_order_independent(engine):
    """A minimum of zero with both -0.0 and 0.0 present (and a maximum likewise): the kernel orders -0.0 below 0.0, so min is
    -0.0 and max is 0.0 wherever they sit.  NumPy's float32 min/max return whichever zero its loop met last, which depends on
    position, length and stride; a prompt formats the value with f"{v:.1f}", where the kernel prints "-0.0" for X here.
    The values compare equal to NumPy's; only the sign of a zero extreme can differ."""
    rng = np.random.default_rng(11)
    n = 5000
    pc = np.zeros((n, 4), np.float32)
    pc[:, 0] = rng.uniform(0.5, 40, n)       # x >= 0: minimum is a zero
    pc[:, 1] = rng.uniform(-40, -0.5, n)     # y <= 0: maximum is a zero
    pc[:, 2] = rng.uniform(-2, 2, n)
    pc[[10, 4000], 0] = (0.0, -0.0)
    pc[[20, 30], 1] = (-0.0, 0.0)
    for perm in (np.arange(n), np.arange(n)[::-1], rng.permutation(n)):
        mn, mx, _ = ops.cloud_stats(engine, pc[perm])
        assert mn[0] == 0 and np.signbit(mn[0]) and f"{mn[0]:.1f}" == "-0.0"
        assert mx[1] == 0 and not np.signbit(mx[1]) and f"{mx[1]:.1f}" == "0.0"
        assert mn[0] == pc[perm, 0].min() and mx[1] == pc[perm, 1].max()
    # NumPy's sign follows the order: both answers occur for the same set of values
    signs = {bool(np.signbit(np.array(v, np.float32).min())) for v in ([0.0, -0.0], [-0.0, 0.0])}
    assert signs == {True, False}


# ------------------------------------------------------------------------------------------------ cluster AABB
def _np_cluster_aabb(pts, labels, k):
    """lidar_agent.py:200-204 per cluster in float32 (min, max, (min+max)/2, sqrt(cx^2+cy^2), count); empty clusters keep the
    +inf / -inf starting values, so their centre and distance are NaN."""
    ok = (labels >= 0) & (labels < k)
    lab, p = labels[ok], pts[ok, :3].astype(np.float32)
    mn = np.full((k, 3), np.inf, np.float32)
    mx = np.full((k, 3), -np.inf, np.float32)
    np.minimum.at(mn, lab, p)
    np.maximum.at(mx, lab, p)
    with np.errstate(invalid="ignore"):
        ctr = (mn + mx) / f32(2)
        dist = np.sqrt(ctr[:, 0] * ctr[:, 0] + ctr[:, 1] * ctr[:, 1])
    cnt = np.bincount(lab, minlength=k).astype(np.float32)
    return np.column_stack([mn, mx, ctr, dist, cnt]).astype(np.float32)


@pytest.mark.parametrize("pitch", [4, 5])
def test_cluster_aabb_empty_single_outside_labels_and_many_clusters(engine, pitch):
    rng = np.random.default_rng(40 + pitch)
    k, n = 5000, 200_000
    raw = np.full((n, pitch), 1.0, np.float32)
    raw[:, :3] = rng.uniform(-50, 50, (n, 3))
    view = raw[:, :4]
    labels = rng.integers(20, k, n).astype(np.int32)
    labels[rng.random(n) < 0.1] = -1
    outside = rng.random(n) < 0.05
    labels[outside] = rng.choice(np.array([k, k + 1, 2 * k, 2 ** 31 - 1, -2, -2 ** 31], np.int64), int(outside.sum())).astype(np.int32)
    labels[rng.choice(n, 10, replace=False)] = np.arange(10, 20)          # clusters 10..19 hold one point, 0..9 none
    got = ops.cluster_aabb(engine, view, labels, k)
    ref = OB.oracle_cluster_aabb(view, labels, k)
    want = _np_cluster_aabb(np.ascontiguousarray(view), labels, k)
    assert _same_f32(got, ref) and _same_f32(got, want)
    assert np.isnan(got[:10, 6:10]).all() and (got[:10, 10] == 0).all() and (got[10:20, 10] == 1).all()
    assert np.array_equal(got[10:20, 0:3], got[10:20, 3:6])
    assert int(got[:, 10].sum()) == int(((labels >= 0) & (labels < k)).sum())


# ------------------------------------------------------------------------------------------------ annotation table
_ZONES = [(0, 10, 0), (10, 30, 0), (30, 50, 0), (0, 10, 1), (10, 30, 1), (0, 10, 3), (10, 30, 3), (0, 10, 2), (10, 30, 2)]


def _diag_on_circle(d):
    """x > 0 with sqrt(x*x + x*x) == d in float64 when one exists nearby, and its two neighbours."""
    x = d / math.sqrt(2.0)
    for _ in range(200):
        if math.sqrt(x * x + x * x) == d:
            break
        x = math.nextafter(x, math.inf if math.sqrt(x * x + x * x) < d else -math.inf)
    return [x, math.nextafter(x, -math.inf), math.nextafter(x, math.inf)]


def _annotation_edge_rows():
    """(x, y, vx, vy, on_a_bin_edge_exactly): axes and diagonals at distance 0, 10, 30, 50 and around them, signed zeros,
    Pythagorean points exactly on the zone radii, speeds 0.5 and NaN."""
    rows = []
    for d in (10.0, 30.0, 50.0, 5.0, 20.0, 40.0):
        for v in (d, math.nextafter(d, 0), math.nextafter(d, 100)):
            for sx, sy in ((v, 0.0), (-v, 0.0), (0.0, v), (0.0, -v), (v, -0.0), (-v, -0.0), (-0.0, v), (-0.0, -v)):
                rows.append((sx, sy, True))
        for x in _diag_on_circle(d):
            for sx, sy in ((1, 1), (-1, 1), (-1, -1), (1, -1)):
                rows.append((sx * x, sy * x, True))
    for a, b in ((6, 8), (18, 24), (30, 40)):
        for sx, sy in ((1, 1), (-1, 1), (-1, -1), (1, -1)):
            rows += [(sx * a, sy * b, True), (sx * b, sy * a, True)]
    for z in ((0.0, 0.0), (-0.0, 0.0), (0.0, -0.0), (-0.0, -0.0)):
        rows.append((*z, True))
    for x in (3.0, 12.5, 0.1):                                  # one float off the diagonals: the exact predicates decide
        for sx, sy in ((1, 1), (-1, 1), (-1, -1), (1, -1)):
            rows.append((sx * x, sy * math.nextafter(x, math.inf), False))
            rows.append((sx * x, sy * math.nextafter(x, 0.0), False))
    vel = [(0.5, 0.0), (0.0, -0.5), (-0.5, -0.0), (math.nextafter(0.5, 1), 0.0), (math.nextafter(0.5, 0), 0.0), (0.3, 0.4),
           (np.nan, 0.0), (0.0, np.nan), (np.nan, np.nan), (np.inf, 0.0), (2.0, 1.0), (0.0, 0.0)]
    return [(x, y, *vel[i % len(vel)], exact) for i, (x, y, exact) in enumerate(rows)]


def _ref_annotation(x, y, vx, vy):
    """scenegraph_agent.py:186-225 (Python floats, ** and atan2 bins), :281-295 (first zone that matches),
    baseline_gpt4o.py:304-317 (front: x > 0, left: y > 0)."""
    distance = float(np.sqrt(x ** 2 + y ** 2))
    angle = float(np.arctan2(y, x)) * 180 / np.pi
    angle = (angle + 360) % 360
    direction = 0 if 45 <= angle < 135 else 1 if 135 <= angle < 225 else 2 if 225 <= angle < 315 else 3
    moving = 1 if np.sqrt(vx ** 2 + vy ** 2) > 0.5 else 0
    zone = next((k for k, (lo, hi, dr) in enumerate(_ZONES) if dr == direction and lo <= distance < hi), 255)
    return distance, direction, moving, zone, (1 if x > 0 else 0) | (2 if y > 0 else 0)


@pytest.mark.parametrize("n", [1, 255, 256, 257, 10_000])
def test_annotation_table_zone_edges_signed_zeros_speed_and_blocks(engine, n):
    rng = np.random.default_rng(60 + n)
    edges = _annotation_edge_rows()
    xy = rng.uniform(-60, 60, (n, 2))
    vel = rng.uniform(-2, 2, (n, 2))
    exact = np.ones(n, bool)
    pos = rng.permutation(n)[: len(edges)] if n >= len(edges) else np.arange(n)     # edge rows spread over the blocks
    for i, p in enumerate(pos):
        x, y, vx, vy, e = edges[i]
        xy[p] = (x, y); vel[p] = (vx, vy); exact[p] = e
    if n == 1:
        xy[0], vel[0] = (0.0, 10.0), (0.5, 0.0)              # exactly on the front_close / front_medium edge
    got = ops.annotation_table(engine, xy, vel)
    orc = OB.oracle_annotation_table(xy, vel)
    # the table's own arithmetic: sqrt(x*x + y*y) in float64
    assert _same_f64(got["distance"], np.sqrt(xy[:, 0] * xy[:, 0] + xy[:, 1] * xy[:, 1]))
    for k in ("direction", "moving", "zone", "region_bits"):
        assert np.array_equal(got[k], orc[k]), k
    # the oracle and the reference square with pow(): within 2 ulp
    assert (np.abs(got["distance"] - orc["distance"]) <= 2 * np.spacing(orc["distance"])).all()
    ref = np.array([_ref_annotation(*(float(v) for v in (*xy[i], *vel[i]))) for i in range(n)], dtype=np.float64)
    assert (np.abs(got["distance"] - ref[:, 0]) <= 2 * np.spacing(ref[:, 0])).all()
    for j, k in enumerate(("direction", "moving", "zone", "region_bits"), start=1):
        rows = exact if k in ("direction", "zone") else np.ones(n, bool)
        bad = np.flatnonzero(rows & (got[k] != ref[:, j].astype(np.uint8)))
        assert bad.size == 0, (k, [(xy[b].tolist(), vel[b].tolist(), int(got[k][b]), int(ref[b, j])) for b in bad[:5]])
    if n == 1:
        assert int(got["zone"][0]) == 1 and got["moving"][0] == 0
    if n >= len(edges):
        assert np.isin(got["distance"], [0.0, 10.0, 30.0, 50.0]).sum() >= 40


# ------------------------------------------------------------------------------------------------ relation tables
def _rel_boxes(rng, n):
    """n boxes (translation, w l h, quaternion wxyz): random yawed boxes, and where n allows axis-aligned dyadic pairs that touch
    exactly (t == ra + rb) or sit one float apart, and pairs at dy = +-0 and a tiny negative dy (the 0/360 bearing wrap)."""
    b = np.zeros((n, 10))
    b[:, 0:2] = rng.uniform(-60, 60, (n, 2))
    b[:, 2] = rng.uniform(-1, 2, n)
    b[:, 3:6] = rng.uniform(0.5, 6, (n, 3))
    yaw = rng.uniform(-np.pi, np.pi, n)
    b[:, 6], b[:, 9] = np.cos(yaw / 2), np.sin(yaw / 2)
    crafted = []
    x0, y0 = 4.0, -8.0
    for la, wa, lb, wb in ((2.0, 1.0, 4.0, 0.5), (0.75, 3.0, 1.25, 2.0)):
        A = (x0, y0, la, wa)
        crafted += [A, (x0 + la / 2 + lb / 2, y0, lb, wb),                                    # touching along x
                    (x0, y0 - wa / 2 - wb / 2, lb, wb),                                        # touching along y
                    (x0 - la / 2 - lb / 2, y0 + wa / 2 + wb / 2, lb, wb),                      # touching at a corner
                    (math.nextafter(x0 + la / 2 + lb / 2, math.inf), y0 + 0.25, lb, wb),        # one float apart
                    (x0 + 0.5, math.nextafter(y0 - wa / 2 - wb / 2, -math.inf), lb, wb)]
        x0 += 20.0
    crafted += [(-30.0, 0.0, 1.0, 1.0), (-20.0, -0.0, 1.0, 1.0), (-10.0, -1e-9, 1.0, 1.0), (-40.0, 1e-300, 1.0, 1.0),
                (-25.0, -1e-300, 1.0, 1.0), (-0.0, 30.0, 1.0, 1.0), (0.0, 45.0, 1.0, 1.0)]
    m = min(n, len(crafted))
    at = rng.permutation(n)[:m]
    for i, (x, y, l, w) in zip(at, crafted[:m]):
        b[i] = (x, y, 0.5, w, l, 1.5, 1.0, 0.0, 0.0, 0.0)
    return b


def _np_footprints(boxes):
    """box_footprints without an ego pose: centre xy, normalised xy of the box x axis (quat_to_rot, same order), l/2, w/2."""
    q = boxes[:, 6:10]
    nn = np.sqrt(((q[:, 0] * q[:, 0] + q[:, 1] * q[:, 1]) + q[:, 2] * q[:, 2]) + q[:, 3] * q[:, 3])
    w, x, y, z = (q[:, k] / nn for k in range(4))
    ux = 1.0 - 2.0 * (y * y + z * z)
    uy = 2.0 * (x * y + w * z)
    h = np.sqrt(ux * ux + uy * uy)
    ux, uy = np.where(h > 0, ux / np.where(h > 0, h, 1), 1.0), np.where(h > 0, uy / np.where(h > 0, h, 1), 0.0)
    return np.column_stack([boxes[:, 0], boxes[:, 1], ux, uy, boxes[:, 4] / 2.0, boxes[:, 3] / 2.0])


def _np_bearing4(dx, dy):
    cat = np.full(dx.shape, 3, np.uint8)
    cat[(dx < 0) & (dy <= -dx) & (dy > dx)] = 1
    cat[(dy < 0) & (dx >= dy) & (dx < -dy)] = 2
    cat[(dy > 0) & (dx <= dy) & (-dx < dy)] = 0
    zero = (dx == 0) & (dy == 0)
    cat[zero] = np.where(np.signbit(dx[zero]), 1, 3)
    return cat


def _np_relations(rect):
    """Pairwise table in float64 with the kernel's operation order (NumPy does not fuse): distance, atan2 bearing in degrees
    wrapped by fmod, bearing4 category, separating-axis overlap (touching counts as overlap)."""
    A, B = rect[:, None, :], rect[None, :, :]
    dx, dy = B[..., 0] - A[..., 0], B[..., 1] - A[..., 1]
    ang = np.fmod(np.arctan2(dy, dx) * 180.0 / 3.14159265358979323846 + 360.0, 360.0)
    sep = np.zeros(dx.shape, bool)
    for ex, ey in ((A[..., 2], A[..., 3]), (-A[..., 3], A[..., 2]), (B[..., 2], B[..., 3]), (-B[..., 3], B[..., 2])):
        t = np.abs(dx * ex + dy * ey)
        ra = A[..., 4] * np.abs(A[..., 2] * ex + A[..., 3] * ey) + A[..., 5] * np.abs(-A[..., 3] * ex + A[..., 2] * ey)
        rb = B[..., 4] * np.abs(B[..., 2] * ex + B[..., 3] * ey) + B[..., 5] * np.abs(-B[..., 3] * ex + B[..., 2] * ey)
        sep |= t > ra + rb
    return {"dist": np.sqrt(dx * dx + dy * dy).astype(np.float32), "bearing": ang.astype(np.float32), "category": _np_bearing4(dx, dy),
            "overlap": (~sep).astype(np.uint8)}


def _bearing_close(a, b):
    """Same angle on the circle within 1e-5 relative: 359.99998 and 0 are neighbours, not 360 degrees apart."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    d = np.abs(np.mod(a - b + 180.0, 360.0) - 180.0)
    return bool((d <= 1e-5 * np.maximum(np.abs(b), 1.0)).all() and ((a >= 0) & (a <= 360)).all())


def _check_relations(got, rect):
    ref = OB.oracle_relations(rect)
    mine = _np_relations(rect)
    for k in ("dist", "category", "overlap"):
        assert np.array_equal(got[k], ref[k]) and np.array_equal(got[k], mine[k]), k
    assert _bearing_close(got["bearing"], ref["bearing"]) and _bearing_close(got["bearing"], mine["bearing"])


@pytest.mark.parametrize("n", [1, 15, 16, 17, 33, 1000])
def test_relation_table_tile_edges_touching_and_bearing_wrap(engine, n):
    rng = np.random.default_rng(800 + n)
    boxes = _rel_boxes(rng, n)
    ego = np.array([3.0, -2.0, 0.5, np.cos(0.3), 0.0, 0.0, np.sin(0.3)])
    for pose in (None, ego):
        got = ops.relation_table(engine, boxes, pose)
        rect = OB.oracle_footprints(boxes, pose)
        assert np.array_equal(got["rect"], rect)
        if pose is None:
            assert np.array_equal(rect, _np_footprints(boxes))
        _check_relations(got, rect)
    got = ops.relation_table(engine, boxes)
    assert (np.diag(got["overlap"]) == 1).all() and (np.diag(got["category"]) == 3).all()
    if n >= 17:
        assert got["overlap"].sum() > n          # the crafted touching pairs overlap
        assert (got["bearing"] == 360.0).any()   # dy = -1e-9 at dx = 20: the float32 bearing rounds up to 360


def test_relation_table_batch_ragged_samples_writes_only_its_slices(engine):
    import torch
    rng = np.random.default_rng(900)
    d = engine.device
    for counts in (rng.choice([0, 1, 16, 17, 200], 44), rng.choice([0, 1, 16, 17], 41)):
        counts = counts.astype(np.int64)
        counts[rng.integers(0, len(counts))] = counts.max()
        S, max_boxes = len(counts), int(counts.max())
        assert max_boxes % 16
        boxes = [_rel_boxes(rng, int(c)) for c in counts]
        rect = np.vstack([OB.oracle_footprints(b, None) for b in boxes if len(b)])
        box_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        gaps = rng.integers(1, 40, S)                              # untouched guard elements before every sample's slice
        pair_off = np.zeros(S, np.int64)
        cur = 0
        for s in range(S):
            cur += int(gaps[s])
            pair_off[s] = cur
            cur += int(counts[s]) ** 2
        total = cur + 37
        SENT_F, SENT_U = np.float32(-1234.5), 0xEE
        out = {"dist": torch.full((total,), float(SENT_F), dtype=torch.float32, device=d),
               "bearing": torch.full((total,), float(SENT_F), dtype=torch.float32, device=d),
               "category": torch.full((total,), SENT_U, dtype=torch.uint8, device=d),
               "overlap": torch.full((total,), SENT_U, dtype=torch.uint8, device=d)}
        t_rect = torch.from_numpy(rect).to(d)
        t_box = torch.from_numpy(box_off).to(d)
        t_pair = torch.from_numpy(pair_off).to(d)
        _capi.check(engine.lib.msc_relation_table_batch(S, max_boxes, t_box.data_ptr(), t_pair.data_ptr(), t_rect.data_ptr(),
                                                        out["dist"].data_ptr(), out["bearing"].data_ptr(), out["category"].data_ptr(),
                                                        out["overlap"].data_ptr(), ops._stream(engine)), "msc_relation_table_batch")
        torch.cuda.synchronize()
        host = {k: v.cpu().numpy() for k, v in out.items()}
        written = np.zeros(total, bool)
        for s in range(S):
            n = int(counts[s])
            sl = slice(int(pair_off[s]), int(pair_off[s]) + n * n)
            written[sl] = True
            if n == 0:
                continue
            got = {k: host[k][sl].reshape(n, n) for k in host}
            _check_relations(got, rect[box_off[s]:box_off[s + 1]])
        for k, v in host.items():
            sent = SENT_F if v.dtype == np.float32 else SENT_U
            assert (v[~written] == sent).all(), k


# ------------------------------------------------------------------------------------------------ box -> camera projection
def _py_quat_to_rot(q):
    w, x, y, z = (float(v) for v in q)
    n = math.sqrt(((w * w + x * x) + y * y) + z * z)
    w, x, y, z = w / n, x / n, y / n, z / n
    xx, yy, zz, xy, xz, yz, wx, wy, wz = x * x, y * y, z * z, x * y, x * z, y * z, w * x, w * y, w * z
    return [1.0 - 2.0 * (yy + zz), 2.0 * (xy - wz), 2.0 * (xz + wy), 2.0 * (xy + wz), 1.0 - 2.0 * (xx + zz), 2.0 * (yz - wx),
            2.0 * (xz - wy), 2.0 * (yz + wx), 1.0 - 2.0 * (xx + yy)]


def _py_frame_change(pose7, c, R):
    P = _py_quat_to_rot(pose7[3:7])
    d0, d1, d2 = c[0] - float(pose7[0]), c[1] - float(pose7[1]), c[2] - float(pose7[2])
    c = [(P[0] * d0 + P[3] * d1) + P[6] * d2, (P[1] * d0 + P[4] * d1) + P[7] * d2, (P[2] * d0 + P[5] * d1) + P[8] * d2]
    R = [(P[0 * 3 + r] * R[0 * 3 + k] + P[1 * 3 + r] * R[1 * 3 + k]) + P[2 * 3 + r] * R[2 * 3 + k] for r in range(3) for k in range(3)]
    return c, R


def _py_project(boxes, pose, calib, K, W, H):
    """devkit get_sample_data + view_points + box_in_image(BoxVisibility.ANY) in float64, one operation at a time."""
    nb, nc = len(boxes), len(pose)
    vis = np.zeros((nb, nc), np.uint8)
    ext = np.zeros((nb, nc, 4), np.float32)
    for b in range(nb):
        box = [float(v) for v in boxes[b]]
        hl, hw, hh = box[4] / 2.0, box[3] / 2.0, box[5] / 2.0
        for c in range(nc):
            ctr, R = _py_frame_change(pose[c], box[0:3], _py_quat_to_rot(box[6:10]))
            ctr, R = _py_frame_change(calib[c], ctr, R)
            k = [float(v) for v in K[c]]
            any_vis, all_front = False, True
            umin = vmin = math.inf
            umax = vmax = -math.inf
            for j in range(8):
                lx = hl if j < 4 else -hl
                ly = hw if j in (0, 3, 4, 7) else -hw
                lz = hh if j in (0, 1, 4, 5) else -hh
                X = ((R[0] * lx + R[1] * ly) + R[2] * lz) + ctr[0]
                Y = ((R[3] * lx + R[4] * ly) + R[5] * lz) + ctr[1]
                Z = ((R[6] * lx + R[7] * ly) + R[8] * lz) + ctr[2]
                pu, pv, pw = (k[0] * X + k[1] * Y) + k[2] * Z, (k[3] * X + k[4] * Y) + k[5] * Z, (k[6] * X + k[7] * Y) + k[8] * Z
                with np.errstate(all="ignore"):
                    u, v = float(np.float64(pu) / np.float64(pw)), float(np.float64(pv) / np.float64(pw))
                if u > 0.0 and u < W and v > 0.0 and v < H and Z > 1.0:
                    any_vis = True
                if not Z > 0.1:
                    all_front = False
                umin, umax, vmin, vmax = (u if u < umin else umin), (u if u > umax else umax), (v if v < vmin else vmin), (v if v > vmax else vmax)
            if any_vis and all_front:
                vis[b, c] = 1
                ext[b, c] = (0.0 if umin < 0.0 else umin, 0.0 if vmin < 0.0 else vmin, W if umax > W else umax, H if vmax > H else vmax)
    return vis, ext


def _solve_offset(target, half):
    """c with (-half) + c == target exactly in float64 (the kernel adds the rotated corner offset to the centre)."""
    c = target + half
    for _ in range(8):
        if (-half) + c == target:
            return c
        c = math.nextafter(c, math.inf if (-half) + c < target else -math.inf)
    raise AssertionError("no exact centre")


def _projection_boxes():
    """Axis-aligned boxes for identity camera poses and K = [[1000, 0, 800], [0, 1000, 450], [0, 0, 1]], W x H = 1600 x 900:
    a face exactly on Z = 0.1 or Z = 1.0, or one float beyond; boxes straddling Z = 0; corners exactly on u = 0, u = W and
    v = H; zero-size boxes.  Returns (boxes, expected visibility through camera 0)."""
    I = (1.0, 0.0, 0.0, 0.0)
    rows = []

    def box(c, w, l, h, want):
        rows.append(((*c, w, l, h, *I), want))
    # an exact Z = 0.1 face needs a centre below 0.25 (0.1 is an odd multiple of 2^-55), so these boxes are also too near
    # for Z > 1.0; the oracle and the float64 restatement hold the comparison itself
    box((0.0, 0.0, _solve_offset(0.1, 0.0625)), 1.0, 1.0, 0.125, 0)                  # near face on Z = 0.1
    box((0.0, 0.0, math.nextafter(_solve_offset(0.1, 0.0625), 9)), 1.0, 1.0, 0.125, 0)
    box((0.0, 0.0, 0.75), 0.5, 1.0, 0.5, 0)                                          # Z in {0.5, 1.0}: no corner with Z > 1
    box((0.0, 0.0, math.nextafter(1.0, 2.0) - 0.25), 0.5, 1.0, 0.5, 1)              # far face one float beyond Z = 1.0
    box((0.0, 0.0, 1.0), 1.0, 1.0, 0.0, 0)                                           # flat box on Z = 1.0
    box((0.0, 0.0, 0.0), 1.0, 1.0, 4.0, 0)                                           # straddles the camera plane
    box((0.5, -0.5, -1.0), 2.0, 2.0, 6.0, 0)
    box((0.0, 0.0, -5.0), 1.0, 1.0, 1.0, 0)                                          # behind the camera
    # u = (1000 X + 800 Z) / Z: X = -0.8 Z gives u = 0, X = 0.8 Z gives u = W; v = H at Y = 0.45 Z.  Z = 5 (zero height).
    box((-4.0, 0.0, 5.0), 1.0, 0.0, 0.0, 0)                                          # every corner on u = 0
    box((-3.5, 0.0, 5.0), 1.0, 1.0, 0.0, 1)                                          # from u = 0 into the image
    box((4.0, 0.0, 5.0), 1.0, 0.0, 0.0, 0)                                           # every corner on u = W
    box((3.5, 0.0, 5.0), 1.0, 1.0, 0.0, 1)                                           # up to u = W
    box((4.5, 0.0, 5.0), 1.0, 1.0, 0.0, 0)                                           # from u = W outwards
    box((0.0, 2.25, 5.0), 0.0, 1.0, 0.0, 0)                                          # every corner on v = H
    box((0.0, 2.0, 5.0), 0.5, 1.0, 0.0, 1)                                           # up to v = H
    box((0.0, -2.25, 5.0), 0.0, 1.0, 0.0, 0)                                         # every corner on v = 0
    box((1.0, 1.0, 5.0), 0.0, 0.0, 0.0, 1)                                           # zero-size box inside
    box((9.0, 1.0, 5.0), 0.0, 0.0, 0.0, 0)                                           # zero-size box outside
    box((-4.0, -2.25, 5.0), 0.0, 0.0, 0.0, 0)                                        # the (0, 0) image corner
    box((4.0, 2.25, 5.0), 0.0, 0.0, 0.0, 0)                                          # the (W, H) image corner
    box((0.0, 0.0, 30.0), 3.0, 8.0, 2.0, 1)
    return np.array([r[0] for r in rows]), np.array([r[1] for r in rows], np.uint8)


@pytest.mark.parametrize("n_cams", [1, 8])
def test_project_boxes_planes_image_edges_and_camera_counts(engine, n_cams):
    rng = np.random.default_rng(300 + n_cams)
    edge_boxes, want0 = _projection_boxes()
    ident = np.tile([0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0], (n_cams, 1))
    K = np.tile(np.array([1000.0, 0.0, 800.0, 0.0, 1000.0, 450.0, 0.0, 0.0, 1.0]), (n_cams, 1))
    K[1:, 0] = K[1:, 4] = rng.uniform(500, 1500, n_cams - 1)
    K[1:, 2] = rng.uniform(700, 900, n_cams - 1)
    # random boxes through random camera poses (yawed, pitched, offset) to cover the general path
    nb = 120
    rnd = np.zeros((nb, 10))
    rnd[:, 0:3] = rng.uniform(-30, 30, (nb, 3))
    rnd[:, 3:6] = rng.uniform(0.0, 5.0, (nb, 3))
    q = rng.normal(size=(nb, 4)); rnd[:, 6:10] = q
    pose = np.zeros((n_cams, 7)); calib = np.zeros((n_cams, 7))
    for c in range(n_cams):
        a = rng.uniform(-np.pi, np.pi)
        pose[c] = (*rng.uniform(-2, 2, 3), np.cos(a / 2), 0.0, 0.0, np.sin(a / 2))
        cq = rng.normal(size=4); cq /= np.linalg.norm(cq)
        calib[c] = (*rng.uniform(-1, 1, 3), *cq)
    for boxes, P, Cc in ((edge_boxes, ident, ident), (rnd, pose, calib), (np.vstack([edge_boxes, rnd]), pose, ident)):
        vis, ext = ops.project_boxes(engine, boxes, P, Cc, K)
        rv, re = OB.oracle_project(boxes, P, Cc, K)
        pv, pe = _py_project(boxes, P, Cc, K, 1600.0, 900.0)
        assert np.array_equal(vis, rv) and _same_f32(ext, re)
        assert np.array_equal(vis, pv) and _same_f32(ext, pe)
    vis, ext = ops.project_boxes(engine, edge_boxes, ident, ident, K)
    assert np.array_equal(vis[:, 0], want0), np.flatnonzero(vis[:, 0] != want0)
    assert not ext[vis == 0].any()
    e = ext[:, 0]
    assert e[9, 0] == 0.0 and e[11, 2] == 1600.0 and e[14, 3] == 900.0


# ------------------------------------------------------------------------------------------------ DBSCAN below 12 points
def _exact_dbscan(X, eps, min_samples):
    """The rule the device implements: neighbours when (dx^2 + dy^2) + dz^2 <= eps^2 in float64 (x, then y, then z); core points
    have >= min_samples neighbours (themselves included); clusters are expanded from cores in index order; a border point takes
    the first cluster that reaches it; the rest is noise."""
    X = np.asarray(X, np.float64)
    n = len(X)
    d = (X[:, None, 0] - X[None, :, 0]) ** 2
    d = d + (X[:, None, 1] - X[None, :, 1]) ** 2
    d = d + (X[:, None, 2] - X[None, :, 2]) ** 2
    nb = d <= eps * eps
    core = nb.sum(1) >= min_samples
    lab = np.full(n, -1, np.int64)
    k = 0
    for i in range(n):
        if lab[i] != -1 or not core[i]:
            continue
        stack = [i]
        lab[i] = k
        while stack:
            j = stack.pop()
            if core[j]:
                for m in np.flatnonzero(nb[j] & (lab == -1)):
                    lab[m] = k
                    stack.append(m)
        k += 1
    return lab


def _min_gap_to_eps(X, eps):
    X = np.asarray(X, np.float64)
    d = np.sqrt(((X[:, None, :] - X[None, :, :]) ** 2).sum(-1))
    iu = np.triu_indices(len(X), 1)
    return np.abs(d[iu] - eps).min() if iu[0].size else np.inf


def test_dbscan_small_inputs_sklearn_brute_force_and_exact_eps(engine):
    """scikit-learn's DBSCAN searches neighbours by brute force when n <= 11 (its NearestNeighbors keeps n_neighbors = 5, and
    5 >= n // 2), with a BLAS expansion of the distance that can drop a pair whose distance is exactly eps.  The device
    applies the float64 x -> y -> z rule (the KD-tree path's) at every n.  Away from exact-eps pairs both agree; on exact-eps
    pairs the device follows the rule, which _exact_dbscan restates."""
    from sklearn.cluster import DBSCAN
    rng = np.random.default_rng(1234)
    # the chain of five points at spacing exactly 0.5 where scikit-learn's brute force drops the 3-4 pair
    X = np.repeat(np.float32([[-7.2988081, 29.107883, -1.7544454]]), 5, 0)
    X[:, 1] = (X[0, 1] + np.float32(0.5) * np.arange(5, dtype=np.float32)).astype(np.float32)
    assert float(X[4, 1]) - float(X[3, 1]) == 0.5
    assert np.array_equal(ops.dbscan(engine, X, 0.5, 1), [0, 0, 0, 0, 0])
    assert np.array_equal(_exact_dbscan(X, 0.5, 1), [0, 0, 0, 0, 0])
    checked_sklearn = 0
    for t in range(300):
        n = int(rng.integers(1, 12))
        ms = int(rng.choice([1, 2, 3, 4, 10]))
        X = (rng.uniform(-2, 2, 3) + rng.normal(0, 0.4, (n, 3))).astype(np.float32)
        got = ops.dbscan(engine, X, 0.5, ms)
        assert np.array_equal(got, _exact_dbscan(X, 0.5, ms)), (t, X.tolist(), ms)
        if _min_gap_to_eps(X, 0.5) > 1e-6:
            assert np.array_equal(got, DBSCAN(eps=0.5, min_samples=ms).fit(X).labels_), (t, X.tolist(), ms)
            checked_sklearn += 1
    assert checked_sklearn > 250
    # the reference's call (min_samples = 10) at 10 and 11 points: one cluster, all noise, and a single core point's border
    for n in (10, 11):
        for spread in (0.05, 0.2, 3.0):
            X = (rng.uniform(-5, 5, 3) + rng.normal(0, spread, (n, 3))).astype(np.float32)
            got = ops.dbscan(engine, X, 0.5, 10)
            assert np.array_equal(got, _exact_dbscan(X, 0.5, 10))
            if _min_gap_to_eps(X, 0.5) > 1e-6:
                assert np.array_equal(got, DBSCAN(eps=0.5, min_samples=10).fit(X).labels_)
    # chains at spacing exactly 0.5 along one axis, 2..11 points and one more (12 points: scikit-learn's KD tree agrees)
    for t in range(120):
        n = int(rng.integers(2, 13)) if t < 110 else 12
        off = rng.uniform(-45, 45, 3).astype(np.float32)
        k = int(rng.integers(0, 3))
        X = np.repeat(off[None], n, 0)
        X[:, k] = (off[k] + np.float32(0.5) * np.arange(n, dtype=np.float32)).astype(np.float32)
        ms = int(rng.integers(1, min(n, 10) + 1))
        got = ops.dbscan(engine, X, 0.5, ms)
        assert np.array_equal(got, _exact_dbscan(X, 0.5, ms)), (X.tolist(), ms)
        if n >= 12:
            assert np.array_equal(got, DBSCAN(eps=0.5, min_samples=ms).fit(X).labels_)
