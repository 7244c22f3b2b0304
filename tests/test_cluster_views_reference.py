"""The cluster 4-view image (LiDARAgent._generate_cluster_visualization, lidar_agent.py:241-356) against a plain restatement of the
reference's own drawing loop: NumPy for the mean, the scale and the pixels, then one filled radius-2 cv2.circle per point and view,
in draw order.  Both device entry points -- ops.cluster_views (msc_cluster_views, the mean and scale from the host) and
GeometryEngine.run_cluster_views (msc_cluster_views_batch, which gathers the rows and computes the mean and scale itself) -- must
give the restated image byte for byte, on a seeded corpus built for the edges the reference goldens miss: clusters of 1 to 100,000
rows, flat, line and single-position clusters, clusters far from the origin, isometric points outside their quadrant (discs bleeding
into the quadrants (0,1) and (1,0) and clipped at the 512 edge), isometric float pixel coordinates one float either side of -1, 0
and 256, axis-view coordinates on an integer where a fused multiply-add would truncate differently, overdraw, and intensities that are constant, negative, above 255, 1e-3 apart, up to 1e30 in size, infinite or NaN.

A NaN or infinite intensity makes the view's normalised intensities NaN, which NumPy casts to uint8 0 on the usual hosts (x86-64
and AArch64 truncate through int32) and the device's __float2int_rz turns into 0; test_restatement_pins_its_numpy_assumptions
checks the host's cast, so a host where it differs fails there rather than in an image comparison.

The isometric view: the kernels evaluate centered @ rot_x.T @ rot_y.T as explicit unfused float64 products and sums, NumPy's
matmul in its own order, so the coordinates differ in the last ulp for about a third of the points; the pixels (after
truncation) agree for every point of the corpus, which test_corpus_is_well_posed checks.  A failing image comparison says
whether its differing pixels lie where the two formulas truncate differently."""
import ctypes as C
import functools

import numpy as np
import pytest

from msc_geom import _capi
from msc_geom.lidar_agent import cluster_mosaic, cluster_view_stamp, finish_cluster_view, set_order

F32 = np.float32
SIZES = (1, 2, 5, 13, 255, 256, 257, 511, 4097, 20000, 100000)
KEY_LIMIT = (1 << 24) - 1  # the largest view the 24-bit draw-order key (rank + 1) holds


# ------------------------------------------------------------------------------------------------ restatement
def _rotations():
    ang = np.pi / 6
    rot_x = np.array([[1, 0, 0], [0, np.cos(ang), -np.sin(ang)], [0, np.sin(ang), np.cos(ang)]])
    rot_y = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
    return rot_x, rot_y


def view_coords(centered, scale, v):
    """Float pixel coordinates (x, y) of view v before the reference's astype(int): float32 for the axis views, float64 for the
    isometric one (lidar_agent.py:276-280, :322-336)."""
    if v < 3:
        a, b = [(0, 1), (0, 2), (1, 2)][v]
        return centered[:, a] * scale + 128, centered[:, b] * scale + 128
    rot_x, rot_y = _rotations()
    r = centered @ rot_x.T @ rot_y.T
    return (r[:, 0] + r[:, 1] * 0.5) * scale + 128, (r[:, 2] - r[:, 1] * 0.5) * scale + 128


def view_pixels(centered, scale, v):
    with np.errstate(invalid="ignore"):
        return tuple(c.astype(int) for c in view_coords(centered, scale, v))


def kernel_iso_pixels(centered, scale):
    """The isometric pixels as cluster_views.cu evaluates them: the same rotation written out in unfused float64 (the library is
    built with -fmad=false), in the kernel's order."""
    c, s = np.cos(np.pi / 6), np.sin(np.pi / 6)
    x, y, z = (centered[:, a].astype(np.float64) for a in range(3))
    r1y, r1z = y * c - z * s, y * s + z * c
    r2x, r2z = x * c + r1z * s, -x * s + r1z * c
    sc = np.float64(scale)
    with np.errstate(invalid="ignore"):
        return ((r2x + r1y * 0.5) * sc + 128.0).astype(int), ((r2z - r1y * 0.5) * sc + 128.0).astype(int)


def geometry(points, center=None):
    """(center, centered, scale) of lidar_agent.py:255-264; `center` overrides the mean."""
    pts = points[:, :3]
    if center is None:
        center = pts.mean(axis=0)
    centered = pts - center
    max_range = max(centered[:, 0].max() - centered[:, 0].min(), centered[:, 1].max() - centered[:, 1].min(),
                    centered[:, 2].max() - centered[:, 2].min())
    scale = (256 * 0.35) / max_range if max_range > 0 else 1
    return center, centered, scale


def reference_cluster_view(points, center=None, inten_range=None):
    """The reference's 512 x 512 image of one cluster, (n, 4) float32 rows in draw order.  `center` overrides the mean and
    inten_range[v] the (min, max) intensity of view v; both default to what these rows give."""
    import cv2
    center, centered, scale = geometry(points, center)
    grid = np.full((512, 512, 3), 255, np.uint8)
    for v in range(4):
        px, py = view_pixels(centered, scale, v)
        valid = (px >= 0) & (px < 256) & (py >= 0) & (py < 256)
        if not valid.any():
            continue
        inten = points[valid, 3]
        lo, hi = (inten.min(), inten.max()) if inten_range is None else inten_range[v]
        with np.errstate(invalid="ignore", over="ignore"):
            norm = ((inten - lo) / (hi - lo + 1e-6) * 255).astype(np.uint8)
        qx, qy = v & 1, v >> 1
        for x, y, g in zip(px[valid], py[valid], norm):
            cv2.circle(grid, (int(qx * 256 + x), int(qy * 256 + 255 - y)), 2, (int(g),) * 3, -1)
    return finish_cluster_view(grid)


# ------------------------------------------------------------------------------------------------ corpus
def _with_intensity(xyz, inten):
    return np.concatenate([np.asarray(xyz, np.float64), np.asarray(inten, np.float64).reshape(-1, 1)], 1).astype(F32)


def _blob(rng, n, centre, spread):
    return _with_intensity(rng.normal(0, 1, (n, 3)) * spread + centre, rng.uniform(0, 255, n))


def _iso_float(pts, coord):
    """Float isometric coordinate `coord` (0: x, 1: y) of the last row of pts."""
    _, centered, scale = geometry(pts)
    return float(view_coords(centered[-1:], scale, 3)[coord][0])


def _edge_probes(bulk, probe, axis, coord, target):
    """bulk + a probe row whose coordinate `axis` is one of two adjacent float32 values in [probe[axis], probe[axis] + 1], chosen
    so that the probe's isometric float coordinate `coord` lies below `target` with one and at or above it with the other (a
    bisection over the float32 values, each step evaluated with the restatement itself)."""
    def cloud(t):
        p = np.array(probe, F32)
        p[axis] = t
        return np.concatenate([bulk, p[None]])

    lo = F32(probe[axis]).view(np.int32)
    hi = F32(probe[axis] + 1).view(np.int32)
    assert lo >= 0 and _iso_float(cloud(lo.view(F32)), coord) < target <= _iso_float(cloud(hi.view(F32)), coord)
    while hi - lo > 1:
        mid = np.int32((int(lo) + int(hi)) // 2)
        if _iso_float(cloud(mid.view(F32)), coord) < target:
            lo = mid
        else:
            hi = mid
    return [cloud(lo.view(F32)), cloud(hi.view(F32))]


def _probe_clusters(rng):
    """Isometric float pixel coordinates one float either side of -1, 0 and 256, for x and for y.  The bulk fixes the mean near one
    corner of a unit cube; the probe moves along an edge that leaves the largest extent (x, 1) and so the scale alone."""
    out = []
    base = np.array([12.0, 7.0, 1.0])
    # (bulk corner, probe start, moved axis, coordinate, targets): px' = .866x + .683y + .183z, py' = z - .5x (centred, times scale)
    for corner, probe, axis, coord, targets in (((1, 1, 1), (0, 0, 0), 1, 0, (-1.0, 0.0)), ((0, 0, 0), (1, 0, 1), 1, 0, (256.0,)),
                                                ((0, 0, 1), (1, 0, 0), 2, 1, (-1.0, 0.0)), ((1, 0, 0), (0, 0, 0), 2, 1, (256.0,))):
        bulk = _with_intensity(base + corner + rng.normal(0, 2e-3, (40, 3)), rng.uniform(0, 255, 40))
        for target in targets:
            # the probe's intensity, 300, is the view's maximum only where the probe is inside the view
            for pts in _edge_probes(bulk, np.r_[base + probe, 300.0], axis, coord, target):
                out.append((f"probe_{'xy'[coord]}_{target:g}_{_iso_float(pts, coord):.6f}", pts))
    return out


def fma_axis_pixels(centered, scale):
    """Axis-view pixels as fl(c * scale + 128) rounded once (a fused multiply-add), where the reference rounds the product and then
    the sum: the two truncate differently only where the exact value sits near a float32 midpoint just below an integer."""
    s = np.longdouble(F32(scale))
    return (centered.astype(np.longdouble) * s + 128).astype(F32).astype(int)


def _axis_edge_probes(rng, keep=4):
    """Small clusters whose last row sits on an axis-view truncation edge: its float32 x pixel coordinate is the largest float
    below an integer or the integer itself (a bisection over the row's x, as _edge_probes), and `keep` where rounding the product
    and the sum once each and rounding a fused multiply-add truncate differently (found among the float32 neighbours of every
    crossing, over as many random bulks as it takes).  The row is drawn last, so its disc lies on top in views 0 and 1."""
    base = np.array([-6.0, 3.0, 0.5])
    out = []
    while len(out) < 2 + keep:
        bulk = _with_intensity(base + np.r_[[[0, 0.5, 0.5], [1, 0.5, 0.5]], rng.uniform(0, 1, (38, 3))], rng.uniform(0, 255, 40))

        def cloud(x):
            return np.concatenate([bulk, np.array([[x, base[1] + 0.5, base[2] + 0.5, 300.0]], F32)])

        def coord(x):
            _, centered, scale = geometry(cloud(x))
            return view_coords(centered[-1:], scale, 0)[0][0], fma_axis_pixels(centered[-1:, 0], scale)[0]

        lo0, hi0 = F32(base[0] + 0.1).view(np.int32), F32(base[0] + 0.9).view(np.int32)   # negative: the bits decrease with x
        for target in range(int(coord(lo0.view(F32))[0]) + 1, int(coord(hi0.view(F32))[0]) + 1):
            lo, hi = lo0, hi0
            while abs(int(hi) - int(lo)) > 1:
                mid = np.int32((int(lo) + int(hi)) // 2)
                if coord(mid.view(F32))[0] < target:
                    lo = mid
                else:
                    hi = mid
            if not out:
                out += [(f"axis_edge_{coord(b.view(F32))[0]:.6f}", cloud(b.view(F32))) for b in (lo, hi)]
            for step in range(-32, 33):
                x = np.int32(int(hi) + step).view(F32)
                c, fused = coord(x)
                if int(c) != fused and len(out) < 2 + keep:
                    out.append((f"axis_fma_{len(out) - 2}_{c:.6f}", cloud(x)))
    return out


def _interleave(rng, parts):
    """Rows of the clusters in `parts` merged in a random order that keeps each cluster's own order; returns rows and owner."""
    owner = rng.permutation(np.repeat(np.arange(len(parts)), [len(p) for p in parts]))
    rows = np.empty((len(owner), 4), F32)
    for k, p in enumerate(parts):
        rows[owner == k] = p
    return rows, owner


@functools.lru_cache(maxsize=None)
def corpus():
    """[(name, (n, 4) float32 rows)]: the seeded clusters every test here draws."""
    rng = np.random.default_rng(20261022)
    out = []
    for n in SIZES:
        out.append((f"blob_{n}", _blob(rng, n, rng.uniform(-40, 40, 3), rng.uniform(0.2, 3.0))))
    for i, n in enumerate((13, 257, 4097, 20000, 100000)):                          # one extent 0
        p = _blob(rng, n, rng.uniform(-30, 30, 3), 1.5)
        p[:, i % 3] = F32(rng.uniform(-2, 2))
        out.append((f"flat_{'xyz'[i % 3]}_{n}", p))
    for n, d in ((2, (1, 0, 0)), (5, (0, 0, 1)), (256, (1, 1, 0)), (4097, (0.3, -1, 0.2)), (100000, (-1, 0.5, 0.1))):  # lines
        t = np.sort(rng.uniform(0, 6, n)) if n > 2 else np.array([0.0, 6.0])
        out.append((f"line_{n}", _with_intensity(np.outer(t, d) + rng.uniform(-30, 30, 3), rng.uniform(0, 255, n))))
    for n in (1, 2, 256, 4097):                                                      # max_range == 0: scale 1
        out.append((f"same_{n}", _with_intensity(np.tile(rng.uniform(-45, 45, 3), (n, 1)), rng.uniform(0, 255, n))))
    for i, n in enumerate((511, 100000, 100000, 100000)):                           # far from the origin: the centring rounds
        sx, sy = (1, -1, 1, -1)[i], (1, 1, -1, -1)[i]
        out.append((f"far_{sx:+d}{sy:+d}_{n}", _blob(rng, n, (49 * sx, 49 * sy, 3), rng.uniform(0.1, 1.5))))
    # isometric: rows along (+-1, +-1, +-1), most near the start, so the far ones fall outside quadrant (1,1); those carry the
    # largest intensities, which must not enter the view's range
    for i, n in enumerate((257, 100000, 20000, 100000, 511, 100000, 4097, 13)):
        d = np.array([1 if i & 1 else -1, 1 if i & 2 else -1, 1 if i & 4 else -1], np.float64)
        t = 6.0 * rng.uniform(0, 1, n) ** 3
        xyz = np.outer(t, d) + rng.normal(0, 0.05, (n, 3)) + rng.uniform(-20, 20, 3)
        out.append((f"iso_{i}_{n}", _with_intensity(xyz, 100 * t + rng.uniform(0, 5, n))))
    out += _probe_clusters(rng)
    out += _axis_edge_probes(rng)
    # overdraw: 20 positions 0.5 m apart, each drawn 30 times with other intensities, rows 1e-4 m apart (one pixel), exact duplicates
    grid = np.stack(np.meshgrid(np.arange(5) * 0.5, np.arange(4) * 0.5, [0.0]), -1).reshape(-1, 3) + [3, -8, 1]
    reps = _with_intensity(grid[rng.integers(0, 20, 600)], rng.uniform(0, 255, 600))
    near = _with_intensity(grid[rng.integers(0, 20, 200)] + rng.uniform(0, 1e-4, (200, 3)), rng.uniform(0, 255, 200))
    over, _ = _interleave(rng, [reps, near])
    out.append(("overdraw_900", np.concatenate([over, over[rng.integers(0, 800, 100)]])))
    quant = rng.normal(0, 2.0, (3000, 3)) + [-15, 22, 0.5]
    out.append(("overdraw_100000", _with_intensity(quant[rng.integers(0, 3000, 100000)], rng.uniform(0, 255, 100000))))
    # intensities
    for name, make in (("constant", lambda n: np.full(n, 7.0)), ("negative", lambda n: rng.uniform(-100, -1, n)),
                       ("above_255", lambda n: rng.uniform(300, 5000, n)), ("spread_1e-3", lambda n: 100 + rng.uniform(0, 1e-3, n)),
                       ("huge", lambda n: rng.uniform(-1e30, 1e30, n))):
        out.append((f"intensity_{name}", _with_intensity(rng.normal(0, 1, (511, 3)) + rng.uniform(-30, 30, 3), make(511))))
    for name, special in (("inf", [np.inf]), ("-inf", [-np.inf]), ("+-inf", [np.inf, -np.inf]), ("nan", [np.nan]), ("-nan", [-np.nan])):
        p = _blob(rng, 257, rng.uniform(-30, 30, 3), 1.0)
        p[rng.integers(0, 257, 3 * len(special)), 3] = np.repeat(np.array(special, F32), 3)
        out.append((f"intensity_{name}", p))
    return out


@functools.lru_cache(maxsize=None)
def reference_images():
    return [reference_cluster_view(p) for _, p in corpus()]


def _iso_disagreements(pts):
    """Rows whose isometric pixel differs between NumPy's matmul and the kernels' explicit formula."""
    _, centered, scale = geometry(pts)
    a, b = view_pixels(centered, scale, 3), kernel_iso_pixels(centered, scale)
    return int(((a[0] != b[0]) | (a[1] != b[1])).sum())


def assert_image_equal(got, want, what, pts=None):
    if np.array_equal(got, want):
        return
    bad = (got != want).any(-1)
    ys, xs = np.nonzero(bad)
    msg = f"{what}: {int(bad.sum())} pixels differ, first at (x, y) = {list(zip(xs[:5].tolist(), ys[:5].tolist()))}"
    if pts is not None:
        iso = _iso_disagreements(pts)
        msg += f"; {iso} rows whose isometric pixel NumPy's matmul and the kernels' formula truncate differently"
        if iso == 0:
            msg += " (none: the difference is not that rounding)"
    raise AssertionError(msg)


# ------------------------------------------------------------------------------------------------ CPU
def test_restatement_pins_its_numpy_assumptions():
    """NEP 50 keeps (256 * 0.35) / max_range and the normalisation in float32; NaN casts to uint8 0 (as the device's does); NumPy's
    float32 mean along axis 0 is a sequential sum over the rows, which view_gather_kernel restates."""
    assert int(np.__version__.split(".")[0]) >= 2, np.__version__
    assert (89.6 / F32(3)).dtype == np.float32
    with np.errstate(invalid="ignore"):
        for n in (1, 7, 8, 33, 1000):
            assert not np.full(n, np.nan, F32).astype(np.uint8).any() and not np.full(n, -np.nan, F32).astype(np.uint8).any()
    for _, p in corpus():
        n = len(p)
        if n >= 4097:
            assert np.array_equal(p[:, :3].mean(axis=0), np.cumsum(p[:, :3], axis=0, dtype=F32)[-1] / F32(n))


def test_restatement_equals_the_reference_goldens(golden_dir):
    import os
    g = np.load(os.path.join(golden_dir, "cluster_views.npz"))
    for i in range(int(g["n"])):
        assert_image_equal(reference_cluster_view(g[f"pts_{i}"]), g[f"img_{i}"], i)


def test_corpus_is_well_posed():
    """The corpus reaches every edge it is built for, and the isometric pixels of NumPy's matmul and of the kernels' formula agree on
    every row of it (so exact image equality is the right bar)."""
    items = corpus()
    names = [n for n, _ in items]
    assert len(set(names)) == len(names)
    total = sum(len(p) for _, p in items)
    assert 1_000_000 <= total <= 1_600_000, total
    sizes = {len(p) for _, p in items}
    assert set(SIZES) <= sizes
    outside = bleed_01 = bleed_10 = clip_x = clip_y = 0
    coords = {"x": [], "y": []}
    for name, p in items:
        assert p.dtype == np.float32 and p.shape[1] == 4 and np.isfinite(p[:, :3]).all(), name
        assert _iso_disagreements(p) == 0, name
        _, centered, scale = geometry(p)
        px, py = view_pixels(centered, scale, 3)
        inside = (px >= 0) & (px < 256) & (py >= 0) & (py < 256)
        outside += int((~inside).sum())
        bleed_01 += int((inside & (px <= 1)).sum())        # disc reaches x = 254, 255 of quadrant (0,1)
        bleed_10 += int((inside & (py >= 254)).sum())      # disc reaches y = 254, 255 of quadrant (1,0)
        clip_x += int((inside & (px >= 254)).sum())        # disc clipped at x = 512
        clip_y += int((inside & (py <= 1)).sum())          # disc clipped at y = 512
        if name.startswith("probe"):
            coords[name[6]].append(view_coords(centered[-1:], scale, 3)["xy".index(name[6])][0])
        if name.startswith("axis"):
            c = view_coords(centered[-1:], scale, 0)[0][0]
            assert abs(c - round(c)) < 1e-4 and (int(c) != fma_axis_pixels(centered[-1:, 0], scale)[0]) == name.startswith("axis_fma"), name
    assert min(outside, bleed_01, bleed_10, clip_x, clip_y) > 0, (outside, bleed_01, bleed_10, clip_x, clip_y)
    for axis, c in coords.items():
        c = np.array(c)
        assert ((c > -2) & (c < -1)).any(), (axis, "below -1: outside")
        assert ((c > -1) & (c < 0)).any(), (axis, "in (-1, 0): truncates to 0, inside")
        assert ((c >= 0) & (c < 1e-3)).any(), (axis, "at or just above 0")
        assert ((c > 255.999) & (c < 256)).any(), (axis, "just below 256: inside")
        assert ((c >= 256) & (c < 256.001)).any(), (axis, "at or just above 256: outside")


def test_non_finite_cluster_refused_on_the_host():
    """A NaN or infinite coordinate makes the cluster's mean non-finite: the reference places none of its points (astype(int) of
    a non-finite value is INT64_MIN), so the device, whose float-to-int turns NaN into 0, must not draw it.  ops.cluster_views
    refuses such a cluster before it touches the device."""
    import types
    from msc_geom import ops
    from msc_geom.lidar_agent import LiDARAgent
    stub = types.SimpleNamespace(device="cpu")   # never reached
    good = _blob(np.random.default_rng(3), 50, (1, 2, 3), 1.0)
    for bad_value, col in ((np.nan, 0), (np.inf, 1), (-np.inf, 2), (np.nan, 2)):
        bad = good.copy()
        bad[17, col] = bad_value
        with pytest.raises(ValueError, match="not finite"):
            ops.cluster_views(stub, bad, [np.arange(50)])
        with pytest.raises(ValueError, match="not finite"):
            LiDARAgent(object(), "m", "LiDARAgent", engine=stub)._generate_cluster_visualization(bad)
        both = np.concatenate([good, bad])
        labels = np.repeat(np.int32([0, 1]), 50)
        with pytest.raises(ValueError, match="cluster 1"):
            LiDARAgent(object(), "m", "LiDARAgent", engine=stub)._cluster_visualizations(both, labels, [0, 1])
    huge = np.full((2, 4), 3e38, F32)   # finite rows whose float32 sum overflows
    with pytest.raises(ValueError, match="not finite"), np.errstate(over="ignore"):
        ops.cluster_views(stub, huge, [np.arange(2)])


# ------------------------------------------------------------------------------------------------ GPU
def _agent(engine, **kw):
    from msc_geom.lidar_agent import LiDARAgent
    return LiDARAgent(object(), "m", "LiDARAgent", engine=engine, **kw)


@functools.lru_cache(maxsize=None)
def batched_layout(seed=7, n_samples=4):
    """The corpus as one rows / labels buffer of `n_samples` samples: each sample's clusters (labelled 0.. per sample, like a
    LidarBatchResult) interleaved with each other and with noise rows (-1).  Returns rows, labels, the samples' row offsets and, per
    view, (row_begin, row_end, label, sample, corpus index): every cluster's range runs from somewhere before its first row to
    somewhere after its last, inside its sample, so ranges overlap and cover rows of other labels; the last sample's first cluster
    is viewed a second time, with the sample's whole range."""
    rng = np.random.default_rng(seed)
    items = corpus()
    sample_of = rng.integers(0, n_samples, len(items))
    rows, labels, views, off = [], [], [], [0]
    for s in range(n_samples):
        members = np.flatnonzero(sample_of == s)
        merged, owner = _interleave(rng, [items[k][1] for k in members] + [_blob(rng, 300, (0, 0, 0), 20.0)])
        lab = np.where(owner == len(members), -1, owner).astype(np.int32)
        for j, k in enumerate(members):
            at = np.flatnonzero(lab == j)
            views.append((off[-1] + int(rng.integers(0, at[0] + 1)), off[-1] + int(rng.integers(at[-1] + 1, len(lab) + 1)), j, s, int(k)))
        rows.append(merged)
        labels.append(lab)
        off.append(off[-1] + len(lab))
    views.append((off[-2], off[-1], 0, n_samples - 1, int(np.flatnonzero(sample_of == n_samples - 1)[0])))
    return np.concatenate(rows), np.concatenate(labels), np.array(off), np.array(views, np.int64)


@pytest.mark.gpu
def test_single_path_equals_the_restatement(engine):
    """agent._generate_cluster_visualization on every cluster, and agent._cluster_visualizations (one launch of all a sample's
    clusters, gathered from interleaved labels) on every sample of batched_layout."""
    agent = _agent(engine)
    items, want = corpus(), reference_images()
    for (name, p), w in zip(items, want):
        assert_image_equal(agent._generate_cluster_visualization(p), w, name, p)
    rows, labels, off, views = batched_layout()
    for s in range(len(off) - 1):
        vs = views[(views[:, 3] == s)][:, [2, 4]]
        got = agent._cluster_visualizations(rows[off[s]:off[s + 1]], labels[off[s]:off[s + 1]], [int(l) for l in vs[:, 0]])
        assert len(got) == len(vs) >= 3
        for g, (_, k) in zip(got, vs):
            assert_image_equal(g, want[k], ("sample", s, items[k][0]), items[k][1])


@pytest.mark.gpu
def test_batched_path_equals_the_restatement(engine, monkeypatch):
    """run_cluster_views on batched_layout, nine views per call."""
    import torch
    from msc_geom import engine as engine_mod
    items, want = corpus(), reference_images()
    rows, labels, _, views = batched_layout()
    n = len(views)
    per = int(engine.lib.msc_cluster_views_batch_workspace_bytes(1, int((views[:, 1] - views[:, 0]).max())))
    monkeypatch.setattr(engine_mod, "CLUSTER_VIEWS_WORKSPACE_PER_CALL", 9 * per)
    t_rows, t_labels = torch.from_numpy(rows).to(engine.device), torch.from_numpy(labels).to(engine.device)
    launches = engine.kernel_launches
    got = engine.run_cluster_views(t_rows, t_labels, views[:, :3]).to_host()
    assert engine.kernel_launches - launches == 6 * ((n + 8) // 9) and n > 27
    for i, k in enumerate(views[:, 4]):
        assert_image_equal(got[i], want[k], ("view", i, items[k][0]), items[k][1])


@pytest.mark.gpu
def test_oversized_view_is_isolated(engine):
    """msc_cluster_views_batch with one view above max_view_points among ordinary ones, every range the whole buffer: the status
    is set, to_host raises, the oversized view comes out empty (axes and titles on white), every other view is still exact, and
    sentinel images on either side of the output are untouched."""
    import torch
    from msc_geom.engine import ClusterViewsResult
    items, want = corpus(), reference_images()
    names = [n for n, _ in items]
    picks = [names.index(n) for n in ("blob_4097", "iso_7_13", "blob_20000", "overdraw_900", "line_256")]
    parts = [items[k][1] for k in picks]
    rows = np.concatenate(parts)
    labels = np.repeat(np.arange(len(parts), dtype=np.int32), [len(p) for p in parts])
    n, maxp = len(parts), 4097
    views = np.array([(0, len(rows), j) for j in range(n)], np.int32)
    dev = engine.device
    t_rows, t_labels = torch.from_numpy(rows).to(dev), torch.from_numpy(labels).to(dev)
    out = torch.full((n + 2, 512, 512, 3), 0xA5, dtype=torch.uint8, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    need = int(engine.lib.msc_cluster_views_batch_workspace_bytes(n, maxp))
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    stamp = torch.from_numpy(cluster_view_stamp().view(np.int32)).to(dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = engine.lib.msc_cluster_views_batch(t_rows.data_ptr(), t_labels.data_ptr(), views.ctypes.data, n, maxp, stamp.data_ptr(), stamp.shape[0],
                                            out[1].data_ptr(), status.data_ptr(), ws.data_ptr(), need, stream)
    assert rc == 0
    assert int(status.item()) == 1
    with pytest.raises(_capi.MscError, match="max_view_points"):
        ClusterViewsResult(n, out[1:n + 1], status).to_host()
    host = out.cpu().numpy()
    assert (host[0] == 0xA5).all() and (host[n + 1] == 0xA5).all()
    for j, k in enumerate(picks):
        if len(items[k][1]) > maxp:
            assert_image_equal(host[1 + j], finish_cluster_view(np.full((512, 512, 3), 255, np.uint8)), "oversized view")
        else:
            assert_image_equal(host[1 + j], want[k], items[k][0], items[k][1])


def _key_limit_view(seed=24):
    """KEY_LIMIT rows drawn from 3,000 positions in a seeded random order (every position occurs), with their own intensities, and
    the restated image: copies of one position cover the same pixels, so the image is that of each position's last occurrence, in
    the order of last occurrences, drawn with the mean and the views' intensity ranges of all rows."""
    rng = np.random.default_rng(seed)
    n_pos = 3000
    pos = rng.normal(0, 0.5, (n_pos, 3)) + [20, -5, 1]
    pos[:40] = [20, -5, 1] + np.outer(rng.uniform(8, 12, 40), (1, 1, 1))   # some outside the isometric view
    pos = pos.astype(F32)
    idx = rng.integers(0, n_pos, KEY_LIMIT)
    idx[rng.choice(KEY_LIMIT, n_pos, replace=False)] = np.arange(n_pos)
    rows = np.empty((KEY_LIMIT, 4), F32)
    rows[:, :3] = pos[idx]
    rows[:, 3] = rng.uniform(-50, 300, KEY_LIMIT)
    center = rows[:, :3].mean(axis=0)
    last = np.sort(KEY_LIMIT - 1 - np.unique(idx[::-1], return_index=True)[1])
    _, centered, scale = geometry(pos, center)
    ranges = []
    for v in range(4):
        px, py = view_pixels(centered, scale, v)
        valid = ((px >= 0) & (px < 256) & (py >= 0) & (py < 256))[idx]
        assert valid.any() and (v < 3 or not valid.all())
        ranges.append((rows[valid, 3].min(), rows[valid, 3].max()))
    assert len(last) == n_pos and last[-1] == KEY_LIMIT - 1
    return rows, reference_cluster_view(rows[last], center=center, inten_range=ranges)


@pytest.mark.gpu
def test_largest_view_the_draw_order_key_holds(engine):
    """One view of 2^24 - 1 rows, max_view_points = 2^24 - 1, through both entry points."""
    import torch
    rows, want = _key_limit_view()
    assert_image_equal(_agent(engine)._generate_cluster_visualization(rows), want, "single path")
    t_rows = torch.from_numpy(rows).to(engine.device)
    t_labels = torch.zeros(KEY_LIMIT, dtype=torch.int32, device=engine.device)
    got = engine.run_cluster_views(t_rows, t_labels, [(0, KEY_LIMIT, 0)], max_view_points=KEY_LIMIT).to_host()
    assert_image_equal(got[0], want, "batched path")


@pytest.mark.gpu
def test_agent_images_and_mosaics_equal_the_restatement(engine):
    """process_batch on synthetic samples with many clusters: every image the classifier is handed equals the restated image of
    its cluster (obj[labels == l] of run_lidar's rows), every mosaic cluster_mosaic of the restated images, both as arrays and,
    with png=True, as the device-drawn mosaic's PNG."""
    import base64
    import io
    from PIL import Image
    from msc_geom.layout import pack_batch
    from msc_geom.synthetic import make_sample
    from tests.test_lidar_batch import _Recorder
    samples = [make_sample(i, n_sweeps=1, n_boxes=40) for i in (5, 6, 7)]
    plain = _agent(engine)
    per = engine.run_lidar(engine.upload(pack_batch(samples)), params=plain._params(), eps=plain.dbscan_eps,
                           min_samples=plain.dbscan_min_samples).to_host()
    batches = []
    for r in per:
        if len(r["object"]) < plain.dbscan_min_samples:
            continue
        order = [l for l in set_order(r["cluster_first"], r["noise_first"]) if int(r["clusters"][l, 10]) >= 5]
        images = [reference_cluster_view(r["object"][r["labels"] == l]) for l in order]
        batches += [images[a:a + 10] for a in range(0, len(images), 10)]
    assert sum(len(b) for b in batches) >= 30 and len(batches) >= 4
    rec, rec_png = _Recorder(), _Recorder()
    _agent(engine, cluster_classifier=rec.classifier).process_batch(samples)
    _agent(engine, cluster_classifier=rec_png.classifier).process_batch(samples, png=True)
    assert len(rec.calls) == len(rec_png.calls) == len(batches)
    for c, ((images, mosaic, _), (none, png, _), want) in enumerate(zip(rec.calls, rec_png.calls, batches)):
        assert len(images) == len(want) and none is None
        for i, (g, w) in enumerate(zip(images, want)):
            assert_image_equal(g, w, ("call", c, "image", i))
        assert_image_equal(mosaic, cluster_mosaic(want), ("call", c, "mosaic"))
        decoded = np.asarray(Image.open(io.BytesIO(base64.b64decode(png))).convert("RGB"))[..., ::-1]
        assert_image_equal(decoded, cluster_mosaic(want), ("call", c, "png mosaic"))


@pytest.mark.gpu
def test_non_finite_cluster_refused_on_the_device_path(engine):
    """_generate_cluster_visualization refuses a cluster with one NaN or one infinite row, and still draws the finite cluster."""
    agent = _agent(engine)
    name, p = corpus()[0 + SIZES.index(257)]
    for value in (np.nan, np.inf):
        bad = p.copy()
        bad[100, 1] = value
        with pytest.raises(ValueError, match="not finite"):
            agent._generate_cluster_visualization(bad)
    assert_image_equal(agent._generate_cluster_visualization(p), reference_images()[SIZES.index(257)], name, p)
