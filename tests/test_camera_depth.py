"""[EXT] row e7, LiDAR -> camera projection (msc_camera_depth_batch, csrc/camera_depth.cu; definition in tests/depth_oracle.c).

CPU part: the oracle against an independent devkit-style NumPy restatement (from_file_multisweep, then map_pointcloud_to_image),
the oracle's exact edges on a hand-built rig, and the ctypes structs.  GPU part: the kernels bit for bit against the oracle, the
support counts against the box projection and a NumPy count over the device's own depth maps, order / partition independence,
interaction with the fused pass, the error paths and the host evidence."""
import json

import numpy as np
import pytest

from msc_geom import _capi
from msc_geom.geometry import rot_to_quat
from msc_geom.layout import DepthParams, GeomParams, HostBatch, pack_batch
from msc_geom.synthetic import make_sample
from tests import depth_oracle as DO
from tests.oracle_bridge import oracle_project

W, H = 1600, 900


# ------------------------------------------------------------------------------------------------ devkit-style NumPy restatement
def _qrot(q):
    """pyquaternion's Quaternion(q).rotation_matrix (normalised first)."""
    w, x, y, z = (float(v) for v in q)
    n = np.sqrt(w * w + x * x + y * y + z * z)
    w, x, y, z = w / n, x / n, y / n, z / n
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _transform_matrix(pose, inverse=False):
    R, t, T = _qrot(pose[3:]), np.asarray(pose[:3], np.float64), np.eye(4)
    T[:3, :3], T[:3, 3] = (R.T, R.T @ -t) if inverse else (R, t)
    return T


def devkit_multisweep(sample):
    """LidarPointCloud.from_file_multisweep: (4, N) f32 cloud in the keyframe LIDAR_TOP frame and, per column, its row in the
    concatenated raw sweeps."""
    clouds, rows, off = [], [], 0
    for sw in sample["lidar_sweeps"]:
        pts = np.asarray(sw["points_raw"], np.float32)[:, :4].T.copy()
        keep = ~((np.abs(pts[0]) < 1.0) & (np.abs(pts[1]) < 1.0))  # remove_close(1.0)
        pts = pts[:, keep]
        M = (_transform_matrix(sample["lidar_calib"], True) @ _transform_matrix(sample["ego_pose"], True) @ _transform_matrix(sw["ego_pose"])
             @ _transform_matrix(sw["calib"]))
        pts[:3, :] = M.dot(np.vstack((pts[:3, :], np.ones(pts.shape[1]))))[:3, :]  # stored back into the f32 cloud
        clouds.append(pts)
        rows.append(np.nonzero(keep)[0] + off)
        off += keep.size
    return np.concatenate(clouds, 1), np.concatenate(rows)


def devkit_map_to_image(pc, sample, cam, dtype=np.float32, min_dist=1.0):
    """NuScenesExplorer.map_pointcloud_to_image for one camera: (u, v, depth, mask, |global coordinate| per point).  dtype=float32
    stores the cloud back after every rotate / translate like LidarPointCloud; float64 keeps the whole chain in f64."""
    p = pc.astype(dtype, copy=True)

    def rotate(R):
        p[:3, :] = np.dot(R, p[:3, :])

    def translate(t):
        for i in range(3):
            p[i, :] = p[i, :] + t[i]
    rotate(_qrot(sample["lidar_calib"][3:])); translate(sample["lidar_calib"][:3])
    rotate(_qrot(sample["ego_pose"][3:])); translate(sample["ego_pose"][:3])
    gmax = np.abs(p[:3]).max(0)
    translate(-np.asarray(cam["ego_pose"][:3])); rotate(_qrot(cam["ego_pose"][3:]).T)
    translate(-np.asarray(cam["calib"][:3])); rotate(_qrot(cam["calib"][3:]).T)
    depths = p[2, :]
    viewpad = np.eye(4)
    viewpad[:3, :3] = cam["intrinsic"]
    q = np.dot(viewpad, np.concatenate((p[:3, :], np.ones((1, p.shape[1])))))[:3, :]
    q = q / q[2:3, :].repeat(3, 0).reshape(3, -1)
    mask = (depths > min_dist) & (q[0] > 1) & (q[0] < W - 1) & (q[1] > 1) & (q[1] < H - 1)
    return q[0], q[1], depths, mask, gmax


def _edge_distance(u, v):
    """px distance to the nearest mask bound or pixel edge."""
    d = lambda a, lo, hi: np.minimum(np.minimum(np.abs(a - lo), np.abs(a - hi)), np.abs(a - np.round(a)))
    return np.minimum(d(u, 1, W - 1), d(v, 1, H - 1))


@pytest.mark.parametrize("n_sweeps", [1, 10])
def test_oracle_matches_devkit_restatement(n_sweeps):
    """The (camera, pixel) of every return and the block minima agree with the devkit's arithmetic.

    Against the chain in f64 a return may land differently only within 1e-3 px of a mask bound or pixel edge, or within 1e-6 m of
    min_dist.  The devkit's own LidarPointCloud stores the cloud in f32 after every step, also in the global frame, where nuScenes-
    scale coordinates (hundreds of metres) have an ulp of up to 1.2e-4 m; against that chain the allowance adds 2 f ulp(|global|) / Z
    px per return.  Seeds 1 and 10 sweeps: 1 and 18 returns (of 28k / 290k hits) within 1e-3 px of an edge against the f64 chain,
    42 and 512 against the f32 chain, none outside the allowance."""
    s = make_sample(3, n_sweeps=n_sweeps)
    hb = pack_batch([s])
    ds = 8
    depth, cp, pix = DO.camera_depth(hb, 0, ds=ds, with_pixels=True)
    pc, rows = devkit_multisweep(s)
    counts = {}
    for ci, cam in enumerate(s["cameras"]):
        got = pix[rows, ci]
        assert int(cp[ci]) == int((pix[:, ci] >= 0).sum())
        for dt in (np.float64, np.float32):
            u, v, dep, m, gmax = devkit_map_to_image(pc, s, cam, dt)
            ref = np.full(rows.size, -1, np.int64)
            ref[m] = v[m].astype(np.int64) * W + u[m].astype(np.int64)
            mis = ref != got
            tol = 1e-3
            if dt == np.float32:
                tol = 1e-3 + 2 * cam["intrinsic"][0, 0] * np.spacing(gmax.astype(np.float32)).astype(np.float64) / np.maximum(np.abs(dep), 1e-3)
            near = (_edge_distance(u, v) <= tol) | (np.abs(dep.astype(np.float64) - 1.0) <= 1e-6)
            assert not (mis & ~near).any(), (cam["channel"], np.dtype(dt).name, int((mis & ~near).sum()))
            counts[(ci, np.dtype(dt).name)] = int(mis.sum())
            if dt == np.float64:
                # block minima wherever no exceptional return is involved
                Hb, Wb = depth.shape[1:]
                blk = lambda pixel: (pixel // W // ds) * Wb + (pixel % W) // ds
                bad_blocks = np.unique(np.concatenate([blk(ref[mis & (ref >= 0)]), blk(got[mis & (got >= 0)])]))
                mind = np.full(Hb * Wb, np.inf)
                np.minimum.at(mind, blk(ref[m]), dep[m])
                mind[bad_blocks] = np.nan
                ok = ~np.isnan(mind)
                o = depth[ci].reshape(-1).astype(np.float64)
                assert np.array_equal(np.isinf(o[ok]), np.isinf(mind[ok]))
                fin = ok & np.isfinite(mind)
                assert fin.sum() > 100
                np.testing.assert_allclose(o[fin], mind[fin], rtol=1e-5)
    total_hits = int(cp.sum())
    assert sum(v for (c, k), v in counts.items() if k == "float64") <= 1e-3 * total_hits
    assert sum(v for (c, k), v in counts.items() if k == "float32") <= 1e-2 * total_hits


# ------------------------------------------------------------------------------------------------ exact rig
_R_CAM = np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])  # camera (x right, y down, z forward) -> ego


def exact_rig_sample(points):
    """One sample whose every step is exact: integer translations that cancel, axis-permutation rotations (quaternion components 0,
    +-0.5, +-1) and K = diag(2, 2, 1).  cam_from_ref is then X = -y, Y = -z, Z = x, so u = -2y / x, v = -2z / x, w = x."""
    ident = np.array([1.0, 0.0, 0.0, 0.0])
    ego = np.concatenate([[100.0, -50.0, 0.0], [0.0, 0.0, 0.0, 1.0]])   # 180 degrees about z
    lcal = np.concatenate([[2.0, 3.0, 5.0], ident])
    cam = {"channel": "CAM_EXACT", "ego_pose": ego, "calib": np.concatenate([[2.0, 3.0, 5.0], rot_to_quat(_R_CAM)]),
           "intrinsic": np.diag([2.0, 2.0, 1.0])}
    raw = np.zeros((len(points), 5), np.float32)
    raw[:, :3] = np.asarray(points, np.float32)
    sweep = {"points_raw": raw, "ref_from_sensor": np.eye(4)[:3], "ego_pose": ego, "calib": lcal, "time_lag": 0.0}
    return {"lidar_sweeps": [sweep], "ego_pose": ego, "lidar_calib": lcal, "cameras": [cam], "annotations": []}


def _up(x):
    return float(np.nextafter(np.float32(x), np.float32(np.inf)))


def _dn(x):
    return float(np.nextafter(np.float32(x), np.float32(-np.inf)))


# (x, y, z) in the sweep frame -> expected pixel (px, py) or None
EDGE_POINTS = [
    ((2.0, -1.0, -450.0), None), ((2.0, -_up(1.0), -450.0), (1, 450)),          # u = 1 out, next float in
    ((2.0, -1599.0, -450.0), None), ((2.0, -_dn(1599.0), -450.0), (1598, 450)),  # u = W - 1
    ((2.0, -800.0, -1.0), None), ((2.0, -800.0, -_up(1.0)), (800, 1)),            # v = 1
    ((2.0, -800.0, -899.0), None), ((2.0, -800.0, -_dn(899.0)), (800, 898)),      # v = H - 1
    ((1.0, -400.0, -225.0), None), ((_up(1.0), -400.0, -225.0), (799, 449)),      # w = min_dist = 1 out, next float in
    ((-2.0, 800.0, 450.0), None),                                                 # behind the camera (would land at (800, -450) / w)
    ((float("nan"), -800.0, -450.0), None), ((2.0, float("nan"), -450.0), None), ((2.0, -800.0, float("nan")), None),
    ((2.0, -1598.5, -898.5), (1598, 898)),                                        # last partial block row and column with ds = 7
    ((4.0, -6.0, -8.0), (3, 4)),
]


def test_exact_rig_matrix():
    s = exact_rig_sample([(2.0, -800.0, -450.0)])
    P = DO.camera_matrix(s["ego_pose"], s["lidar_calib"], s["cameras"][0]["ego_pose"], s["cameras"][0]["calib"], s["cameras"][0]["intrinsic"])
    assert np.array_equal(P, np.array([[0, -2, 0, 0], [0, 0, -2, 0], [1, 0, 0, 0]], np.float32))


@pytest.mark.parametrize("ds", [1, 7, 8])
def test_oracle_exact_edges(ds):
    s = exact_rig_sample([p for p, _ in EDGE_POINTS])
    hb = pack_batch([s], n_cams=1)
    depth, cp, pix = DO.camera_depth(hb, 0, ds=ds, with_pixels=True)
    for r, (p, want) in enumerate(EDGE_POINTS):
        assert pix[r, 0] == (-1 if want is None else want[1] * W + want[0]), (p, want, pix[r, 0])
    assert cp[0] == sum(w is not None for _, w in EDGE_POINTS)
    Hb, Wb = DO.block_shape(W, H, ds)
    assert depth.shape == (1, Hb, Wb)
    exp = np.full((Hb, Wb), np.inf, np.float32)
    for p, want in EDGE_POINTS:
        if want is not None:
            exp[want[1] // ds, want[0] // ds] = min(exp[want[1] // ds, want[0] // ds], np.float32(p[0]))
    assert np.array_equal(depth[0], exp)
    if ds == 7:
        assert np.isfinite(depth[0, Hb - 1, Wb - 1]) and (Hb, Wb) == (129, 229)


def test_oracle_support_at_margin_bounds():
    """A box with camera-frame Z in [8, 12] and margin 0.5: blocks at exactly 7.5 are on the box, one float nearer hide it; 12.5 is on
    the box, one float further is only a hit; +inf is no hit."""
    s = exact_rig_sample([(2.0, -800.0, -450.0)])
    cam = s["cameras"][0]
    # global box: identity rotation, l = 4 along global x -> camera Z = 98 - gx in [8, 12]; X = gy + 53 in [399, 401]; Y = 5 - gz
    box = np.array([[88.0, 347.0, -2245.0, 2.0, 4.0, 2.0, 1.0, 0.0, 0.0, 0.0]])
    pose, calib, K = cam["ego_pose"][None], cam["calib"][None], cam["intrinsic"].reshape(1, 9)
    vis, ext = oracle_project(box, pose, calib, K, W, H)
    assert vis[0, 0] == 1
    ds = 8
    Hb, Wb = DO.block_shape(W, H, ds)
    bx0, bx1 = int(ext[0, 0, 0]) // ds, min(int(ext[0, 0, 2]), W - 1) // ds
    by0, by1 = int(ext[0, 0, 1]) // ds, min(int(ext[0, 0, 3]), H - 1) // ds
    classes = [(_dn(7.5), "front"), (7.5, "on"), (12.5, "on"), (_up(12.5), "hit"), (np.inf, "none"), (10.0, "on"), (0.25, "front")]
    depth = np.full((1, Hb, Wb), np.inf, np.float32)
    want = {"front": 0, "on": 0, "hit": 0, "none": 0}
    k = 0
    for by in range(by0, by1 + 1):
        for bx in range(bx0, bx1 + 1):
            val, cls = classes[k % len(classes)]
            depth[0, by, bx] = val
            want[cls] += 1
            k += 1
    depth[0, by0 - 1, bx0] = 0.1  # outside the extent: not counted
    got = DO.box_support(box, pose, calib, K, depth, W, H, ds, 0.5)
    n_hit = want["front"] + want["on"] + want["hit"]
    assert got[0, 0].tolist() == [k, n_hit, want["front"], want["on"]]
    hidden = box.copy(); hidden[0, 1] = 347.0 + 10000.0  # off-image: all four 0
    assert DO.box_support(hidden, pose, calib, K, depth, W, H, ds, 0.5)[0, 0].tolist() == [0, 0, 0, 0]


def test_struct_sizes_match_header():
    import ctypes
    assert ctypes.sizeof(_capi.MscDepthParams) == 12
    assert ctypes.sizeof(_capi.MscDepthOut) == 3 * 8
    assert [f for f, _ in _capi.MscDepthParams._fields_] == ["min_dist", "downsample", "support_margin"]
    assert [f for f, _ in _capi.MscDepthOut._fields_] == ["depth", "cam_points", "box_support"]


# ------------------------------------------------------------------------------------------------ GPU
def _eight_cams(s):
    """The six-camera rig plus two narrower cameras (other focal length and principal point)."""
    extra = []
    for base, f in ((0, 2000.0), (3, 600.0)):
        c = dict(s["cameras"][base])
        c = {**c, "channel": c["channel"] + "_X", "intrinsic": np.array([[f, 0, 700.0], [0, f, 420.0], [0, 0, 1.0]])}
        extra.append(c)
    return {**s, "cameras": s["cameras"] + extra}


def mixed_batch(n_cams=6):
    """12 samples: 1-10 sweeps, 0 / 1 / 60 / 120 boxes, an empty sweep in the middle of a sample and a sample with no rows."""
    spec = [(1, 0), (10, 60), (3, 1), (7, 120), (2, 60), (5, 0), (10, 120), (4, 1), (6, 60), (8, 60), (2, 1), (1, 60)]
    samples = []
    for i, (ns, nb) in enumerate(spec):
        s = make_sample(700 + i, n_sweeps=ns, n_boxes=nb)
        if i == 4:
            s["lidar_sweeps"][1]["points_raw"] = np.zeros((0, 5), np.float32)
        if i == 10:
            for sw in s["lidar_sweeps"]:
                sw["points_raw"] = np.zeros((0, 5), np.float32)
        if n_cams == 8:
            s = _eight_cams(s)
        samples.append(s)
    return samples


def _run(eng, db, p, dp, box_support=True):
    import torch
    res = eng.run_camera_depth(db, eng.alloc_depth(db.host, dp, p, box_support), dp, p)
    torch.cuda.synchronize()
    return res.to_host()


def _assert_equal_to_oracle(got, hb, p, dp):
    D, CP, BS = DO.batch(hb, p.image_w, p.image_h, p.n_cams, dp.min_dist, dp.downsample, dp.support_margin, p.remove_close_radius)
    assert np.array_equal(got["depth"].view(np.uint32), D.view(np.uint32))
    assert np.array_equal(got["cam_points"], CP)
    if "box_support" in got:
        assert np.array_equal(got["box_support"], BS)
    return D, CP, BS


@pytest.fixture(scope="module")
def eng():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from msc_geom.engine import GeometryEngine
    return GeometryEngine(0)


@pytest.mark.gpu
@pytest.mark.parametrize("n_cams,ds", [(6, 8), (6, 4), (6, 7), (1, 8), (8, 8), (8, 7)])
def test_gpu_bit_exact_mixed_batch(eng, n_cams, ds):
    samples = mixed_batch(n_cams)
    if n_cams == 1:
        samples = [{**s, "cameras": s["cameras"][3:4]} for s in samples]
    hb = pack_batch(samples, n_cams=n_cams)
    p, dp = GeomParams(n_cams=n_cams), DepthParams(downsample=ds)
    got = _run(eng, eng.upload(hb), p, dp)
    D, CP, BS = _assert_equal_to_oracle(got, hb, p, dp)
    assert CP[10].sum() == 0 and np.isinf(D[10]).all()
    assert CP.sum() > 0 and (BS[..., 1] > 0).any() and (BS[..., 2] > 0).any() and (BS[..., 3] > 0).any()


@pytest.mark.gpu
def test_gpu_bit_exact_full_resolution(eng):
    """downsample 1: one depth value per pixel (1600 x 900 per camera)."""
    hb = pack_batch([make_sample(720, n_sweeps=10, n_boxes=60)])
    p, dp = GeomParams(), DepthParams(downsample=1)
    got = _run(eng, eng.upload(hb), p, dp)
    assert got["depth"].shape == (1, 6, 900, 1600)
    _assert_equal_to_oracle(got, hb, p, dp)


@pytest.mark.gpu
@pytest.mark.parametrize("ds", [1, 7])
def test_gpu_exact_rig_edges(eng, ds):
    s = exact_rig_sample([p for p, _ in EDGE_POINTS])
    hb = pack_batch([s], n_cams=1)
    p, dp = GeomParams(n_cams=1), DepthParams(downsample=ds)
    got = _run(eng, eng.upload(hb), p, dp)
    _assert_equal_to_oracle(got, hb, p, dp)
    assert got["cam_points"][0, 0] == sum(w is not None for _, w in EDGE_POINTS)


def _numpy_support(hb, depth, vis, ext, n_cams, ds, margin):
    """The support counts restated in NumPy over given depth maps, with the visible flag / extent of msc_project_boxes and Z range
    of the 8 corners in the order of project_box."""
    out = np.zeros((hb.n_boxes, n_cams, 4), np.uint32)
    Hb, Wb = depth.shape[2:]
    for s in range(hb.n_samples):
        for b in range(int(hb.sample_box_off[s]), int(hb.sample_box_off[s + 1])):
            box = hb.boxes[b]
            for c in range(n_cams):
                if not vis[b, c]:
                    continue
                ctr = box[:3].copy()
                R = _qrot_f(box[6:10])
                for pose in (hb.cam_ego_pose[s, c], hb.cam_calib[s, c]):
                    ctr, R = _frame_change(pose, ctr, R)
                hl, hw, hh = box[4] / 2.0, box[3] / 2.0, box[5] / 2.0
                Z = [((R[6] * lx + R[7] * ly) + R[8] * lz) + ctr[2] for lx in (hl, -hl) for ly in (hw, -hw) for lz in (hh, -hh)]
                e = ext[b, c]
                bx0, bx1 = int(e[0]) // ds, min(int(e[2]), W - 1) // ds
                by0, by1 = int(e[1]) // ds, min(int(e[3]), H - 1) // ds
                d = depth[s, c, by0:by1 + 1, bx0:bx1 + 1].astype(np.float64)
                hit = np.isfinite(d)
                front = hit & (d < min(Z) - margin)
                on = hit & ~front & (d <= max(Z) + margin)
                out[b, c] = [d.size, hit.sum(), front.sum(), on.sum()]
    return out


def _qrot_f(q):
    w, x, y, z = (float(v) for v in q)
    n = np.sqrt(((w * w + x * x) + y * y) + z * z)
    w, x, y, z = w / n, x / n, y / n, z / n
    xx, yy, zz, xy, xz, yz, wx, wy, wz = x * x, y * y, z * z, x * y, x * z, y * z, w * x, w * y, w * z
    return [1.0 - 2.0 * (yy + zz), 2.0 * (xy - wz), 2.0 * (xz + wy), 2.0 * (xy + wz), 1.0 - 2.0 * (xx + zz), 2.0 * (yz - wx),
            2.0 * (xz - wy), 2.0 * (yz + wx), 1.0 - 2.0 * (xx + yy)]


def _frame_change(pose, c, R):
    P = _qrot_f(pose[3:])
    d = [c[0] - pose[0], c[1] - pose[1], c[2] - pose[2]]
    c2 = [(P[0 + r] * d[0] + P[3 + r] * d[1]) + P[6 + r] * d[2] for r in range(3)]
    R2 = [(P[0 + r] * R[0 + k] + P[3 + r] * R[3 + k]) + P[6 + r] * R[6 + k] for r in range(3) for k in range(3)]
    return np.array(c2), R2


@pytest.mark.gpu
def test_gpu_support_matches_projection_and_numpy(eng):
    import torch
    from msc_geom import ops
    samples = mixed_batch(6)
    hb = pack_batch(samples)
    p, dp = GeomParams(), DepthParams(downsample=8)
    got = _run(eng, eng.upload(hb), p, dp)
    vis = np.zeros((hb.n_boxes, 6), np.uint8); ext = np.zeros((hb.n_boxes, 6, 4), np.float32)
    for s in range(hb.n_samples):
        b0, b1 = int(hb.sample_box_off[s]), int(hb.sample_box_off[s + 1])
        if b1 > b0:
            vis[b0:b1], ext[b0:b1] = ops.project_boxes(eng, hb.boxes[b0:b1], hb.cam_ego_pose[s], hb.cam_calib[s], hb.cam_K[s])
    bs = got["box_support"]
    assert np.array_equal(bs[..., 0] > 0, vis.astype(bool))
    assert np.array_equal(bs, _numpy_support(hb, got["depth"], vis, ext, 6, 8, 0.5))
    torch.cuda.synchronize()


def _permute_rows(hb: HostBatch, seed=5) -> HostBatch:
    rng = np.random.default_rng(seed)
    pts = hb.points.copy()
    for st, n in zip(hb.sweep_start, hb.sweep_count):
        st, n = int(st), int(n)
        pts[st:st + n] = pts[st:st + n][rng.permutation(n)]
    return HostBatch(hb.n_samples, pts, hb.sample_sweep_off, hb.sweep_start, hb.sweep_count, hb.sweep_pose, hb.sweep_time_lag,
                     hb.sample_box_off, hb.boxes, hb.ego_pose, hb.lidar_calib, hb.cam_ego_pose, hb.cam_calib, hb.cam_K, hb.n_cams,
                     hb.max_boxes_per_sample)


@pytest.mark.gpu
def test_gpu_order_and_partition_independence(eng):
    import ctypes as C
    import torch
    samples = mixed_batch(6)
    hb = pack_batch(samples)
    p, dp = GeomParams(), DepthParams(downsample=8)
    db = eng.upload(hb)
    a = _run(eng, db, p, dp)
    b = _run(eng, db, p, dp)
    c = _run(eng, eng.upload(_permute_rows(hb)), p, dp)
    for r in (b, c):
        for k in ("depth", "cam_points", "box_support"):
            assert np.array_equal(a[k].view(np.uint32), r[k].view(np.uint32)), k
    # sample by sample
    for i, s in enumerate(samples):
        one = _run(eng, eng.upload(pack_batch([s])), p, dp)
        b0, b1 = int(hb.sample_box_off[i]), int(hb.sample_box_off[i + 1])
        assert np.array_equal(one["depth"][0].view(np.uint32), a["depth"][i].view(np.uint32))
        assert np.array_equal(one["cam_points"][0], a["cam_points"][i])
        assert np.array_equal(one["box_support"], a["box_support"][b0:b1])
    # other launch partitions: the points-per-sample hint sets the CTAs per sample (1 ... 4096)
    for hint in (1, 20000, 2 ** 30):
        out = eng.alloc_depth(hb, dp, p)
        st = db.struct()
        bi = _capi.MscBatchIn(*[getattr(st, f) for f, _ in _capi.MscBatchIn._fields_])
        bi.points_per_sample_hint = hint
        stream = torch.cuda.current_stream().cuda_stream
        _capi.check(eng.lib.msc_camera_depth_batch(C.byref(eng_params(p)), C.byref(_capi.MscDepthParams(1.0, 8, 0.5)), C.byref(bi),
                                                   C.byref(out.struct()), C.c_void_p(stream)), "msc_camera_depth_batch")
        torch.cuda.synchronize()
        h = out.to_host()
        for k in ("depth", "cam_points", "box_support"):
            assert np.array_equal(a[k].view(np.uint32), h[k].view(np.uint32)), (hint, k)


def eng_params(p):
    from msc_geom.engine import make_params
    return make_params(p)


@pytest.mark.gpu
def test_gpu_fused_unchanged_around_camera_depth(eng):
    import torch
    hb = pack_batch(mixed_batch(6))
    db = eng.upload(hb)
    before = eng.run_fused(db).to_host()
    _run(eng, db, GeomParams(), DepthParams())
    after = eng.run_fused(db).to_host()
    torch.cuda.synchronize()
    for k in before:
        assert np.array_equal(np.asarray(before[k]), np.asarray(after[k])), k


@pytest.mark.gpu
def test_gpu_error_paths(eng):
    import ctypes as C
    import torch
    hb = pack_batch([make_sample(730, n_sweeps=1, n_boxes=3)])
    db = eng.upload(hb)
    p = GeomParams()
    out = eng.alloc_depth(hb, DepthParams(), p)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(mp=None, dp=None, bi=None, bo=None):
        mp = mp or eng_params(p)
        dp = dp or _capi.MscDepthParams(1.0, 8, 0.5)
        return eng.lib.msc_camera_depth_batch(C.byref(mp), C.byref(dp), C.byref(bi or db.struct()), C.byref(bo or out.struct()), stream)

    def refused(what, **kw):
        rc = call(**kw)
        assert rc == _capi.MSC_ERR_BAD_ARGUMENT, what
        assert what in eng.lib.msc_last_error().decode(), (what, eng.lib.msc_last_error())
    refused("downsample", dp=_capi.MscDepthParams(1.0, 0, 0.5))
    for nc in (0, 9):
        refused("n_cams", mp=eng_params(GeomParams(n_cams=nc)))
    refused("image_w", mp=eng_params(GeomParams(image_w=2)))
    refused("image_w", mp=eng_params(GeomParams(image_h=1)))
    refused("support_margin", dp=_capi.MscDepthParams(1.0, 8, float("nan")))
    refused("support_margin", dp=_capi.MscDepthParams(1.0, 8, -0.5))
    refused("min_dist", dp=_capi.MscDepthParams(float("nan"), 8, 0.5))
    refused("must not be NULL", bo=_capi.MscDepthOut(None, out.cam_points.data_ptr(), None))
    refused("must not be NULL", bo=_capi.MscDepthOut(out.depth.data_ptr(), None, None))
    # through the engine: MscError with the library's message
    with pytest.raises(_capi.MscError, match="downsample") as ei:
        eng.run_camera_depth(db, dp=DepthParams(downsample=0))
    assert ei.value.status == _capi.MSC_ERR_BAD_ARGUMENT
    # n_samples = 0: success, nothing launched, NULL outputs allowed
    empty = pack_batch([])
    n0 = eng.kernel_launches
    bi = db.struct()
    bi0 = _capi.MscBatchIn(*[getattr(bi, f) for f, _ in _capi.MscBatchIn._fields_])
    bi0.n_samples = 0
    assert call(bi=bi0, bo=_capi.MscDepthOut(None, None, None)) == 0
    res = eng.run_camera_depth(eng.upload(empty))
    assert eng.kernel_launches == n0 and res.depth.numel() == 0
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_gpu_lidar_evidence_and_context(eng):
    from msc_geom import camera_agent, ops, serialize
    s = make_sample(740, n_sweeps=10, n_boxes=60)
    ev = camera_agent.lidar_evidence(eng, s)
    assert json.loads(json.dumps(ev)) == ev
    res = ops.camera_depth(eng, s)
    hb = pack_batch([s])
    D, CP, BS = DO.batch(hb)
    assert np.array_equal(res["depth"].view(np.uint32), D[0].view(np.uint32)) and np.array_equal(res["box_support"], BS)
    for ci, cam in enumerate(s["cameras"]):
        e = ev[cam["channel"]]
        assert e["lidar_returns"] == int(CP[0, ci])
        assert [o["annotation"] for o in e["objects"]] == [int(i) for i in np.nonzero(BS[:, ci, 0])[0]]
        for o in e["objects"]:
            assert [o["blocks"], o["blocks_with_returns"], o["occluded"], o["on_object"]] == BS[o["annotation"], ci].tolist()
    base = camera_agent.evidence_context(eng, s)
    assert camera_agent.evidence_context(eng, s, lidar=False) == base == {"box_projection": camera_agent.projection_evidence(eng, s)}
    ctx = camera_agent.evidence_context(eng, s, lidar=True)
    assert ctx["box_projection"] == base["box_projection"] and ctx["lidar_in_camera"] == ev
    seen = []
    llm = lambda messages, **kw: seen.append(messages[0]["content"][0]["text"]) or ""
    camera_agent.CameraAgent(None, "m", "camera", engine=eng, llm=llm).process([], [], sample=s)
    camera_agent.CameraAgent(None, "m", "camera", engine=eng, llm=llm, lidar=True).process([], [], sample=s)
    assert seen[0] == camera_agent.CameraAgent.context_block(base)["text"]
    assert seen[1] == camera_agent.CameraAgent.context_block(ctx)["text"]
    fused = eng.process_samples([s])
    names = [c["channel"] for c in s["cameras"]]
    args = (s["annotations"], fused["box_count"], fused["box_nearest"], fused["box_centroid"], fused["proj_visible"], names)
    plain = serialize.ext_evidence(*args)
    assert serialize.ext_evidence(*args, camera_support=None) == plain
    withs = serialize.ext_evidence(*args, camera_support=res["box_support"])
    assert json.loads(json.dumps(withs)) == withs
    for i, o in enumerate(withs["objects"]):
        assert {k: v for k, v in o.items() if k != "lidar_in_camera"} == plain["objects"][i]
        assert sorted(o["lidar_in_camera"]) == sorted(n for c, n in enumerate(names) if BS[i, c, 0])
