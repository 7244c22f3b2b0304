"""Thin host wrappers over the single-sample / small-table entry points of the C-ABI (include/msc_geom.h).
Inputs and outputs are NumPy arrays on the host (the reference's functions take and return NumPy); device buffers
are torch tensors that live for the duration of the call."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _capi
from .engine import GeometryEngine, make_params
from .layout import GeomParams


def _stream(eng: GeometryEngine):
    return C.c_void_p(torch.cuda.current_stream(eng.device).cuda_stream)


def _raw_rows(pc: np.ndarray) -> Tuple[np.ndarray, int]:
    """Return a C-contiguous float32 buffer and its row pitch (floats) for an (N, >=4) cloud WITHOUT repacking the
    devkit's 20-byte-pitch view (nuscenes_loader.py:152-155: (N,5)[:, :4] seen through two transposes)."""
    pc = np.asarray(pc)
    if pc.dtype != np.float32:
        pc = pc.astype(np.float32)
    n = pc.shape[0]
    if n == 0:
        return np.zeros((0, 4), np.float32), 4
    if pc.flags["C_CONTIGUOUS"]:
        return pc, pc.shape[1]
    if pc.ndim == 2 and pc.strides[1] == 4 and pc.strides[0] % 4 == 0 and pc.strides[0] // 4 >= pc.shape[1]:
        pitch = pc.strides[0] // 4
        base = pc
        while isinstance(base.base, np.ndarray):
            base = base.base
        lo = base.__array_interface__["data"][0]
        hi = lo + base.nbytes
        start = pc.__array_interface__["data"][0]
        if lo <= start and start + n * pitch * 4 <= hi:
            return np.lib.stride_tricks.as_strided(pc, shape=(n, pitch), strides=(pitch * 4, 4)), pitch
    return np.ascontiguousarray(pc), pc.shape[1]


def keyframe_filter_split(eng: GeometryEngine, pc: np.ndarray, params: Optional[GeomParams] = None, split_only: bool = False):
    """LiDARAgent._preprocess_point_cloud + _segment_ground (lidar_agent.py:103-132): kept, ground, object as (n,4) f32."""
    p = params or GeomParams(bev_res=800)
    rows, pitch = _raw_rows(pc)
    n = rows.shape[0]
    d = eng.device
    if n == 0:
        z = np.zeros((0, 4), np.float32)
        return z, z.copy(), z.copy()
    src = torch.from_numpy(np.ascontiguousarray(rows)).to(d)
    kept = torch.empty((n, 4), dtype=torch.float32, device=d)
    ground = torch.empty((n, 4), dtype=torch.float32, device=d)
    obj = torch.empty((n, 4), dtype=torch.float32, device=d)
    counts = torch.zeros(3, dtype=torch.int32, device=d)
    n_blocks = (n + 1023) // 1024
    scratch = torch.empty(n_blocks * 2 + 2, dtype=torch.int32, device=d)
    mp = make_params(p)
    _capi.check(eng.lib.msc_keyframe_filter_split(C.byref(mp), src.data_ptr(), n, pitch, int(split_only), kept.data_ptr(), ground.data_ptr(), obj.data_ptr(),
                                                  counts.data_ptr(), scratch.data_ptr(), scratch.numel(), _stream(eng)), "msc_keyframe_filter_split")
    eng.kernel_launches += 3
    nk, ng, no = (int(v) for v in counts.cpu().tolist())
    return kept[:nk].cpu().numpy(), ground[:ng].cpu().numpy(), obj[:no].cpu().numpy()


def keyframe_bev_layers(eng: GeometryEngine, ground: np.ndarray, obj: np.ndarray, res: int = 800, bev_range: float = 50.0):
    """Raster half of _generate_multi_layer_bev (lidar_agent.py:539-597): count u32, height f32, semantic BGR u8 (unflipped)."""
    p = GeomParams(bev_res=res, bev_range=bev_range)
    d = eng.device
    g = torch.from_numpy(np.ascontiguousarray(ground[:, :4], np.float32)).to(d) if len(ground) else torch.zeros((1, 4), device=d)
    o = torch.from_numpy(np.ascontiguousarray(obj[:, :4], np.float32)).to(d) if len(obj) else torch.zeros((1, 4), device=d)
    count = torch.empty((res, res), dtype=torch.int32, device=d)
    height = torch.empty((res, res), dtype=torch.float32, device=d)
    sem = torch.empty((res, res, 3), dtype=torch.uint8, device=d)
    winner = torch.empty((res, res), dtype=torch.int32, device=d)
    zr = torch.empty(2, dtype=torch.int32, device=d)
    mp = make_params(p)
    _capi.check(eng.lib.msc_keyframe_bev(C.byref(mp), g.data_ptr(), len(ground), o.data_ptr(), len(obj), count.data_ptr(), height.data_ptr(),
                                         sem.data_ptr(), winner.data_ptr(), zr.data_ptr(), _stream(eng)), "msc_keyframe_bev")
    eng.kernel_launches += 2
    return count.cpu().numpy().view(np.uint32), height.cpu().numpy(), sem.cpu().numpy()


def cloud_stats(eng: GeometryEngine, pc: np.ndarray):
    """RawGPT4oBaseline._describe_point_cloud numbers (baseline_gpt4o.py:276-285): (min3, max3, mean radial distance)."""
    rows, pitch = _raw_rows(pc)
    n = rows.shape[0]
    if n == 0:
        return None
    src = torch.from_numpy(np.ascontiguousarray(rows)).to(eng.device)
    out = torch.zeros(7, dtype=torch.float64, device=eng.device)
    _capi.check(eng.lib.msc_cloud_stats(src.data_ptr(), n, pitch, out.data_ptr(), _stream(eng)), "msc_cloud_stats")
    eng.kernel_launches += 2
    o = out.cpu().numpy()
    return o[:3].astype(np.float32), o[3:6].astype(np.float32), float(o[6] / n)


def cluster_aabb(eng: GeometryEngine, pts: np.ndarray, labels: np.ndarray, n_clusters: int) -> np.ndarray:
    """Per-cluster min3, max3, center3, distance, num_points (lidar_agent.py:200-204) for DBSCAN labels."""
    if n_clusters == 0:
        return np.zeros((0, 11), np.float32)
    rows, pitch = _raw_rows(pts)
    src = torch.from_numpy(np.ascontiguousarray(rows)).to(eng.device)
    lab = torch.from_numpy(np.ascontiguousarray(labels, np.int32)).to(eng.device)
    out = torch.empty((n_clusters, 11), dtype=torch.float32, device=eng.device)
    _capi.check(eng.lib.msc_cluster_aabb(src.data_ptr(), rows.shape[0], pitch, lab.data_ptr(), n_clusters, out.data_ptr(), _stream(eng)),
                "msc_cluster_aabb")
    eng.kernel_launches += 3
    return out.cpu().numpy()


def annotation_table(eng: GeometryEngine, xy: np.ndarray, vel: np.ndarray) -> Dict[str, np.ndarray]:
    """Numeric half of SceneGraphAgent._parse_annotations / _build_spatial_zones (scenegraph_agent.py:186-225, :281-295)."""
    n = int(xy.shape[0])
    d = eng.device
    if n == 0:
        return {"distance": np.zeros(0), "direction": np.zeros(0, np.uint8), "moving": np.zeros(0, np.uint8), "zone": np.zeros(0, np.uint8),
                "region_bits": np.zeros(0, np.uint8)}
    x = torch.from_numpy(np.ascontiguousarray(xy, np.float64)).to(d)
    v = torch.from_numpy(np.ascontiguousarray(vel, np.float64)).to(d)
    dist = torch.empty(n, dtype=torch.float64, device=d)
    u8 = [torch.empty(n, dtype=torch.uint8, device=d) for _ in range(4)]
    _capi.check(eng.lib.msc_annotation_table(n, x.data_ptr(), v.data_ptr(), dist.data_ptr(), *[t.data_ptr() for t in u8], _stream(eng)),
                "msc_annotation_table")
    eng.kernel_launches += 1
    return {"distance": dist.cpu().numpy(), "direction": u8[0].cpu().numpy(), "moving": u8[1].cpu().numpy(), "zone": u8[2].cpu().numpy(),
            "region_bits": u8[3].cpu().numpy()}


def relation_table(eng: GeometryEngine, boxes: np.ndarray, ego_pose: Optional[np.ndarray] = None) -> Dict[str, np.ndarray]:
    """[EXT] pairwise relations (distance, bearing, 4-way category, footprint overlap) between n annotation boxes."""
    n = int(boxes.shape[0])
    d = eng.device
    if n == 0:
        z = np.zeros((0, 0))
        return {"dist": z.astype(np.float32), "bearing": z.astype(np.float32), "category": z.astype(np.uint8), "overlap": z.astype(np.uint8), "rect": np.zeros((0, 6))}
    b = torch.from_numpy(np.ascontiguousarray(boxes, np.float64)).to(d)
    rect = torch.empty((n, 6), dtype=torch.float64, device=d)
    ego = None if ego_pose is None else torch.from_numpy(np.ascontiguousarray(ego_pose, np.float64)).to(d)
    _capi.check(eng.lib.msc_box_footprints(n, b.data_ptr(), ego.data_ptr() if ego is not None else None, rect.data_ptr(), _stream(eng)), "msc_box_footprints")
    dist = torch.empty((n, n), dtype=torch.float32, device=d)
    bearing = torch.empty((n, n), dtype=torch.float32, device=d)
    cat = torch.empty((n, n), dtype=torch.uint8, device=d)
    ov = torch.empty((n, n), dtype=torch.uint8, device=d)
    _capi.check(eng.lib.msc_relation_table(n, rect.data_ptr(), dist.data_ptr(), bearing.data_ptr(), cat.data_ptr(), ov.data_ptr(), _stream(eng)),
                "msc_relation_table")
    eng.kernel_launches += 2
    return {"dist": dist.cpu().numpy(), "bearing": bearing.cpu().numpy(), "category": cat.cpu().numpy(), "overlap": ov.cpu().numpy(),
            "rect": rect.cpu().numpy()}


def project_boxes(eng: GeometryEngine, boxes: np.ndarray, cam_ego_pose: np.ndarray, cam_calib: np.ndarray, cam_K: np.ndarray, image_w=1600, image_h=900):
    """[EXT] box -> camera projection for one sample: visible [B,C] u8, extent [B,C,4] f32."""
    nb, nc = int(boxes.shape[0]), int(cam_calib.shape[0])
    d = eng.device
    if nb == 0 or nc == 0:
        return np.zeros((nb, nc), np.uint8), np.zeros((nb, nc, 4), np.float32)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float64)).to(d)
    b, p, c, k = t(boxes), t(cam_ego_pose), t(cam_calib), t(np.asarray(cam_K).reshape(nc, 9))
    vis = torch.empty((nb, nc), dtype=torch.uint8, device=d)
    ext = torch.empty((nb, nc, 4), dtype=torch.float32, device=d)
    _capi.check(eng.lib.msc_project_boxes(nb, b.data_ptr(), nc, p.data_ptr(), c.data_ptr(), k.data_ptr(), image_w, image_h, vis.data_ptr(),
                                          ext.data_ptr(), _stream(eng)), "msc_project_boxes")
    eng.kernel_launches += 1
    return vis.cpu().numpy(), ext.cpu().numpy()


def aggregate_sweeps(eng: GeometryEngine, sweeps, remove_close_radius: float = 1.0):
    """[EXT] devkit LidarPointCloud.from_file_multisweep (App. A.1): sweeps = [(raw (n,5) f32, M 3x4 f64, time_lag)];
    returns (N,4) f32 rows x', y', z', intensity and (N,) f32 time lags, order-preserving."""
    if not sweeps:
        return np.zeros((0, 4), np.float32), np.zeros(0, np.float32)
    d = eng.device
    counts = np.array([s[0].shape[0] for s in sweeps], np.uint32)
    starts = np.zeros(len(sweeps), np.uint32)
    starts[1:] = np.cumsum(counts)[:-1]
    total = int(counts.sum())
    if total == 0:
        return np.zeros((0, 4), np.float32), np.zeros(0, np.float32)
    pts = torch.from_numpy(np.ascontiguousarray(np.concatenate([np.asarray(s[0], np.float32) for s in sweeps], 0))).to(d)
    pose = torch.from_numpy(np.ascontiguousarray(np.stack([np.asarray(s[1], np.float64).reshape(-1)[:12] for s in sweeps]))).to(d)
    lag = torch.from_numpy(np.array([s[2] for s in sweeps], np.float32)).to(d)
    st = torch.from_numpy(starts.view(np.int32)).to(d)
    ct = torch.from_numpy(counts.view(np.int32)).to(d)
    max_pts = int(counts.max())
    n_blocks = (len(sweeps) * max_pts + 1023) // 1024
    scratch = torch.empty(n_blocks * 2 + 8, dtype=torch.int32, device=d)
    out = torch.empty((total, 4), dtype=torch.float32, device=d)
    out_t = torch.empty(total, dtype=torch.float32, device=d)
    n_out = torch.zeros(1, dtype=torch.int32, device=d)
    _capi.check(eng.lib.msc_aggregate_sweeps(C.c_float(remove_close_radius), pts.data_ptr(), len(sweeps), st.data_ptr(), ct.data_ptr(), pose.data_ptr(),
                                             lag.data_ptr(), max_pts, out.data_ptr(), out_t.data_ptr(), n_out.data_ptr(), scratch.data_ptr(),
                                             scratch.numel(), _stream(eng)), "msc_aggregate_sweeps")
    eng.kernel_launches += 3
    m = int(n_out.item())
    return out[:m].cpu().numpy(), out_t[:m].cpu().numpy()


def cluster_views(eng: GeometryEngine, points: np.ndarray, clusters) -> np.ndarray:
    """Point discs of LiDARAgent._generate_cluster_visualization (lidar_agent.py:241-351) for a list of clusters of one cloud.
    points: (N,4) f32; clusters: list of index arrays into points (original order inside a cluster).  Returns u8
    [K,512,512,3] without axes / titles (see lidar_agent.finish_cluster_view).  The cluster mean and pixel scale are
    evaluated on the host with NumPy exactly as the reference does (:255-264) -- a few hundred floats per cluster."""
    K = len(clusters)
    if K == 0:
        return np.zeros((0, 512, 512, 3), np.uint8)
    d = eng.device
    pts = np.ascontiguousarray(points[:, :4], np.float32)
    cs = np.zeros((K, 4), np.float32)
    off = np.zeros(K + 1, np.int32)
    for k, idx in enumerate(clusters):
        cp = pts[idx, :3]
        center = cp.mean(axis=0)
        centered = cp - center
        max_range = max(centered[:, 0].max() - centered[:, 0].min(), centered[:, 1].max() - centered[:, 1].min(),
                        centered[:, 2].max() - centered[:, 2].min())
        cs[k, :3] = center
        cs[k, 3] = (256 * 0.35) / max_range if max_range > 0 else 1
        off[k + 1] = off[k] + len(idx)
    order = np.concatenate([np.asarray(i, np.int64) for i in clusters]).astype(np.uint32)
    t_pts = torch.from_numpy(pts).to(d)
    t_order = torch.from_numpy(order.view(np.int32)).to(d)
    t_off = torch.from_numpy(off).to(d)
    t_cs = torch.from_numpy(cs).to(d)
    keys = torch.empty((K, 512, 512), dtype=torch.int32, device=d)
    irange = torch.empty((K, 4, 2), dtype=torch.int32, device=d)
    out = torch.empty((K, 512, 512, 3), dtype=torch.uint8, device=d)
    max_n = int(np.diff(off).max())
    _capi.check(eng.lib.msc_cluster_views(t_pts.data_ptr(), t_order.data_ptr(), t_off.data_ptr(), K, max_n, t_cs.data_ptr(), keys.data_ptr(),
                                          irange.data_ptr(), out.data_ptr(), _stream(eng)), "msc_cluster_views")
    eng.kernel_launches += 2
    return out.cpu().numpy()


def dbscan(eng: GeometryEngine, xyz: np.ndarray, eps: float = 0.5, min_samples: int = 10) -> np.ndarray:
    """sklearn.cluster.DBSCAN(eps, min_samples).fit(xyz).labels_ (lidar_agent.py:148-153), computed on the device with
    scikit-learn's labelling rule (see csrc/dbscan.cu).  Returns int64 labels like scikit-learn.

    Neighbours are the pairs with (dx^2 + dy^2) + dz^2 <= eps^2 in float64, scikit-learn's KD-tree rule.  The labels equal
    scikit-learn's for 12 or more points.  For 11 or fewer scikit-learn searches by brute force, whose BLAS distance can drop a
    pair at exactly eps; there the labels equal scikit-learn's when no pair is within 1e-6 of eps, and follow the rule above
    otherwise."""
    rows, pitch = _raw_rows(xyz)
    n = int(rows.shape[0])
    if n == 0:
        return np.zeros(0, np.int64)
    if not np.isfinite(rows[:, :3]).all():  # scikit-learn's check_array raises on NaN / inf input too
        raise ValueError("Input X contains NaN or infinity (DBSCAN needs finite coordinates, like sklearn.cluster.DBSCAN.fit).")
    lo = rows[:, :3].min(axis=0).astype(np.float64)
    hi = rows[:, :3].max(axis=0).astype(np.float64)
    cell = float(eps) * (1.0 + 1e-6)  # a hair above eps so float rounding can never put neighbours two cells apart
    while True:
        dims = np.maximum(np.floor((hi - lo) / cell).astype(np.int64) + 1, 1)
        if int(dims.prod()) <= (1 << 24):
            break
        cell *= 2.0  # coarser cells stay correct (cell >= eps), only slower
    d = eng.device
    src = torch.from_numpy(np.ascontiguousarray(rows)).to(d)
    labels = torch.empty(n, dtype=torch.int32, device=d)
    c_dims = (C.c_int32 * 3)(*[int(v) for v in dims])
    c_org = (C.c_double * 3)(*[float(v) for v in lo])
    need = int(eng.lib.msc_dbscan_workspace_bytes(n, c_dims))
    ws = torch.empty(need, dtype=torch.uint8, device=d)
    k = C.c_int32(0)
    _capi.check(eng.lib.msc_dbscan(src.data_ptr(), n, pitch, C.c_double(float(eps)), int(min_samples), c_org, C.c_double(cell), c_dims,
                                   labels.data_ptr(), C.byref(k), ws.data_ptr(), need, _stream(eng)), "msc_dbscan")
    eng.kernel_launches += 8
    return labels.cpu().numpy().astype(np.int64)


def decode_jpeg_batch(eng: GeometryEngine, streams, threads: int = 8, to_host: bool = True):
    """Decode JPEG byte strings exactly like `np.array(PIL.Image.open(...))` (NuScenesLoader._load_camera, nuscenes_loader.py:136-144):
    the Huffman decode of every image runs on a host thread (ctypes releases the GIL), coefficients go to the device in one copy per
    image, dequantisation + IDCT + chroma upsampling + colour conversion run there.  Returns uint8 arrays (H, W, 3) -- (H, W) for
    grayscale files -- on the host, or device tensors with to_host=False."""
    from concurrent.futures import ThreadPoolExecutor
    lib = eng.lib
    bufs = [np.frombuffer(s, dtype=np.uint8) if not isinstance(s, np.ndarray) else s for s in streams]
    descs, coefs = [], []
    for b in bufs:
        d = _capi.MscJpegDesc()
        _capi.check(lib.msc_jpeg_info(b.ctypes.data, b.size, C.byref(d)), "msc_jpeg_info")
        descs.append(d)
        coefs.append(torch.empty(int(d.coef_elems), dtype=torch.int16).pin_memory())

    def entropy(i):
        return lib.msc_jpeg_entropy_decode_host(bufs[i].ctypes.data, bufs[i].size, C.byref(descs[i]), coefs[i].data_ptr())
    if len(bufs) > 1 and threads > 1:
        with ThreadPoolExecutor(max_workers=min(threads, len(bufs))) as pool:
            rcs = list(pool.map(entropy, range(len(bufs))))
    else:
        rcs = [entropy(i) for i in range(len(bufs))]
    for rc in rcs:
        _capi.check(rc, "msc_jpeg_entropy_decode_host")
    outs = []
    for d, c in zip(descs, coefs):
        cd = c.to(eng.device, non_blocking=True)
        planes = torch.empty(int(d.plane_bytes), dtype=torch.uint8, device=eng.device)
        shape = (d.height, d.width, 3) if d.n_comp == 3 else (d.height, d.width)
        out = torch.empty(shape, dtype=torch.uint8, device=eng.device)
        _capi.check(lib.msc_jpeg_reconstruct(C.byref(d), cd.data_ptr(), planes.data_ptr(), out.data_ptr(), _stream(eng)), "msc_jpeg_reconstruct")
        outs.append(out)
    if not to_host:
        return outs
    return [o.cpu().numpy() for o in outs]


def decode_jpeg(eng: GeometryEngine, stream) -> np.ndarray:
    return decode_jpeg_batch(eng, [stream], threads=1)[0]
