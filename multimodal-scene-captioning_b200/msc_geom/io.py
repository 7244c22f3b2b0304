"""On-disk format step (SURVEY.md section 8(f) rank 3): nuScenes `.pcd.bin` sweeps -> the fused kernel's batch layout.

The reference reads one keyframe per sample through the devkit (`LidarPointCloud.from_file`: np.fromfile -> reshape(-1,5)[:, :4].T,
then `.T` again, src/nuscenes_loader.py:146-157) and its evaluator loads every sample of every scene once just to collect tokens
(src/evaluation_framework.py:488-496).  Here the raw 5-float rows are read with `readinto` straight into their final place in one
staging buffer (pinned when a CUDA device is present) -- no intermediate arrays, no repack -- by a small thread pool (file reads
release the GIL), and scenes can be scanned for tokens without touching sensor data.
"""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, List, Optional, Sequence

import numpy as np

from .layout import HostBatch, N_CAMS_DEFAULT, boxes_from_annotations

ROW_BYTES = 20  # x, y, z, intensity, ring as float32


def pcd_bin_points(path: str) -> int:
    """Number of points in a .pcd.bin file (size / 20 bytes); raises on a truncated file."""
    size = os.path.getsize(path)
    if size % ROW_BYTES:
        raise ValueError(f"{path}: size {size} is not a multiple of {ROW_BYTES} bytes")
    return size // ROW_BYTES


def read_pcd_bin_into(path: str, dst_rows: np.ndarray) -> None:
    """Read a .pcd.bin file into `dst_rows` ((n,5) float32, C-contiguous view of the staging buffer) without a temporary."""
    buf = memoryview(dst_rows).cast("B")
    with open(path, "rb", buffering=0) as f:
        got = 0
        while got < len(buf):
            k = f.readinto(buf[got:])
            if not k:
                raise IOError(f"{path}: short read ({got} of {len(buf)} bytes)")
            got += k


def stage_batch(samples: Sequence[dict], n_cams: int = N_CAMS_DEFAULT, threads: int = 8, pinned: Optional[bool] = None,
                pool: Optional["PinnedPool"] = None) -> HostBatch:
    """Build a HostBatch whose sweeps come from files.  Each sample is a dict shaped like the loader's, where a sweep is
    {"path": <.pcd.bin>, "ref_from_sensor": 3x4 f64, "time_lag": s} (or carries "points_raw" already in memory).  The `points`
    buffer is allocated once (pinned host memory when CUDA is available, unless `pinned=False`; taken from `pool` when one is given,
    so consecutive batches reuse the same page-locked memory) and files are read into it in place."""
    S = len(samples)
    sweeps = [(i, sw) for i, s in enumerate(samples) for sw in s["lidar_sweeps"]]
    counts = np.array([pcd_bin_points(sw["path"]) if "path" in sw else int(np.asarray(sw["points_raw"]).shape[0]) for _, sw in sweeps], np.uint32)
    starts = np.zeros(len(sweeps), np.uint32)
    cursor = 0
    for k, c in enumerate(counts):
        starts[k] = cursor
        cursor += (int(c) + 3) & ~3
    n_rows = cursor + 4
    if pinned is None:
        try:
            import torch
            pinned = torch.cuda.is_available()
        except Exception:
            pinned = False
    if pool is not None:
        holder = pool.take(n_rows)
        points = holder.numpy()
    elif pinned:
        import torch
        holder = torch.empty((n_rows, 5), dtype=torch.float32).pin_memory()
        points = holder.numpy()
    else:
        holder = None
        points = np.empty((n_rows, 5), np.float32)
    # padding rows (between sweeps and at the tail) must fail every compare
    for k in range(len(sweeps)):
        a, c = int(starts[k]) + int(counts[k]), (int(starts[k + 1]) if k + 1 < len(sweeps) else cursor)
        points[a:c] = np.nan
    points[cursor:] = np.nan

    def load(k):
        sw = sweeps[k][1]
        dst = points[int(starts[k]): int(starts[k]) + int(counts[k])]
        if "path" in sw:
            read_pcd_bin_into(sw["path"], dst)
        else:
            dst[:] = sw["points_raw"]

    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(load, range(len(sweeps))))
    sample_sweep_off = np.zeros(S + 1, np.int32)
    for i, _ in sweeps:
        sample_sweep_off[i + 1] += 1
    sample_sweep_off = np.cumsum(sample_sweep_off).astype(np.int32)
    pose = np.stack([np.asarray(sw["ref_from_sensor"], np.float64).reshape(-1)[:12] for _, sw in sweeps]) if sweeps else np.zeros((0, 12))
    lag = np.array([float(sw.get("time_lag", 0.0)) for _, sw in sweeps], np.float32)
    box_arrays = [boxes_from_annotations(s.get("annotations", [])) for s in samples]
    sample_box_off = np.zeros(S + 1, np.int32)
    sample_box_off[1:] = np.cumsum([b.shape[0] for b in box_arrays])
    boxes = np.ascontiguousarray(np.concatenate(box_arrays, 0) if box_arrays else np.zeros((0, 10)), np.float64).reshape(-1, 10)
    ident = np.array([0, 0, 0, 1, 0, 0, 0.0])
    ego = np.stack([np.asarray(s.get("ego_pose", ident), np.float64) for s in samples]) if S else np.zeros((0, 7))
    lcal = np.stack([np.asarray(s.get("lidar_calib", ident), np.float64) for s in samples]) if S else np.zeros((0, 7))
    cam_pose = np.zeros((S, n_cams, 7)); cam_cal = np.zeros((S, n_cams, 7)); cam_K = np.zeros((S, n_cams, 9))
    cam_pose[..., 3] = 1.0; cam_cal[..., 3] = 1.0
    cam_K[..., 0] = cam_K[..., 4] = cam_K[..., 8] = 1.0
    for i, s in enumerate(samples):
        for c, cam in enumerate(s.get("cameras", [])[:n_cams]):
            cam_pose[i, c] = cam.get("ego_pose", ego[i]); cam_cal[i, c] = cam["calib"]; cam_K[i, c] = np.asarray(cam["intrinsic"], np.float64).reshape(-1)
    hb = HostBatch(S, points, sample_sweep_off, starts, counts, np.ascontiguousarray(pose, np.float64), lag, sample_box_off, boxes, ego, lcal,
                   cam_pose, cam_cal, cam_K, n_cams, int(max([b.shape[0] for b in box_arrays], default=0)))
    hb._pinned_holder = holder  # keeps the pinned allocation alive with the batch
    return hb


class StagedCameras:
    """The camera files of a batch in one host byte buffer (see stage_camera_files).  File k is data[file_off[k]:file_off[k] + size[k]],
    plans[k] its msc_jpeg_plan and index[k] its (sample, camera) position; `unsupported` lists the (sample, camera, path) the planner
    refused as MSC_ERR_UNSUPPORTED (progressive, 12-bit, CMYK ...), which are not in the buffer."""

    def __init__(self, data, holder, file_off, size, plans, index, unsupported, n_cams):
        self.data, self._holder, self.file_off, self.size = data, holder, file_off, size
        self.plans, self.index, self.unsupported, self.n_cams = plans, index, unsupported, n_cams
        self.nbytes = int(file_off[-1] + size[-1]) if len(size) else 0

    def __len__(self):
        return len(self.index)


def stage_camera_files(samples: Sequence[dict], threads: int = 8, pool: Optional["PinnedPool"] = None, pinned: Optional[bool] = None) -> StagedCameras:
    """Read every camera file of a batch (the `path` of each entry of a sample's `cameras`, as NuScenesLoader(lazy_sweeps=True) records
    it) with `readinto` into one byte buffer -- pinned when CUDA is available unless `pinned=False`, taken from `pool` when one is given --
    and plan each file's decode (msc_jpeg_decode_plan).  Files start at 256-byte offsets.  A file the planner refuses as
    MSC_ERR_UNSUPPORTED is listed in `unsupported`; any other planner error raises MscError."""
    import ctypes as C
    from . import _capi
    lib = _capi.load()
    files = [(i, c, cam["path"]) for i, s in enumerate(samples) for c, cam in enumerate(s.get("cameras", []))]
    sizes = np.array([os.path.getsize(p) for _, _, p in files], np.int64)
    offs = np.zeros(len(files), np.int64)
    cursor = 0
    for k, n in enumerate(sizes):
        offs[k] = cursor
        cursor += (int(n) + 255) & ~255
    total = max(cursor, 256)
    if pinned is None:
        try:
            import torch
            pinned = torch.cuda.is_available()
        except Exception:
            pinned = False
    if pool is not None:
        holder = pool.take((total + 19) // 20)
        data = holder.numpy().view(np.uint8).reshape(-1)[:total]
    elif pinned:
        import torch
        holder = torch.empty(total, dtype=torch.uint8).pin_memory()
        data = holder.numpy()
    else:
        holder = None
        data = np.empty(total, np.uint8)
    plans = (_capi.MscJpegPlan * max(len(files), 1))()
    rcs = [0] * len(files)

    def load(k):
        dst = data[int(offs[k]): int(offs[k]) + int(sizes[k])]
        read_pcd_bin_into(files[k][2], dst)
        rcs[k] = lib.msc_jpeg_decode_plan(dst.ctypes.data, int(sizes[k]), C.byref(plans[k]))

    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(load, range(len(files))))
    keep, unsupported = [], []
    for k, rc in enumerate(rcs):
        if rc == _capi.MSC_ERR_UNSUPPORTED:
            unsupported.append(files[k])
        elif rc != 0:
            raise _capi.MscError(f"{files[k][2]}: msc_jpeg_decode_plan failed with status {rc}", rc)
        else:
            keep.append(k)
    kept_plans = (_capi.MscJpegPlan * max(len(keep), 1))()
    for j, k in enumerate(keep):
        kept_plans[j] = plans[k]
    return StagedCameras(data, holder, offs[keep], sizes[keep], kept_plans, [files[k][:2] for k in keep], unsupported,
                         [len(s.get("cameras", [])) for s in samples])


def write_pcd_bin(path: str, rows: np.ndarray) -> None:
    """Write (n,5) float32 rows in the nuScenes .pcd.bin layout (used by tests and synthetic datasets)."""
    np.ascontiguousarray(rows, np.float32).tofile(path)


class PinnedPool:
    """Grow-only pool of pinned host buffers for stage_batch: a loader that stages batch after batch reuses the same page-locked
    allocations instead of paying cudaHostAlloc per batch (slots rotate so a buffer is not rewritten while its upload is in flight)."""

    def __init__(self, slots: int = 3):
        self.slots = [None] * slots
        self.k = 0
        self.allocations = 0

    def take(self, n_rows: int):
        import torch
        i = self.k % len(self.slots)
        self.k += 1
        buf = self.slots[i]
        if buf is None or buf.shape[0] < n_rows:
            buf = self.slots[i] = torch.empty((int(n_rows * 1.25) + 64, 5), dtype=torch.float32).pin_memory()
            self.allocations += 1
        return buf[:n_rows]


def write_nuscenes_tree(root: str, scenes: Sequence[Sequence[dict]], version: str = "v1.0-mini", jpeg_quality: int = 90) -> Dict[str, int]:
    """Write samples (dicts shaped like msc_geom.synthetic.make_sample's) as an on-disk dataset with the nuScenes layout: the relational
    JSON tables under <root>/<version>/ (scene, sample, sample_data, ego_pose, calibrated_sensor, sensor, sample_annotation, instance,
    category, attribute, visibility, log, map) and the sensor files under samples/ (keyframes) and sweeps/ (intermediate LIDAR_TOP sweeps,
    chained through sample_data.prev / next like the real dataset).  For tests and benchmarks of the on-disk step -- there is no dataset
    offline.  Returns table sizes."""
    import json
    from PIL import Image
    T: Dict[str, list] = {k: [] for k in ("scene", "sample", "sample_data", "ego_pose", "calibrated_sensor", "sensor", "sample_annotation",
                                          "instance", "category", "attribute", "visibility", "log", "map")}
    tok = lambda kind, *ids: kind + "_" + "_".join(str(i) for i in ids)
    os.makedirs(os.path.join(root, version), exist_ok=True)
    channels = ["LIDAR_TOP"]
    for sc in scenes:
        for s in sc:
            for c in s.get("cameras", []):
                if c["channel"] not in channels:
                    channels.append(c["channel"])
    for ch in channels:
        T["sensor"].append({"token": tok("sensor", ch), "channel": ch, "modality": "lidar" if ch == "LIDAR_TOP" else "camera"})
        os.makedirs(os.path.join(root, "samples", ch), exist_ok=True)
    os.makedirs(os.path.join(root, "sweeps", "LIDAR_TOP"), exist_ok=True)
    T["log"].append({"token": "log_0", "logfile": "synthetic", "vehicle": "synthetic", "date_captured": "2018-07-24", "location": "synthetic"})
    T["map"].append({"token": "map_0", "log_tokens": ["log_0"], "category": "semantic_prior", "filename": ""})
    cats, attrs, viss = {}, {}, {}

    def intern(table, cache, name, extra=None):
        if name not in cache:
            cache[name] = tok(table, len(cache))
            T[table].append(dict({"token": cache[name], "name": name, "description": name}, **(extra or {})))
        return cache[name]

    def pose_rec(table, token, p7, extra=None):
        T[table].append(dict({"token": token, "translation": [float(v) for v in p7[:3]], "rotation": [float(v) for v in p7[3:7]]}, **(extra or {})))

    for si, sc in enumerate(scenes):
        scene_tok = tok("scene", si)
        sample_toks = [s.get("sample_token", tok("sample", si, k)) for k, s in enumerate(sc)]
        T["scene"].append({"token": scene_tok, "log_token": "log_0", "nbr_samples": len(sc), "first_sample_token": sample_toks[0] if sc else "",
                           "last_sample_token": sample_toks[-1] if sc else "", "name": sc[0].get("scene_name", f"scene-{si:04d}") if sc else f"scene-{si:04d}",
                           "description": sc[0].get("scene_description", "") if sc else ""})
        lidar_chain = []  # sample_data tokens of LIDAR_TOP in increasing time order
        for k, s in enumerate(sc):
            st = sample_toks[k]
            ts = int(s.get("timestamp", 1532402927647951 + k * 500000))
            T["sample"].append({"token": st, "timestamp": ts, "scene_token": scene_tok, "prev": sample_toks[k - 1] if k else "",
                                "next": sample_toks[k + 1] if k + 1 < len(sc) else ""})
            sweeps = s["lidar_sweeps"]
            mine = []
            for w, sw in enumerate(sweeps):  # sweep 0 is the keyframe, later entries go back in time
                sd = tok("sd", st, "LIDAR_TOP", w)
                key = w == 0
                rel = os.path.join("samples" if key else "sweeps", "LIDAR_TOP", f"{st}__LIDAR_TOP__{w}.pcd.bin")
                write_pcd_bin(os.path.join(root, rel), sw["points_raw"])
                pose_rec("ego_pose", tok("pose", sd), sw["ego_pose"], {"timestamp": ts - int(round(sw.get("time_lag", 0.0) * 1e6))})
                pose_rec("calibrated_sensor", tok("cs", sd), sw["calib"], {"sensor_token": tok("sensor", "LIDAR_TOP"), "camera_intrinsic": []})
                T["sample_data"].append({"token": sd, "sample_token": st, "ego_pose_token": tok("pose", sd), "calibrated_sensor_token": tok("cs", sd),
                                         "timestamp": ts - int(round(sw.get("time_lag", 0.0) * 1e6)), "fileformat": "pcd", "is_key_frame": key,
                                         "height": 0, "width": 0, "filename": rel.replace(os.sep, "/"), "prev": "", "next": ""})
                mine.append(sd)
            lidar_chain += mine[::-1]  # oldest sweep first, keyframe last
            images = s.get("images") or []
            for ci, c in enumerate(s.get("cameras", [])):
                sd = tok("sd", st, c["channel"])
                rel = os.path.join("samples", c["channel"], f"{st}__{c['channel']}.jpg")
                h = w_ = 0
                if ci < len(images):
                    Image.fromarray(np.asarray(images[ci], np.uint8)).save(os.path.join(root, rel), format="JPEG", quality=jpeg_quality)
                    h, w_ = int(np.asarray(images[ci]).shape[0]), int(np.asarray(images[ci]).shape[1])
                pose_rec("ego_pose", tok("pose", sd), c.get("ego_pose", s["ego_pose"]), {"timestamp": ts})
                pose_rec("calibrated_sensor", tok("cs", sd), c["calib"], {"sensor_token": tok("sensor", c["channel"]),
                                                                          "camera_intrinsic": np.asarray(c["intrinsic"], np.float64).reshape(3, 3).tolist()})
                T["sample_data"].append({"token": sd, "sample_token": st, "ego_pose_token": tok("pose", sd), "calibrated_sensor_token": tok("cs", sd),
                                         "timestamp": ts, "fileformat": "jpg", "is_key_frame": True, "height": h, "width": w_,
                                         "filename": rel.replace(os.sep, "/"), "prev": "", "next": ""})
            for a, ann in enumerate(s.get("annotations", [])):
                inst = ann.get("instance_token", tok("inst", st, a))
                T["instance"].append({"token": inst, "category_token": intern("category", cats, ann["category_name"]), "nbr_annotations": 1,
                                      "first_annotation_token": ann.get("token", tok("ann", st, a)), "last_annotation_token": ann.get("token", tok("ann", st, a))})
                T["sample_annotation"].append({
                    "token": ann.get("token", tok("ann", st, a)), "sample_token": st, "instance_token": inst,
                    "visibility_token": intern("visibility", viss, ann.get("visibility_token", ""), {"level": ann.get("visibility_token", "")}),
                    "attribute_tokens": [intern("attribute", attrs, n) for n in ann.get("attribute_tokens", [])],
                    "translation": [float(v) for v in ann["translation"]], "size": [float(v) for v in ann["size"]],
                    "rotation": [float(v) for v in ann["rotation"]], "prev": "", "next": "",
                    "num_lidar_pts": int(ann.get("num_lidar_pts", 0)), "num_radar_pts": int(ann.get("num_radar_pts", 0))})
        by_tok = {r["token"]: r for r in T["sample_data"]}
        for a, b in zip(lidar_chain[:-1], lidar_chain[1:]):
            by_tok[a]["next"], by_tok[b]["prev"] = b, a
    for name, rows in T.items():
        with open(os.path.join(root, version, name + ".json"), "w") as f:
            json.dump(rows, f)
    return {k: len(v) for k, v in T.items()}
