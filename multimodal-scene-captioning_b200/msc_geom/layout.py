"""Flat batch layout for the fused kernel (DESIGN.md section 3) and the parameter block.

A batch is a handful of flat arrays (include/msc_geom.h `msc_batch_in`): raw sweep rows of every sample
concatenated (each sweep starting at a multiple of 4 points so 16-byte bulk copies are legal), per-sweep
3x4 float64 transforms, global-frame boxes, and per-sample poses / calibrations.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np

from .geometry import pose7, ref_from_sweep, sqrt_thresholds

N_CAMS_DEFAULT = 6


@dataclass
class GeomParams:
    """Scalar parameters; defaults are the reference's (lidar_agent.py:43-49, :106-115)."""
    remove_close_radius: float = 1.0
    range_min: float = 1.0
    range_max: float = 50.0
    z_min: float = -3.0
    z_max: float = 5.0
    ground_z: float = -1.4
    bev_range: float = 50.0
    bev_res: int = 200
    image_w: int = 1600
    image_h: int = 900
    n_cams: int = N_CAMS_DEFAULT
    fov_keep_mask: int = 0
    intensity_shift: int = 8

    @property
    def centroid_shift(self) -> int:
        # 32 lanes x max |coordinate| x 2^shift must stay below 2^31 (REDUX-safe and s32-safe per point)
        m = max(abs(self.range_max), abs(self.z_min), abs(self.z_max), 1.0)
        # two 12-bit limbs per axis hold the biased coordinate: |c| < 64 m at 2^-17 m (7.6 um) resolution
        return int(min(17, np.floor(np.log2((2.0 ** 23) / m))))

    def thresholds(self):
        return sqrt_thresholds(self.range_min, self.range_max)


@dataclass
class DepthParams:
    """Parameters of the [EXT] LiDAR -> camera projection (msc_camera_depth_batch).  Kept apart from GeomParams, whose values key the
    fused path's parameter cache.  min_dist: devkit map_pointcloud_to_image's (m, >= 0); downsample: pixel block edge of the depth
    maps; support_margin: metres of slack around a box's depth range when its blocks are classed as in front of / on the box."""
    min_dist: float = 1.0
    downsample: int = 8
    support_margin: float = 0.5

    def block_shape(self, image_w: int, image_h: int):
        """(rows, columns) of one depth map."""
        ds = max(int(self.downsample), 1)  # the library refuses downsample < 1
        return (int(image_h) + ds - 1) // ds, (int(image_w) + ds - 1) // ds


def boxes_from_annotations(annotations: List[dict]) -> np.ndarray:
    """(B,10) f64: translation, size (w,l,h), rotation (w,x,y,z) exactly as the loader's dicts hold them
    (nuscenes_loader.py:183-185)."""
    out = np.zeros((len(annotations), 10), dtype=np.float64)
    for i, a in enumerate(annotations):
        out[i, 0:3] = a["translation"]
        out[i, 3:6] = a["size"]
        out[i, 6:10] = a["rotation"]
    return out


@dataclass
class HostBatch:
    n_samples: int
    points: np.ndarray            # (n_points_padded + 4, 5) f32
    sample_sweep_off: np.ndarray  # (S+1,) i32
    sweep_start: np.ndarray       # (n_sweeps,) u32
    sweep_count: np.ndarray       # (n_sweeps,) u32
    sweep_pose: np.ndarray        # (n_sweeps, 12) f64
    sweep_time_lag: np.ndarray    # (n_sweeps,) f32
    sample_box_off: np.ndarray    # (S+1,) i32
    boxes: np.ndarray             # (n_boxes, 10) f64
    ego_pose: np.ndarray          # (S, 7)
    lidar_calib: np.ndarray       # (S, 7)
    cam_ego_pose: np.ndarray      # (S, C, 7)
    cam_calib: np.ndarray         # (S, C, 7)
    cam_K: np.ndarray             # (S, C, 9)
    n_cams: int = N_CAMS_DEFAULT
    max_boxes_per_sample: int = 0

    @property
    def n_points(self) -> int:
        return int(self.sweep_count.sum())

    @property
    def n_boxes(self) -> int:
        return int(self.boxes.shape[0])

    def input_bytes(self) -> int:
        return sum(int(getattr(self, k).nbytes) for k in ("points", "sample_sweep_off", "sweep_start", "sweep_count", "sweep_pose",
                                                          "sample_box_off", "boxes", "ego_pose", "lidar_calib", "cam_ego_pose",
                                                          "cam_calib", "cam_K"))


def _sweeps_of(sample: dict):
    """Raw sweeps of a sample dict.  Samples from a plain reference-style loader (no `lidar_sweeps` key) are a
    single identity sweep made from `point_cloud` (N,4): the 5th column is zero-filled."""
    if "lidar_sweeps" in sample and sample["lidar_sweeps"]:
        out = []
        for sw in sample["lidar_sweeps"]:
            M = sw.get("ref_from_sensor")
            if M is None:
                M = ref_from_sweep(sample["ego_pose"], sample["lidar_calib"], sw["ego_pose"], sw["calib"])
            out.append((np.asarray(sw["points_raw"], dtype=np.float32), np.asarray(M, dtype=np.float64), float(sw.get("time_lag", 0.0))))
        return out
    pc = np.asarray(sample["point_cloud"], dtype=np.float32)
    raw = np.zeros((pc.shape[0], 5), dtype=np.float32)
    raw[:, :4] = pc[:, :4]
    return [(raw, np.eye(4)[:3, :4].copy(), 0.0)]


_IDENTITY7 = pose7([0.0, 0.0, 0.0], [1.0, 0.0, 0.0, 0.0])


def pack_batch(samples: List[dict], n_cams: int = N_CAMS_DEFAULT) -> HostBatch:
    S = len(samples)
    sweep_lists = [_sweeps_of(s) for s in samples]
    n_sweeps = sum(len(l) for l in sweep_lists)
    sweep_start = np.zeros(n_sweeps, np.uint32)
    sweep_count = np.zeros(n_sweeps, np.uint32)
    sweep_pose = np.zeros((n_sweeps, 12), np.float64)
    sweep_lag = np.zeros(n_sweeps, np.float32)
    sample_sweep_off = np.zeros(S + 1, np.int32)
    cursor, k = 0, 0
    for i, l in enumerate(sweep_lists):
        sample_sweep_off[i] = k
        for raw, M, lag in l:
            sweep_start[k] = cursor
            sweep_count[k] = raw.shape[0]
            sweep_pose[k] = np.asarray(M, np.float64).reshape(-1)[:12]
            sweep_lag[k] = lag
            cursor += (raw.shape[0] + 3) & ~3
            k += 1
    sample_sweep_off[S] = k
    points = np.full((cursor + 4, 5), np.nan, dtype=np.float32)  # padding rows are NaN: they fail every compare
    k = 0
    for l in sweep_lists:
        for raw, _, _ in l:
            points[sweep_start[k]: sweep_start[k] + raw.shape[0]] = raw
            k += 1
    box_arrays = [boxes_from_annotations(s.get("annotations", [])) for s in samples]
    sample_box_off = np.zeros(S + 1, np.int32)
    sample_box_off[1:] = np.cumsum([b.shape[0] for b in box_arrays])
    boxes = np.concatenate(box_arrays, 0) if box_arrays else np.zeros((0, 10))
    if boxes.shape[0] == 0:
        boxes = np.zeros((0, 10), np.float64)
    ego = np.stack([np.asarray(s.get("ego_pose", _IDENTITY7), np.float64) for s in samples]) if S else np.zeros((0, 7))
    lcal = np.stack([np.asarray(s.get("lidar_calib", _IDENTITY7), np.float64) for s in samples]) if S else np.zeros((0, 7))
    cam_pose = np.zeros((S, n_cams, 7)); cam_cal = np.zeros((S, n_cams, 7)); cam_K = np.zeros((S, n_cams, 9))
    cam_pose[..., 3] = 1.0; cam_cal[..., 3] = 1.0
    cam_K[..., 0] = cam_K[..., 4] = cam_K[..., 8] = 1.0
    for i, s in enumerate(samples):
        for c, cam in enumerate(s.get("cameras", [])[:n_cams]):
            cam_pose[i, c] = cam.get("ego_pose", ego[i])
            cam_cal[i, c] = cam["calib"]
            cam_K[i, c] = np.asarray(cam["intrinsic"], np.float64).reshape(-1)
    return HostBatch(S, points, sample_sweep_off, sweep_start, sweep_count, sweep_pose, sweep_lag, sample_box_off,
                     np.ascontiguousarray(boxes, np.float64), ego, lcal, cam_pose, cam_cal, cam_K, n_cams,
                     int(max([b.shape[0] for b in box_arrays], default=0)))


def tile_batch(hb: HostBatch, reps: int) -> HostBatch:
    """Repeat a packed batch `reps` times (distinct memory, identical content) to build large synthetic batches."""
    if reps == 1:
        return hb
    npad = hb.points.shape[0] - 4
    points = np.concatenate([hb.points[:npad]] * reps + [hb.points[npad:]], 0)
    n_sw = hb.sweep_start.shape[0]
    sweep_start = np.concatenate([hb.sweep_start + np.uint32(r * npad) for r in range(reps)])
    sso = np.concatenate([hb.sample_sweep_off[:-1] + r * n_sw for r in range(reps)] + [np.array([reps * n_sw], np.int32)]).astype(np.int32)
    nb = hb.boxes.shape[0]
    sbo = np.concatenate([hb.sample_box_off[:-1] + r * nb for r in range(reps)] + [np.array([reps * nb], np.int32)]).astype(np.int32)
    t = lambda a: np.concatenate([a] * reps, 0)
    return HostBatch(hb.n_samples * reps, points, sso, sweep_start, t(hb.sweep_count), t(hb.sweep_pose), t(hb.sweep_time_lag), sbo,
                     t(hb.boxes), t(hb.ego_pose), t(hb.lidar_calib), t(hb.cam_ego_pose), t(hb.cam_calib), t(hb.cam_K), hb.n_cams,
                     hb.max_boxes_per_sample)


def truncate_batch(hb: HostBatch, n: int) -> HostBatch:
    """The first `n` samples of a packed batch (views where possible)."""
    if n >= hb.n_samples:
        return hb
    ns, nb = int(hb.sample_sweep_off[n]), int(hb.sample_box_off[n])
    end = int(hb.sweep_start[ns - 1] + ((int(hb.sweep_count[ns - 1]) + 3) & ~3)) if ns > 0 else 0
    pts = np.concatenate([hb.points[:end], np.full((4, hb.points.shape[1]), np.nan, np.float32)], 0)
    counts = np.diff(hb.sample_box_off[: n + 1])
    return HostBatch(n, pts, hb.sample_sweep_off[: n + 1].copy(), hb.sweep_start[:ns].copy(), hb.sweep_count[:ns].copy(), hb.sweep_pose[:ns].copy(),
                     hb.sweep_time_lag[:ns].copy(), hb.sample_box_off[: n + 1].copy(), hb.boxes[:nb].copy(), hb.ego_pose[:n].copy(),
                     hb.lidar_calib[:n].copy(), hb.cam_ego_pose[:n].copy(), hb.cam_calib[:n].copy(), hb.cam_K[:n].copy(), hb.n_cams,
                     int(counts.max()) if n > 0 else 0)
