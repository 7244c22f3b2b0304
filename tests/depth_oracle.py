"""ctypes bridge to the scalar definition of [EXT] row e7 (tests/depth_oracle.c).  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use with the flags of oracle/Makefile into a temporary directory keyed by the sources' hash, so
the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(_ROOT, "tests", "depth_oracle.c")
_DEPS = (_SRC, os.path.join(_ROOT, "oracle", "c", "msc_oracle.c"))
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha1(b"".join(open(p, "rb").read() for p in _DEPS)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"msc_depth_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(so):
            tmp = so + f".{os.getpid()}.tmp"
            subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                            "-Wextra", "-std=c11", "-o", tmp, _SRC, "-lm"], check=True)
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _c(a, dt):
    return np.ascontiguousarray(a, dt)


def block_shape(image_w: int, image_h: int, ds: int):
    return (image_h + ds - 1) // ds, (image_w + ds - 1) // ds


def camera_matrix(ego_pose, lidar_calib, cam_ego_pose, cam_calib, K) -> np.ndarray:
    P = np.zeros(12, np.float32)
    lib().orc_camera_matrix(*[_p(_c(a, np.float64).reshape(-1)) for a in (ego_pose, lidar_calib, cam_ego_pose, cam_calib, K)], _p(P))
    return P.reshape(3, 4)


def camera_depth(hb, i: int, image_w=1600, image_h=900, n_cams=None, min_dist=1.0, ds=8, remove_close_radius=1.0, with_pixels=False):
    """Sample i of a HostBatch: depth [C, Hb, Wb] f32, cam_points [C] u32 and, with_pixels, pixel [rows, C] i32."""
    C_ = hb.n_cams if n_cams is None else n_cams
    s0, s1 = int(hb.sample_sweep_off[i]), int(hb.sample_sweep_off[i + 1])
    start = _c(hb.sweep_start[s0:s1], np.uint32); count = _c(hb.sweep_count[s0:s1], np.uint32)
    pose = _c(hb.sweep_pose[s0:s1], np.float64)
    Hb, Wb = block_shape(image_w, image_h, ds)
    depth = np.zeros((C_, Hb, Wb), np.float32); cp = np.zeros(C_, np.uint32)
    pix = np.zeros((int(count.sum()), C_), np.int32) if with_pixels else None
    lib().orc_camera_depth_sample(C.c_float(remove_close_radius), C.c_int(image_w), C.c_int(image_h), C.c_int(C_), C.c_float(min_dist),
                                  C.c_int(ds), _p(hb.points), C.c_int(s1 - s0), _p(start), _p(count), _p(pose),
                                  _p(_c(hb.ego_pose[i], np.float64)), _p(_c(hb.lidar_calib[i], np.float64)),
                                  _p(_c(hb.cam_ego_pose[i, :C_], np.float64)), _p(_c(hb.cam_calib[i, :C_], np.float64)),
                                  _p(_c(hb.cam_K[i, :C_], np.float64)), _p(depth), _p(cp), _p(pix) if with_pixels else None)
    return (depth, cp, pix) if with_pixels else (depth, cp)


def box_support(boxes, cam_ego_pose, cam_calib, cam_K, depth, image_w=1600, image_h=900, ds=8, margin=0.5) -> np.ndarray:
    """[n_boxes, C, 4] u32 over one sample's depth maps [C, Hb, Wb]."""
    boxes = _c(boxes, np.float64).reshape(-1, 10)
    nb, nc = boxes.shape[0], depth.shape[0]
    out = np.zeros((nb, nc, 4), np.uint32)
    lib().orc_box_depth_support(C.c_int(nb), _p(boxes), C.c_int(nc), _p(_c(cam_ego_pose, np.float64)), _p(_c(cam_calib, np.float64)),
                                _p(_c(cam_K, np.float64)), C.c_int(image_w), C.c_int(image_h), C.c_int(ds), C.c_float(margin),
                                _p(_c(depth, np.float32)), _p(out))
    return out


def batch(hb, image_w=1600, image_h=900, n_cams=None, min_dist=1.0, ds=8, margin=0.5, remove_close_radius=1.0):
    """The whole batch: depth [S, C, Hb, Wb], cam_points [S, C], box_support [B, C, 4]."""
    C_ = hb.n_cams if n_cams is None else n_cams
    Hb, Wb = block_shape(image_w, image_h, ds)
    D = np.zeros((hb.n_samples, C_, Hb, Wb), np.float32); CP = np.zeros((hb.n_samples, C_), np.uint32)
    BS = np.zeros((hb.n_boxes, C_, 4), np.uint32)
    for i in range(hb.n_samples):
        D[i], CP[i] = camera_depth(hb, i, image_w, image_h, C_, min_dist, ds, remove_close_radius)
        b0, b1 = int(hb.sample_box_off[i]), int(hb.sample_box_off[i + 1])
        if b1 > b0:
            BS[b0:b1] = box_support(hb.boxes[b0:b1], hb.cam_ego_pose[i, :C_], hb.cam_calib[i, :C_], hb.cam_K[i, :C_], D[i], image_w, image_h,
                                    ds, margin)
    return D, CP, BS
