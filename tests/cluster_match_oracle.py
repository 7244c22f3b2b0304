"""ctypes bridge to the scalar definition of the cluster <-> box match (tests/cluster_match_oracle.c).  TEST INFRASTRUCTURE ONLY.

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
_SRC = os.path.join(_ROOT, "tests", "cluster_match_oracle.c")
_DEPS = (_SRC, os.path.join(_ROOT, "oracle", "c", "msc_oracle.c"))
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha1(b"".join(open(p, "rb").read() for p in _DEPS)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"msc_cluster_match_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(so):
            tmp = so + f".{os.getpid()}.tmp"
            subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                            "-Wextra", "-std=c11", "-o", tmp, _SRC, "-lm"], check=True)
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def box_prepare(box, ego_pose, lidar_calib) -> np.ndarray:
    """orc_box_prepare: the f32 record p1[3], i[3], j[3], k[3], ii, jj, kk, pad of one global box."""
    out = np.zeros(16, np.float32)
    lib().orc_box_prepare(*[_p(np.ascontiguousarray(a, np.float64).reshape(-1)) for a in (box, ego_pose, lidar_calib)], _p(out), None)
    return out


def cluster_match(rows, labels, n_clusters: int, boxes, ego_pose, lidar_calib, with_membership: bool = False):
    """One sample: cluster [K, 3] i32, box [B, 5] i32 (and member [n, B] u8 with with_membership)."""
    rows = np.ascontiguousarray(np.asarray(rows, np.float32).reshape(-1, 4))
    labels = np.ascontiguousarray(labels, np.int32)
    boxes = np.ascontiguousarray(boxes, np.float64).reshape(-1, 10)
    n, nb = rows.shape[0], boxes.shape[0]
    cl = np.zeros((n_clusters, 3), np.int32)
    bx = np.zeros((nb, 5), np.int32)
    mem = np.zeros((n, nb), np.uint8) if with_membership else None
    lib().orc_cluster_match_sample(C.c_int(n), _p(rows), _p(labels), C.c_int(n_clusters), C.c_int(nb), _p(boxes),
                                   _p(np.ascontiguousarray(ego_pose, np.float64)), _p(np.ascontiguousarray(lidar_calib, np.float64)),
                                   _p(cl), _p(bx), _p(mem) if with_membership else None)
    return (cl, bx, mem) if with_membership else (cl, bx)


def batch(hb, lidar_per_sample):
    """The whole batch from run_lidar's per-sample host results: per sample (cluster [K_s, 3], box [B_s, 5])."""
    out = []
    for s, r in enumerate(lidar_per_sample):
        b0, b1 = int(hb.sample_box_off[s]), int(hb.sample_box_off[s + 1])
        out.append(cluster_match(r["object"], r["labels"], len(r["clusters"]), hb.boxes[b0:b1], hb.ego_pose[s], hb.lidar_calib[s]))
    return out
