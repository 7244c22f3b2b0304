"""ctypes binding of libmsc_geom.so (C-ABI in include/msc_geom.h).  No CPU fallback: a missing library raises."""
from __future__ import annotations

import ctypes as C
import os

_LIB_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lib", "libmsc_geom.so")

MSC_MAX_CAMS = 8
MSC_MAX_BOXES_FUSED = 255
MSC_STATS_STRIDE = 16
ABI_VERSION = 3


class MscError(RuntimeError):
    """A non-zero status of the C-ABI; `status` is the msc_status value (include/msc_geom.h)."""

    def __init__(self, message: str, status: int = 0):
        super().__init__(message)
        self.status = status


MSC_ERR_BAD_ARGUMENT = -1
MSC_ERR_UNSUPPORTED = -3


class MscParams(C.Structure):
    _fields_ = [
        ("remove_close_radius", C.c_float), ("range_min", C.c_float), ("range_max", C.c_float), ("z_min", C.c_float),
        ("z_max", C.c_float), ("ground_z", C.c_float), ("bev_range", C.c_float), ("bev_res", C.c_int32),
        ("image_w", C.c_int32), ("image_h", C.c_int32), ("n_cams", C.c_int32), ("fov_keep_mask", C.c_uint32),
        ("centroid_shift", C.c_int32), ("intensity_shift", C.c_int32), ("s_lo", C.c_float), ("s_hi", C.c_float),
    ]


class MscBatchIn(C.Structure):
    _fields_ = [
        ("n_samples", C.c_int32), ("max_boxes_per_sample", C.c_int32), ("n_boxes", C.c_int32), ("points_per_sample_hint", C.c_int32),
        ("points", C.c_void_p),
        ("sample_sweep_off", C.c_void_p), ("sweep_start", C.c_void_p), ("sweep_count", C.c_void_p),
        ("sweep_pose", C.c_void_p), ("sample_box_off", C.c_void_p), ("boxes", C.c_void_p), ("ego_pose", C.c_void_p),
        ("lidar_calib", C.c_void_p), ("cam_ego_pose", C.c_void_p), ("cam_calib", C.c_void_p), ("cam_K", C.c_void_p),
    ]


class MscBatchOut(C.Structure):
    _fields_ = [
        ("box_count", C.c_void_p), ("box_nearest", C.c_void_p), ("box_centroid", C.c_void_p), ("proj_visible", C.c_void_p),
        ("proj_extent", C.c_void_p), ("bev_ci", C.c_void_p), ("bev_height", C.c_void_p), ("stats", C.c_void_p),
    ]


class MscDepthParams(C.Structure):
    _fields_ = [("min_dist", C.c_float), ("downsample", C.c_int32), ("support_margin", C.c_float)]


class MscDepthOut(C.Structure):
    _fields_ = [("depth", C.c_void_p), ("cam_points", C.c_void_p), ("box_support", C.c_void_p)]


class MscLidarBatchOut(C.Structure):
    _fields_ = [("row_capacity", C.c_uint32), ("counts", C.c_void_p), ("ground_off", C.c_void_p), ("object_off", C.c_void_p), ("ground", C.c_void_p),
                ("object", C.c_void_p), ("labels", C.c_void_p), ("n_clusters", C.c_void_p), ("clusters", C.c_void_p), ("cluster_first", C.c_void_p),
                ("noise_first", C.c_void_p), ("status", C.c_void_p)]


class MscClusterMatchOut(C.Structure):
    _fields_ = [("cluster", C.c_void_p), ("box", C.c_void_p)]


class MscJpegComp(C.Structure):
    _fields_ = [("h", C.c_int32), ("v", C.c_int32), ("blocks_x", C.c_int32), ("blocks_y", C.c_int32), ("ds_w", C.c_int32), ("ds_h", C.c_int32),
                ("coef_off", C.c_int64), ("plane_off", C.c_int64), ("qt", C.c_uint16 * 64)]


class MscJpegDesc(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("n_comp", C.c_int32), ("hmax", C.c_int32), ("vmax", C.c_int32), ("mcus_x", C.c_int32),
                ("mcus_y", C.c_int32), ("reserved_", C.c_int32), ("coef_elems", C.c_int64), ("plane_bytes", C.c_int64), ("comp", MscJpegComp * 3)]


class MscJpegHuff(C.Structure):
    _fields_ = [("look", C.c_uint16 * 512), ("maxcode", C.c_int32 * 18), ("valptr", C.c_int32 * 17), ("vals", C.c_uint8 * 256)]


class MscJpegPlan(C.Structure):
    _fields_ = [("desc", MscJpegDesc), ("scan_off", C.c_int64), ("scan_bytes", C.c_int64), ("restart_interval", C.c_int32), ("td", C.c_int32 * 3),
                ("ta", C.c_int32 * 3), ("reserved_", C.c_int32), ("dc", MscJpegHuff * 4), ("ac", MscJpegHuff * 4)]


class MscPngImage(C.Structure):
    _fields_ = [("pixels", C.c_void_p), ("row_pitch", C.c_int64), ("height", C.c_int32), ("width", C.c_int32), ("channels", C.c_int32),
                ("swap_rb", C.c_int32)]


_lib = None

_PROTOS = {
    "msc_abi_version": (C.c_int, []),
    "msc_last_error": (C.c_char_p, []),
    "msc_device_info": (C.c_int, [C.POINTER(C.c_int32)] * 4),
    "msc_fused_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "msc_fused_destroy": (C.c_int, [C.c_void_p]),
    "msc_fused_workspace_bytes": (C.c_size_t, [C.c_void_p, C.POINTER(MscParams), C.c_int32, C.c_int32]),
    "msc_fused_evidence_batch": (C.c_int, [C.c_void_p, C.POINTER(MscParams), C.POINTER(MscBatchIn), C.POINTER(MscBatchOut), C.c_void_p,
                                           C.c_size_t, C.c_void_p]),
    "msc_fused_evidence_batch_replicated": (C.c_int, [C.c_void_p, C.POINTER(MscParams), C.POINTER(MscBatchIn), C.POINTER(MscBatchOut), C.c_int32,
                                                      C.POINTER(MscBatchOut), C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_fused_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32]),
    "msc_fused_get_option": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int32)]),
    "msc_fused_kernel_times": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.c_int32]),
    "msc_aggregate_sweeps": (C.c_int, [C.c_float, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_keyframe_filter_split": (C.c_int, [C.POINTER(MscParams), C.c_void_p, C.c_uint32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_keyframe_bev": (C.c_int, [C.POINTER(MscParams), C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msc_cloud_stats": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p]),
    "msc_annotation_table": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "msc_box_footprints": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msc_relation_table": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msc_relation_table_batch": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msc_project_boxes": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "msc_camera_depth_batch": (C.c_int, [C.POINTER(MscParams), C.POINTER(MscDepthParams), C.POINTER(MscBatchIn), C.POINTER(MscDepthOut),
                                         C.c_void_p]),
    "msc_cluster_aabb": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "msc_dbscan_workspace_bytes": (C.c_size_t, [C.c_uint32, C.POINTER(C.c_int32)]),
    "msc_dbscan": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int32, C.c_double, C.c_int32, C.POINTER(C.c_double), C.c_double, C.POINTER(C.c_int32), C.c_void_p,
                             C.POINTER(C.c_int32), C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_lidar_batch_workspace_bytes": (C.c_size_t, [C.POINTER(MscParams), C.c_double, C.c_int32, C.c_uint32]),
    "msc_lidar_batch": (C.c_int, [C.POINTER(MscParams), C.c_double, C.c_int32, C.POINTER(MscBatchIn), C.POINTER(MscLidarBatchOut), C.c_void_p,
                                  C.c_size_t, C.c_void_p]),
    "msc_cluster_match_batch_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_uint32]),
    "msc_cluster_match_batch": (C.c_int, [C.POINTER(MscBatchIn), C.POINTER(MscLidarBatchOut), C.c_int32, C.POINTER(MscClusterMatchOut), C.c_void_p,
                                          C.c_size_t, C.c_void_p]),
    "msc_jpeg_info": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(MscJpegDesc)]),
    "msc_jpeg_entropy_decode_host": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(MscJpegDesc), C.c_void_p]),
    "msc_jpeg_reconstruct": (C.c_int, [C.POINTER(MscJpegDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msc_jpeg_decode_plan": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_jpeg_decode_batch_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_void_p]),
    "msc_jpeg_decode_batch": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_jpeg_encode_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_size_t]),
    "msc_jpeg_encode_batch": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_cluster_views": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msc_keyframe_bev_batch_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "msc_keyframe_bev_batch": (C.c_int, [C.POINTER(MscParams), C.POINTER(MscLidarBatchOut), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                         C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_cluster_views_batch_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "msc_cluster_views_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_png_encode_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_void_p]),
    "msc_png_encode_batch": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "msc_cluster_mosaics_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "msc_cluster_mosaics": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                      C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Load libmsc_geom.so; raises MscError when it has not been built (there is no fallback path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise MscError(f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(make -C multimodal-scene-captioning_b200/csrc). There is no CPU fallback.")
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)  # AttributeError here means the library and the header disagree
        fn.restype = res
        fn.argtypes = args
    if lib.msc_abi_version() != ABI_VERSION:
        raise MscError(f"ABI mismatch: library {lib.msc_abi_version()} vs binding {ABI_VERSION}")
    _lib = lib
    return lib


DEFAULT_FUSED_CONFIG = 0    # auto (fused_evidence.cu: msc_fused_ctx::opt_config): stream4.cu (fused_stream.cu when fov_keep_mask != 0)
FUSED_CONFIGS = (10, 7)     # forced: stream4.cu, fused_stream.cu
DEFAULT_FUSED_PPT = 2       # stream4.cu launch shape: 2 points per lane (1024 threads) or 4 (512 threads)


def check(status: int, what: str):
    if status != 0:
        msg = load().msc_last_error().decode("utf-8", "replace")
        raise MscError(f"{what} failed with status {status}: {msg}", status)


class FusedContext:
    """An msc_fused_ctx: options, side stream and timing ring of one caller (created on the current CUDA device)."""

    def __init__(self):
        self._lib = load()
        h = C.c_void_p()
        check(self._lib.msc_fused_create(C.byref(h)), "msc_fused_create")
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            self._lib.msc_fused_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key: str, value: int):
        check(self._lib.msc_fused_set_option(self.handle, key.encode(), int(value)), f"set_option({key})")

    def get_option(self, key: str) -> int:
        v = C.c_int32(0)
        check(self._lib.msc_fused_get_option(self.handle, key.encode(), C.byref(v)), f"get_option({key})")
        return int(v.value)

    def kernel_times(self, n: int = 64):
        """Durations (ms) of the streaming kernel in the most recent calls timed with set_option("time_kernel", 1), oldest first."""
        buf = (C.c_float * max(n, 1))()
        got = self._lib.msc_fused_kernel_times(self.handle, buf, int(n))
        if got < 0:
            check(got, "msc_fused_kernel_times")
        return [float(buf[i]) for i in range(got)]


_default_ctx = {}


def default_context() -> FusedContext:
    """The context module-level set_option / get_option / kernel_times act on and a GeometryEngine uses unless it is given its own;
    one per CUDA device."""
    import torch
    dev = torch.cuda.current_device()
    ctx = _default_ctx.get(dev)
    if ctx is None:
        ctx = _default_ctx[dev] = FusedContext()
    return ctx


def set_option(key: str, value: int):
    default_context().set_option(key, value)


def get_option(key: str) -> int:
    return default_context().get_option(key)


def kernel_times(n: int = 64):
    return default_context().kernel_times(n)
