"""GeometryEngine -- host driver of the CUDA path.  PyTorch only owns device memory and streams; every
computation goes through the C-ABI (include/msc_geom.h).  There is no CPU fallback anywhere in this file.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _capi
from ._capi import MscBatchIn, MscBatchOut, MscDepthOut, MscDepthParams, MscLidarBatchOut, MscParams
from .layout import DepthParams, GeomParams, HostBatch, pack_batch

_IN_FIELDS = ("points", "sample_sweep_off", "sweep_start", "sweep_count", "sweep_pose", "sample_box_off", "boxes", "ego_pose",
              "lidar_calib", "cam_ego_pose", "cam_calib", "cam_K")

_NP2TORCH = {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64, np.dtype(np.int32): torch.int32,
             np.dtype(np.uint32): torch.int32, np.dtype(np.uint8): torch.uint8}


def _as_torch_cpu(a: np.ndarray) -> torch.Tensor:
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint32:
        a = a.view(np.int32)
    return torch.from_numpy(a)


def make_params(p: GeomParams) -> MscParams:
    s_lo, s_hi = p.thresholds()
    return MscParams(p.remove_close_radius, p.range_min, p.range_max, p.z_min, p.z_max, p.ground_z, p.bev_range, p.bev_res, p.image_w,
                     p.image_h, p.n_cams, p.fov_keep_mask, p.centroid_shift, p.intensity_shift, s_lo, s_hi)


@dataclass
class DeviceBatch:
    """A HostBatch resident in HBM."""
    host: HostBatch
    tensors: Dict[str, torch.Tensor]

    def check_layout(self) -> None:
        """The layout rules of msc_batch_in that the library cannot check from the host (its arrays live on the device): every sweep
        starts at a multiple of 4 rows (16-byte aligned bulk copies) and the points buffer extends at least 16 bytes past the last
        row of every sweep.  A violation would be a misaligned or out-of-bounds cp.async.bulk inside the kernel; here it is an error
        before the first launch (checked once per batch, on the host copy of the sweep table)."""
        hb = self.host
        if hb.sweep_start.size == 0:
            return
        start, count = hb.sweep_start.astype(np.int64), hb.sweep_count.astype(np.int64)
        if (start % 4 != 0).any():
            raise _capi.MscError("msc_batch_in: every sweep must start at a multiple of 4 rows (sweep %d starts at row %d)"
                                 % (int(np.flatnonzero(start % 4)[0]), int(start[np.flatnonzero(start % 4)[0]])))
        rows = int(self.tensors["points"].shape[0])
        end = int((start + count).max())
        if end * 20 + 16 > rows * 20:
            raise _capi.MscError("msc_batch_in: the points buffer (%d rows) must extend 16 bytes past the last sweep row (%d)" % (rows, end))
        if str(self.tensors["points"].dtype) != "torch.float32" or self.tensors["points"].shape[1] != 5 or not self.tensors["points"].is_contiguous():
            raise _capi.MscError("msc_batch_in: points must be a contiguous (rows, 5) float32 tensor")

    def struct(self) -> MscBatchIn:
        """The C struct of this batch (built once: the tensors of a DeviceBatch never move)."""
        st = self.__dict__.get("_struct")
        if st is None or self.__dict__.get("_struct_host") is not self.host:
            t = self.tensors
            hb = self.host
            hint = int(hb.sweep_count.sum() // max(hb.n_samples, 1)) if hb.sweep_count.size else 0
            self.check_layout()
            st = MscBatchIn(hb.n_samples, hb.max_boxes_per_sample, hb.n_boxes, min(hint, 2 ** 31 - 1), *[t[k].data_ptr() for k in _IN_FIELDS])
            self.__dict__["_struct"], self.__dict__["_struct_host"] = st, hb
        return st


@dataclass
class BatchResult:
    """Result tables of msc_fused_evidence_batch, still on the device."""
    n_samples: int
    n_cams: int
    res: int
    intensity_shift: int
    sample_box_off: np.ndarray
    box_count: torch.Tensor
    box_nearest: torch.Tensor
    box_centroid: torch.Tensor
    proj_visible: torch.Tensor
    proj_extent: torch.Tensor
    bev_ci: torch.Tensor
    bev_height: torch.Tensor
    stats: torch.Tensor
    table_arena: Optional[torch.Tensor] = None   # the six small tables above are views into this one buffer (one copy / one collective)

    def struct(self) -> MscBatchOut:
        st = self.__dict__.get("_struct")
        if st is None:
            st = self.__dict__["_struct"] = self._make_struct()
        return st

    def _make_struct(self) -> MscBatchOut:
        return MscBatchOut(self.box_count.data_ptr(), self.box_nearest.data_ptr(), self.box_centroid.data_ptr(),
                           self.proj_visible.data_ptr(), self.proj_extent.data_ptr(), self.bev_ci.data_ptr(), self.bev_height.data_ptr(),
                           self.stats.data_ptr())

    def table_tensors(self):
        """Small per-box / per-sample tables (what NCCL gathers; BEV grids stay sharded)."""
        return [self.box_count, self.box_nearest, self.box_centroid, self.proj_visible, self.proj_extent, self.stats]

    def to_host(self, with_bev: bool = True) -> Dict[str, np.ndarray]:
        out = {
            "box_count": self.box_count.cpu().numpy().view(np.uint32),
            "box_nearest": self.box_nearest.cpu().numpy(),
            "box_centroid": self.box_centroid.cpu().numpy(),
            "proj_visible": self.proj_visible.cpu().numpy(),
            "proj_extent": self.proj_extent.cpu().numpy(),
            "stats": self.stats.cpu().numpy().view(np.uint32),
            "sample_box_off": self.sample_box_off,
        }
        if with_bev:
            ci = self.bev_ci.cpu().numpy().view(np.uint32)
            out["bev_count"] = np.ascontiguousarray(ci[..., 0])
            out["bev_isum_q"] = np.ascontiguousarray(ci[..., 1])
            out["bev_intensity_sum"] = (ci[..., 1].astype(np.float64) / float(1 << self.intensity_shift)).astype(np.float32)
            out["bev_height"] = self.bev_height.cpu().numpy()
        return out


@dataclass
class DepthResult:
    """Outputs of msc_camera_depth_batch ([EXT] row e7), still on the device.  Depth maps stay sharded like the BEV grids."""
    n_samples: int
    n_cams: int
    image_w: int
    image_h: int
    downsample: int
    sample_box_off: np.ndarray
    depth: torch.Tensor                      # f32 [S, C, ceil(H/ds), ceil(W/ds)], +inf where no return lands
    cam_points: torch.Tensor                 # u32 bits in i32 [S, C]
    box_support: Optional[torch.Tensor]      # u32 bits in i32 [B, C, 4]: blocks, blocks with returns, in front, on the box; None: skipped

    def struct(self) -> MscDepthOut:
        return MscDepthOut(self.depth.data_ptr(), self.cam_points.data_ptr(),
                           self.box_support.data_ptr() if self.box_support is not None else None)

    def to_host(self) -> Dict[str, np.ndarray]:
        out = {"depth": self.depth.cpu().numpy(), "cam_points": self.cam_points.cpu().numpy().view(np.uint32),
               "sample_box_off": self.sample_box_off}
        if self.box_support is not None:
            out["box_support"] = self.box_support.cpu().numpy().view(np.uint32)
        return out


@dataclass
class LidarBatchResult:
    """Outputs of msc_lidar_batch (the reference's keyframe evidence for every sample of a batch), still on the device.  `small` holds
    the status word and the per-sample tables in one buffer, so reading them is one copy."""
    n_samples: int
    row_capacity: int
    small: torch.Tensor          # i32 [1 + 7 S]: status, counts [S, 3], ground_off, object_off, n_clusters, noise_first
    ground: torch.Tensor         # f32 [cap, 4]; sample s at ground_off[s]
    object: torch.Tensor         # f32 [cap, 4]; sample s at object_off[s]
    labels: torch.Tensor         # i32 [cap] per object row, numbered per sample, -1 noise
    clusters: torch.Tensor       # f32 [cap, 11]; cluster k of sample s at object_off[s] + k
    cluster_first: torch.Tensor  # i32 [cap] smallest object row (within the sample) of that cluster
    sample_rows: Optional[int] = None  # most keyframe rows of one sample (sizes run_lidar_bev's density table); None: row_capacity

    def _view(self, k: int, n: int) -> torch.Tensor:
        return self.small[1 + k * self.n_samples: 1 + (k + n) * self.n_samples]

    @property
    def counts(self) -> torch.Tensor:
        return self._view(0, 3).view(self.n_samples, 3)

    @property
    def ground_off(self) -> torch.Tensor:
        return self._view(3, 1)

    @property
    def object_off(self) -> torch.Tensor:
        return self._view(4, 1)

    def struct(self) -> MscLidarBatchOut:
        p = lambda t: t.data_ptr() or None
        return MscLidarBatchOut(self.row_capacity, p(self.counts), p(self.ground_off), p(self.object_off), p(self.ground), p(self.object),
                                p(self.labels), p(self._view(5, 1)), p(self.clusters), p(self.cluster_first), p(self._view(6, 1)),
                                p(self.small[:1]))

    def to_host(self) -> List[Dict[str, np.ndarray]]:
        """Per sample: ground / object rows (n, 4) f32 and where they start in the device buffers, counts (kept, ground, object), labels of the object rows (int64, like
        ops.dbscan), clusters (n_clusters, 11) f32 as ops.cluster_aabb, cluster_first (n_clusters,) and noise_first (-1: no noise row).
        This is the synchronisation point; a set status word raises MscError."""
        S = self.n_samples
        small = self.small.cpu().numpy()
        status = int(small[0]) if small.size else 0
        if status:
            why = []
            if status & 1:
                why.append("the component merge left an edge unmerged")
            if status & 2:
                why.append("the keyframes hold more rows than row_capacity (%d)" % self.row_capacity)
            raise _capi.MscError("msc_lidar_batch: status 0x%x: %s" % (status, "; ".join(why)), status)
        tab = small[1:].reshape(7, S) if S else np.zeros((7, 0), np.int32)
        counts = tab[0:3].reshape(S, 3).astype(np.int64)
        goff, ooff, ncl, nfirst = (tab[k].astype(np.int64) for k in (3, 4, 5, 6))
        G, M = int(counts[:, 1].sum()), int(counts[:, 2].sum())
        ground, obj = self.ground[:G].cpu().numpy(), self.object[:M].cpu().numpy()
        labels, clusters, first = self.labels[:M].cpu().numpy(), self.clusters[:M].cpu().numpy(), self.cluster_first[:M].cpu().numpy()
        out = []
        for s in range(S):
            g0, o0, ng, no, k = goff[s], ooff[s], counts[s, 1], counts[s, 2], ncl[s]
            out.append({"counts": counts[s], "ground_off": int(g0), "object_off": int(o0), "ground": ground[g0:g0 + ng], "object": obj[o0:o0 + no], "labels": labels[o0:o0 + no].astype(np.int64),
                        "clusters": clusters[o0:o0 + k], "cluster_first": first[o0:o0 + k], "noise_first": int(nfirst[s])})
        return out


@dataclass
class ClusterMatchResult:
    """Outputs of msc_cluster_match_batch (which annotated box each cluster of a run_lidar result lies in), still on the device."""
    lidar: LidarBatchResult      # the run_lidar result the match was computed from (its status word and per-sample tables)
    sample_box_off: np.ndarray
    cluster: torch.Tensor        # i32 [cap, 3] match_box, match_points, in_any_box; cluster k of sample s at object_off[s] + k
    box: torch.Tensor            # i32 [B, 5] rows, cluster_rows, clusters, best_cluster, best_points
    workspace: torch.Tensor      # u8, msc_cluster_match_batch_workspace_bytes

    def struct(self) -> _capi.MscClusterMatchOut:
        return _capi.MscClusterMatchOut(self.cluster.data_ptr() or None, self.box.data_ptr() or None)

    def to_host(self) -> List[Dict[str, np.ndarray]]:
        """Per sample: "cluster_match" (K_s, 3) i32, row k = cluster k of the sample (match_box as a sample-local box index, -1 none;
        match_points; in_any_box), "box_match" (B_s, 5) i32, row j = the sample's box j (rows, cluster_rows, clusters, best_cluster as a
        sample-local label, -1 none; best_points), and "object_off" / "box_off", where the sample's clusters and boxes start in the
        device tables.  This is the synchronisation point; a set msc_lidar_batch status word raises MscError (the rows were invalid)."""
        lr = self.lidar
        S = lr.n_samples
        small = lr.small.cpu().numpy()
        status = int(small[0]) if small.size else 0
        if status:
            raise _capi.MscError("msc_cluster_match_batch: the msc_lidar_batch status is 0x%x, its rows and the match must not be used" % status,
                                 status)
        tab = small[1:].reshape(7, S) if S else np.zeros((7, 0), np.int32)
        counts, ooff, ncl = tab[0:3].reshape(S, 3).astype(np.int64), tab[4].astype(np.int64), tab[5].astype(np.int64)
        M = int(counts[:, 2].sum())
        cl, bx = self.cluster[:M].cpu().numpy(), self.box.cpu().numpy()
        out = []
        for s in range(S):
            o0, b0, b1 = int(ooff[s]), int(self.sample_box_off[s]), int(self.sample_box_off[s + 1])
            out.append({"cluster_match": cl[o0:o0 + int(ncl[s])], "box_match": bx[b0:b1], "object_off": o0, "box_off": b0})
        return out


@dataclass
class LidarBevResult:
    """Finished BEVs of msc_keyframe_bev_batch for samples first .. first + n_samples - 1 of a LidarBatchResult, still on the device."""
    first: int
    n_samples: int
    res: int
    semantic: torch.Tensor  # u8 [n, res, res, 3] BGR, flipped, overlays drawn
    height: torch.Tensor    # f32 [n, res, res], flipped
    density: torch.Tensor   # u8 [n, res, res], flipped
    status: torch.Tensor    # i32 [1]

    def to_host(self, layers: Sequence[str] = ("semantic", "height", "density")) -> List[Dict[str, np.ndarray]]:
        """Per sample, the layers asked for (finish_bev_layers' dict); only those are copied.  This is the synchronisation point; a set
        status word (a cell count beyond the density table) raises MscError."""
        self.check()
        host = {k: getattr(self, k).cpu().numpy() for k in layers}
        return [{k: host[k][i] for k in layers} for i in range(self.n_samples)]

    def check(self) -> None:
        """Reads the status word (a synchronisation point): a cell count beyond the density table raises MscError."""
        if int(self.status.cpu()[0]):
            raise _capi.MscError("msc_keyframe_bev_batch: a cell count has no entry in the density table", 1)


@dataclass
class ClusterViewsResult:
    """Finished cluster images of msc_cluster_views_batch, still on the device."""
    n_views: int
    images: torch.Tensor  # u8 [n, 512, 512, 3]
    status: torch.Tensor  # i32 [1]

    def to_host(self) -> np.ndarray:
        """u8 [n, 512, 512, 3].  This is the synchronisation point; a view above the maximum view size raises MscError."""
        self.check()
        return self.images.cpu().numpy()

    def check(self) -> None:
        """Reads the status word (a synchronisation point): a view above the maximum view size raises MscError."""
        if int(self.status.cpu()[0]):
            raise _capi.MscError("msc_cluster_views_batch: a view holds more points than max_view_points", 1)


@dataclass
class MosaicsResult:
    """Classifier mosaics of msc_cluster_mosaics, still on the device: mosaic j is images[j], a view into one arena."""
    groups: np.ndarray          # i32 [n, 2]: (first view, count)
    images: List[torch.Tensor]  # u8 (512 rows, 512 cols, 3) each
    arena: torch.Tensor


def mosaic_shape(count: int) -> tuple:
    """(H, W, 3) of lidar_agent.cluster_mosaic over `count` 512 x 512 views: min(3, count) columns, ceil(count / 3) rows."""
    return (512 * ((count + 2) // 3), 512 * min(3, count), 3)


PNG_FRAMING_BYTES = 63  # signature, IHDR, IDAT framing, IEND (57) and the zlib header and Adler-32 (6) of every msc_png_encode_batch file


@dataclass
class PngBatchResult:
    """Files of msc_png_encode_batch, still on the device: image i is arena[out_off[i] : out_off[i + 1]].  `small` holds the status
    word and out_off in one buffer, so reading them is one copy."""
    n_images: int
    shapes: List[tuple]       # (H, W, C) per image
    small: torch.Tensor       # i64 [n + 2]: status (low 32 bits of word 0), out_off [n + 1]
    arena: torch.Tensor       # u8 [out_bytes]
    workspace: torch.Tensor   # u8, msc_png_encode_workspace_bytes
    needed: Optional[int] = None  # arena bytes the last call needed, known after to_host()

    @property
    def out_off(self) -> torch.Tensor:
        return self.small[1:]

    def to_host(self) -> List[bytes]:
        """The files as bytes.  This is the synchronisation point: one copy of status and offsets, then one copy of the used prefix of
        the arena.  A set status word (the files need more than the arena) raises MscError with status 1 and the size they need."""
        small = self.small.cpu().numpy()
        off = small[1:].astype(np.int64)
        self.needed = int(off[-1])
        if int(small[0]) & 0xffffffff:
            raise _capi.MscError("msc_png_encode_batch: the files need %d bytes, the arena holds %d" % (self.needed, self.arena.numel()), 1)
        data = self.arena[:self.needed].cpu().numpy().tobytes()
        return [data[off[i]:off[i + 1]] for i in range(self.n_images)]


BEV_WORKSPACE_PER_CALL = 2 << 30            # workspace bytes of one msc_keyframe_bev_batch call (8 res^2 bytes per sample)
CLUSTER_VIEWS_WORKSPACE_PER_CALL = 2 << 30  # workspace bytes of one msc_cluster_views_batch call (1 MiB + 4 max_view_points per view)


JPEG_HEADER_BYTES = 625  # SOI .. SOS (623 bytes) and EOI of every file msc_jpeg_encode_batch writes


@dataclass
class JpegBatchResult:
    """Files of msc_jpeg_encode_batch, still on the device: image i is arena[out_off[i] : out_off[i + 1]].  `small` holds the status
    word and out_off in one buffer, so reading them is one copy."""
    n_images: int
    height: int
    width: int
    small: torch.Tensor       # i64 [n + 2]: status (low 32 bits of word 0), out_off [n + 1]
    arena: torch.Tensor       # u8 [out_bytes]
    workspace: torch.Tensor   # u8, msc_jpeg_encode_workspace_bytes
    needed: Optional[int] = None  # arena bytes the last call needed, known after to_host()

    @property
    def out_off(self) -> torch.Tensor:
        return self.small[1:]

    def to_host(self) -> List[bytes]:
        """The files as bytes.  This is the synchronisation point: one copy of status and offsets, then one copy of the used prefix of
        the arena.  A set status word (the files need more than the arena) raises MscError with status 1 and the size they need."""
        small = self.small.cpu().numpy()
        off = small[1:].astype(np.int64)
        self.needed = int(off[-1])
        if int(small[0]) & 0xffffffff:
            raise _capi.MscError("msc_jpeg_encode_batch: the files need %d bytes, the arena holds %d" % (self.needed, self.arena.numel()), 1)
        data = self.arena[:self.needed].cpu().numpy().tobytes()
        return [data[off[i]:off[i + 1]] for i in range(self.n_images)]


# Workspace bytes of one msc_jpeg_decode_batch call (a 1600 x 900 4:2:0 frame needs about 2.5 MB).  It bounds the workspace only: the
# coefficient (4.4 MB) and frame (4.3 MB) arenas of a 1600 x 900 frame are allocated for every staged file, so device memory grows with
# the number of files staged at once (about 31 GB for 3,552 such frames); stage fewer samples per run_jpeg_decode to bound it.
JPEG_DECODE_WORKSPACE_PER_CALL = 2 << 30


def jpeg_decode_layout(staged):
    """Frame shapes, coefficient offsets (elements) and frame offsets (bytes, one more than the files) of run_jpeg_decode's arenas for
    the files of an io.StagedCameras."""
    n = len(staged)
    descs = [staged.plans[k].desc for k in range(n)]
    shapes = [(d.height, d.width, 3) if d.n_comp == 3 else (d.height, d.width) for d in descs]
    coef_off = np.zeros(n, np.int64)
    out_off = np.zeros(n + 1, np.int64)
    c = 0
    for k, d in enumerate(descs):
        coef_off[k] = c
        c += int(d.coef_elems)
        out_off[k + 1] = out_off[k] + int(np.prod(shapes[k]))
    return shapes, coef_off, out_off


@dataclass
class JpegDecodeResult:
    """Frames and coefficients of msc_jpeg_decode_batch for the files of an io.StagedCameras, still on the device: file k (staged.index[k])
    is out[out_off[k]:] with shape shapes[k], its coefficients coef[coef_off[k]:] and its status status[k]."""
    shapes: List[tuple]
    coef: torch.Tensor      # i16, every file's coefficients
    coef_off: np.ndarray    # i64 [n]
    out: torch.Tensor       # u8, every file's frame
    out_off: np.ndarray     # i64 [n + 1]
    status: torch.Tensor    # i32 [n]
    files: torch.Tensor     # u8, the device copy of the staged bytes
    workspace: torch.Tensor
    staged: object = None   # the io.StagedCameras of the last run (its host buffer must outlive the upload)

    def frames(self) -> List[torch.Tensor]:
        """Device views of the frames, (H, W, 3) or (H, W); nothing is synchronised."""
        return [self.out[int(self.out_off[k]):int(self.out_off[k + 1])].view(shape) for k, shape in enumerate(self.shapes)]

    def check(self) -> None:
        """Synchronise on the status words; raise MscError naming the first file that failed and its status."""
        st = self.status.cpu().numpy()
        bad = np.flatnonzero(st)
        if len(bad):
            k = int(bad[0])
            where = self.staged.index[k] if self.staged is not None else k
            raise _capi.MscError("msc_jpeg_decode_batch: file %d (sample, camera %s) failed with status %d" % (k, where, int(st[k])), int(st[k]))

    def to_host(self) -> List[np.ndarray]:
        """The frames as host arrays.  This is the synchronisation point: one copy of the status words, then one of the frames."""
        self.check()
        host = self.out.cpu().numpy()
        return [host[int(self.out_off[k]):int(self.out_off[k + 1])].reshape(shape) for k, shape in enumerate(self.shapes)]


def _keyframe_row_counts(hb: HostBatch) -> np.ndarray:
    """Keyframe rows (sweep sample_sweep_off[s]) of every sample that has sweeps."""
    sso = hb.sample_sweep_off
    first = sso[:-1][sso[1:] > sso[:-1]]
    return hb.sweep_count[first].astype(np.int64)


def keyframe_rows(hb: HostBatch) -> int:
    """Total keyframe rows of a batch: the row capacity of run_lidar."""
    return int(_keyframe_row_counts(hb).sum())


class InputArena:
    """One pinned host buffer and one device buffer holding a batch's twelve input arrays at fixed offsets (see
    GeometryEngine.input_arena).  `load(hb)` copies a batch of the same shape into the pinned side (the step a real loader replaces by
    reading files straight into `host_view("points")`, msc_geom.io.stage_batch); `upload()` is one async copy."""

    def __init__(self, eng: "GeometryEngine", hb: HostBatch):
        self.eng = eng
        al = lambda v: (v + 255) & ~255
        off, self.layout = 0, {}
        for k in _IN_FIELDS:
            a = getattr(hb, k)
            self.layout[k] = (off, int(a.nbytes), a.dtype, a.shape)
            off = al(off + int(a.nbytes))
        self.nbytes = max(off, 256)
        self.host = torch.empty(self.nbytes, dtype=torch.uint8).pin_memory()
        self.dev = torch.empty(self.nbytes, dtype=torch.uint8, device=eng.device)
        self.meta = hb
        self._host_np = self.host.numpy()
        self.tensors = {}
        for k, (o, n, dt, shape) in self.layout.items():
            tdt = _NP2TORCH[np.dtype(dt)]
            self.tensors[k] = self.dev[o:o + n].view(tdt).view(shape) if n else torch.empty(shape, dtype=tdt, device=eng.device)

    def host_view(self, k: str) -> np.ndarray:
        o, n, dt, shape = self.layout[k]
        return self._host_np[o:o + n].view(dt).reshape(shape)

    def load(self, hb: HostBatch) -> None:
        for k, (o, n, dt, shape) in self.layout.items():
            a = getattr(hb, k)
            if a.shape != shape:
                raise _capi.MscError(f"InputArena: {k} has shape {a.shape}, the arena was sized for {shape}")
            if n:
                self.host_view(k)[...] = a
        self.meta = hb

    def upload(self, non_blocking: bool = True) -> DeviceBatch:
        self.dev.copy_(self.host, non_blocking=non_blocking)
        return DeviceBatch(self.meta, self.tensors)


class GeometryEngine:
    """Owns the device, the loaded library and reusable output buffers."""

    def __init__(self, device: Optional[int] = None, params: Optional[GeomParams] = None, own_context: bool = False):
        if not torch.cuda.is_available():
            raise _capi.MscError("GeometryEngine needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _capi.load()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        torch.cuda.set_device(self.device)
        # options / side stream / timing ring of the fused path; own_context=True gives this engine private ones (one per host thread)
        self.ctx = _capi.FusedContext() if own_context else _capi.default_context()
        self.params = params or GeomParams()
        sm, smem, maj, mnr = (C.c_int32() for _ in range(4))
        _capi.check(self.lib.msc_device_info(C.byref(sm), C.byref(smem), C.byref(maj), C.byref(mnr)), "msc_device_info")
        self.sm_count, self.smem_optin, self.cc = sm.value, smem.value, (maj.value, mnr.value)
        self._workspaces: Dict[int, torch.Tensor] = {}  # one work counter per stream (kernels on different streams overlap)
        self._ws_need: Dict[tuple, int] = {}
        self._params_cache: Dict[tuple, tuple] = {}
        self._stamps: Dict[object, torch.Tensor] = {}  # overlay stamps of the LiDAR agent's images, per image geometry
        self._bev_lut: Optional[torch.Tensor] = None    # the BEV density table
        self.kernel_launches = 0

    # ------------------------------------------------------------------ transfers
    def upload(self, hb: HostBatch, pinned: Optional[Dict[str, torch.Tensor]] = None, non_blocking: bool = False) -> DeviceBatch:
        tensors = {}
        for k in _IN_FIELDS:
            src = pinned[k] if pinned is not None else _as_torch_cpu(getattr(hb, k))
            tensors[k] = src.to(self.device, non_blocking=non_blocking)
        return DeviceBatch(hb, tensors)

    def upload_tiled(self, hb: HostBatch, reps: int, n_samples: Optional[int] = None) -> DeviceBatch:
        """Upload `hb` once and replicate it `reps` times ON THE DEVICE (distinct memory, identical content), optionally keeping only
        the first `n_samples` samples.  Host memory stays at one copy, so shards of tens of gigabytes can be built from a small pool of
        distinct samples; the returned DeviceBatch's host side carries the metadata only (its `points` array is empty)."""
        from .layout import tile_batch, truncate_batch
        npad = hb.points.shape[0] - 4
        meta_src = HostBatch(hb.n_samples, np.zeros((npad + 4, 0), np.float32), hb.sample_sweep_off, hb.sweep_start, hb.sweep_count, hb.sweep_pose,
                             hb.sweep_time_lag, hb.sample_box_off, hb.boxes, hb.ego_pose, hb.lidar_calib, hb.cam_ego_pose, hb.cam_calib, hb.cam_K,
                             hb.n_cams, hb.max_boxes_per_sample)
        meta = tile_batch(meta_src, reps)
        if n_samples is not None and n_samples < meta.n_samples:
            meta = truncate_batch(meta, n_samples)
        ns = meta.sweep_start.shape[0]
        rows = int(meta.sweep_start[ns - 1] + ((int(meta.sweep_count[ns - 1]) + 3) & ~3)) if ns else 0
        src = _as_torch_cpu(hb.points).to(self.device)
        pts = torch.empty((rows + 4, 5), dtype=torch.float32, device=self.device)
        pts[rows:] = float("nan")
        for r in range((rows + npad - 1) // npad if npad else 0):
            a = r * npad
            b = min(a + npad, rows)
            pts[a:b] = src[: b - a]
        tensors = {"points": pts}
        for k in _IN_FIELDS:
            if k != "points":
                tensors[k] = _as_torch_cpu(getattr(meta, k)).to(self.device)
        meta.points = np.zeros((0, 5), np.float32)
        return DeviceBatch(meta, tensors)

    @staticmethod
    def pin(hb: HostBatch) -> Dict[str, torch.Tensor]:
        return {k: _as_torch_cpu(getattr(hb, k)).pin_memory() for k in _IN_FIELDS}

    def input_arena(self, hb: HostBatch) -> "InputArena":
        """A reusable staging slot sized for batches shaped like `hb`: one pinned host buffer + one device buffer with the twelve input
        arrays at fixed 256-byte-aligned offsets, so a batch goes up in ONE cudaMemcpyAsync and nothing is allocated per batch."""
        return InputArena(self, hb)

    @staticmethod
    def table_layout(n_samples: int, n_boxes: int, n_cams: int):
        """Byte offsets of the six small result tables inside one arena (256-byte aligned) and its size: what one D2H copy or one
        all_gather moves per shard (SURVEY.md section 8(e): fixed-stride tables, one collective)."""
        al = lambda v: (v + 255) & ~255
        off, lay = 0, {}
        for name, nbytes in (("box_count", 4 * n_boxes), ("box_nearest", 4 * n_boxes), ("box_centroid", 12 * n_boxes),
                             ("proj_visible", n_cams * n_boxes), ("proj_extent", 16 * n_cams * n_boxes),
                             ("stats", 4 * _capi.MSC_STATS_STRIDE * n_samples)):
            lay[name] = (off, nbytes)
            off = al(off + nbytes)
        return lay, max(off, 256)

    def alloc_result(self, hb: HostBatch, params: Optional[GeomParams] = None, arena_bytes: Optional[int] = None,
                     arena: Optional[torch.Tensor] = None) -> BatchResult:
        """Output buffers for `hb`.  The small tables live in ONE arena (`arena_bytes` pads it, e.g. to the largest shard of a job,
        so every rank gathers the same size; `arena` places it in caller-owned memory, e.g. this rank's row of a symmetric gathered
        buffer); the BEV layers, which stay sharded, are separate."""
        p = params or self.params
        S, B, Cn, R = hb.n_samples, hb.n_boxes, p.n_cams, p.bev_res
        d = self.device
        lay, size = self.table_layout(S, B, Cn)
        if arena is None:
            arena = torch.zeros(max(size, arena_bytes or 0), dtype=torch.uint8, device=d)
        elif arena.numel() < size or arena.dtype != torch.uint8:
            raise _capi.MscError("alloc_result: the caller's arena is smaller than the tables (%d < %d bytes)" % (arena.numel(), size))

        def view(name, dtype, shape):
            o, n = lay[name]
            return arena[o:o + n].view(dtype).view(shape)
        return BatchResult(
            S, Cn, R, p.intensity_shift, hb.sample_box_off.copy(),
            view("box_count", torch.int32, (B,)), view("box_nearest", torch.float32, (B,)), view("box_centroid", torch.float32, (B, 3)),
            view("proj_visible", torch.uint8, (B, Cn)), view("proj_extent", torch.float32, (B, Cn, 4)),
            torch.empty((S, R, R, 2), dtype=torch.int32, device=d), torch.empty((S, R, R), dtype=torch.float32, device=d),
            view("stats", torch.int32, (S, _capi.MSC_STATS_STRIDE)), arena)

    # ------------------------------------------------------------------ the hot path
    def replica_structs(self, hb: HostBatch, arenas: Sequence[torch.Tensor], params: Optional[GeomParams] = None):
        """A C array of msc_batch_out for msc_fused_evidence_batch_replicated: entry r points at the six small tables laid out (like
        alloc_result) in arenas[r] -- this shard's row of peer r's gathered buffer, peer-mapped memory.  BEV members stay null."""
        p = params or self.params
        lay, size = self.table_layout(hb.n_samples, hb.n_boxes, p.n_cams)
        arr = (MscBatchOut * max(len(arenas), 1))()
        for r, a in enumerate(arenas):
            if a.numel() < size:
                raise _capi.MscError("replica arena %d is smaller than the tables (%d < %d bytes)" % (r, a.numel(), size))
            base = a.data_ptr()
            arr[r] = MscBatchOut(base + lay["box_count"][0], base + lay["box_nearest"][0], base + lay["box_centroid"][0],
                                 base + lay["proj_visible"][0], base + lay["proj_extent"][0], 0, 0, base + lay["stats"][0])
        return arr, len(arenas)

    def run_fused(self, db: DeviceBatch, out: Optional[BatchResult] = None, params: Optional[GeomParams] = None, replicas=None) -> BatchResult:
        """One pass of the hot path over a device-resident batch.  `replicas` = replica_structs(...): the kernels also store every
        small-table entry on those peers (the gather of a sharded batch without a collective)."""
        p = params or self.params
        if p.n_cams != db.host.n_cams:
            raise _capi.MscError(f"params.n_cams={p.n_cams} but the batch was packed for {db.host.n_cams} cameras")
        if out is None:
            out = self.alloc_result(db.host, p)
        key = tuple(p.__dict__.values())  # GeomParams is mutable: the cache is keyed by value
        mp = self._params_cache.get(key)
        if mp is None:
            mp = self._params_cache[key] = make_params(p)
        bi, bo = db.struct(), out.struct()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        wkey = (db.host.n_samples, db.host.n_boxes, p.bev_res, p.bev_range, self.ctx.get_option("cull_shift"))
        ws = self._workspaces.get(stream)
        if self._ws_need.get(wkey) is None:
            self._ws_need[wkey] = int(self.lib.msc_fused_workspace_bytes(self.ctx.handle, C.byref(mp), db.host.n_samples, db.host.n_boxes))
        need = self._ws_need[wkey]
        if ws is None or ws.numel() < need:
            ws = self._workspaces[stream] = torch.zeros(need, dtype=torch.uint8, device=self.device)
        if replicas is not None and replicas[1] > 0:
            _capi.check(self.lib.msc_fused_evidence_batch_replicated(self.ctx.handle, C.byref(mp), C.byref(bi), C.byref(bo), replicas[1], replicas[0],
                                                                     ws.data_ptr(), ws.numel(), C.c_void_p(stream)), "msc_fused_evidence_batch_replicated")
        else:
            _capi.check(self.lib.msc_fused_evidence_batch(self.ctx.handle, C.byref(mp), C.byref(bi), C.byref(bo), ws.data_ptr(), ws.numel(),
                                                          C.c_void_p(stream)), "msc_fused_evidence_batch")
        self.kernel_launches += self.ctx.get_option("last_launches")  # table kernels + the streaming kernel, counted by the library
        return out

    # ------------------------------------------------------------------ LiDAR -> camera projection ([EXT] e7)
    def alloc_depth(self, hb: HostBatch, dp: Optional[DepthParams] = None, params: Optional[GeomParams] = None,
                    box_support: bool = True) -> DepthResult:
        """Output buffers of run_camera_depth for `hb` (image size and camera count from `params`); box_support=False skips the
        per-box counts."""
        p = params or self.params
        dp = dp or DepthParams()
        hbk, wbk = dp.block_shape(p.image_w, p.image_h)
        d = self.device
        S, Cn = hb.n_samples, p.n_cams
        return DepthResult(S, Cn, p.image_w, p.image_h, int(dp.downsample), hb.sample_box_off.copy(),
                           torch.empty((S, Cn, hbk, wbk), dtype=torch.float32, device=d), torch.empty((S, Cn), dtype=torch.int32, device=d),
                           torch.empty((hb.n_boxes, Cn, 4), dtype=torch.int32, device=d) if box_support else None)

    def run_camera_depth(self, db: DeviceBatch, out: Optional[DepthResult] = None, dp: Optional[DepthParams] = None,
                         params: Optional[GeomParams] = None) -> DepthResult:
        """Per-camera depth maps, per-camera return counts and per-(box, camera) LiDAR support of a device-resident batch
        (msc_camera_depth_batch): the devkit's map_pointcloud_to_image over every sample's multi-sweep cloud, in one pass."""
        p = params or self.params
        dp = dp or DepthParams()
        if p.n_cams != db.host.n_cams:
            raise _capi.MscError(f"params.n_cams={p.n_cams} but the batch was packed for {db.host.n_cams} cameras")
        if out is None:
            out = self.alloc_depth(db.host, dp, p)
        hbk, wbk = dp.block_shape(p.image_w, p.image_h)
        if out.n_samples != db.host.n_samples or tuple(out.depth.shape) != (db.host.n_samples, p.n_cams, hbk, wbk) or (
                out.box_support is not None and tuple(out.box_support.shape) != (db.host.n_boxes, p.n_cams, 4)):
            raise _capi.MscError("run_camera_depth: the output buffers do not match the batch, parameters and downsample")
        mp = make_params(p)
        mdp = MscDepthParams(dp.min_dist, int(dp.downsample), dp.support_margin)
        bi, bo = db.struct(), out.struct()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _capi.check(self.lib.msc_camera_depth_batch(C.byref(mp), C.byref(mdp), C.byref(bi), C.byref(bo), C.c_void_p(stream)),
                    "msc_camera_depth_batch")
        if db.host.n_samples > 0:  # fill + depth pass (+ the support scan)
            self.kernel_launches += 2 + int(out.box_support is not None and db.host.n_boxes > 0)
        return out

    # ------------------------------------------------------------------ the reference's keyframe evidence, batched
    def alloc_lidar(self, hb: HostBatch) -> LidarBatchResult:
        """Output buffers of run_lidar for `hb`: row arrays sized by the batch's total keyframe rows (known on the host)."""
        rows = _keyframe_row_counts(hb)
        S, cap, d = hb.n_samples, int(rows.sum()), self.device
        return LidarBatchResult(S, cap, torch.zeros(1 + 7 * S, dtype=torch.int32, device=d), torch.empty((cap, 4), dtype=torch.float32, device=d),
                                torch.empty((cap, 4), dtype=torch.float32, device=d), torch.empty(cap, dtype=torch.int32, device=d),
                                torch.empty((cap, 11), dtype=torch.float32, device=d), torch.empty(cap, dtype=torch.int32, device=d),
                                int(rows.max()) if rows.size else 0)

    def run_lidar(self, db: DeviceBatch, out: Optional[LidarBatchResult] = None, params: Optional[GeomParams] = None, eps: float = 0.5,
                  min_samples: int = 10) -> LidarBatchResult:
        """The reference's LiDAR evidence for every sample of a device-resident batch in one stream-ordered call (msc_lidar_batch): the
        keyframe filter and ground split, DBSCAN(eps, min_samples) over each sample's object rows and the per-cluster boxes.  Only the
        gate / split parameters of `params` are used (LiDARAgent._params()).  Nothing is synchronised; out.to_host() reads the results."""
        p = params or self.params
        hb = db.host
        if out is None:
            out = self.alloc_lidar(hb)
        if out.n_samples != hb.n_samples or out.row_capacity < keyframe_rows(hb):
            raise _capi.MscError("run_lidar: the output buffers do not match the batch")
        mp = make_params(p)
        need = int(self.lib.msc_lidar_batch_workspace_bytes(C.byref(mp), C.c_double(float(eps)), hb.n_samples, out.row_capacity))
        ws = torch.empty(max(need, 256), dtype=torch.uint8, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        bi, bo = db.struct(), out.struct()
        _capi.check(self.lib.msc_lidar_batch(C.byref(mp), C.c_double(float(eps)), int(min_samples), C.byref(bi), C.byref(bo), ws.data_ptr(),
                                             need, C.c_void_p(stream)), "msc_lidar_batch")
        if hb.n_samples > 0:
            self.kernel_launches += 15  # 13 own kernels + the CUB sort and scan (each of those launches several kernels of its own)
        return out

    # ------------------------------------------------------------------ LiDAR clusters -> annotated boxes ([EXT])
    def alloc_cluster_match(self, lr: LidarBatchResult, hb: HostBatch) -> ClusterMatchResult:
        """Output buffers and workspace of run_cluster_match for the run_lidar result `lr` of the batch `hb`."""
        need = int(self.lib.msc_cluster_match_batch_workspace_bytes(hb.n_samples, hb.n_boxes, lr.row_capacity))
        if need == 0 and hb.n_samples > 0:
            raise _capi.MscError("alloc_cluster_match: row_capacity %d is out of range" % lr.row_capacity, _capi.MSC_ERR_BAD_ARGUMENT)
        d = self.device
        return ClusterMatchResult(lr, hb.sample_box_off.copy(), torch.empty((lr.row_capacity, 3), dtype=torch.int32, device=d),
                                  torch.empty((hb.n_boxes, 5), dtype=torch.int32, device=d), torch.empty(max(need, 256), dtype=torch.uint8, device=d))

    def run_cluster_match(self, lr: LidarBatchResult, db: DeviceBatch, out: Optional[ClusterMatchResult] = None) -> ClusterMatchResult:
        """Which annotated box each cluster of `lr` lies in, and which clusters each box holds, for every sample of the device-resident
        batch `db` that `lr` was computed from (msc_cluster_match_batch), stream-ordered behind run_lidar.  With `out` given nothing is
        allocated.  Nothing is synchronised; out.to_host() reads the results."""
        hb = db.host
        if out is None:
            out = self.alloc_cluster_match(lr, hb)
        if (lr.n_samples != hb.n_samples or out.lidar is not lr or tuple(out.cluster.shape) != (lr.row_capacity, 3)
                or tuple(out.box.shape) != (hb.n_boxes, 5) or not np.array_equal(out.sample_box_off, hb.sample_box_off)):
            raise _capi.MscError("run_cluster_match: the output buffers do not match the batch and its run_lidar result", _capi.MSC_ERR_BAD_ARGUMENT)
        bi, rows, bo = db.struct(), lr.struct(), out.struct()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _capi.check(self.lib.msc_cluster_match_batch(C.byref(bi), C.byref(rows), hb.n_samples, C.byref(bo), out.workspace.data_ptr(),
                                                     out.workspace.numel(), C.c_void_p(stream)), "msc_cluster_match_batch")
        if hb.n_samples > 0:
            self.kernel_launches += 3
        return out

    # ------------------------------------------------------------------ the LiDAR agent's images, batched
    def _stamp(self, key, make) -> torch.Tensor:
        """The device copy of an overlay stamp (lidar_agent.overlay_stamp), derived once per image geometry."""
        t = self._stamps.get(key)
        if t is None:
            t = self._stamps[key] = torch.from_numpy(make().view(np.int32)).to(self.device)
        return t

    def _density_table(self, cmax: int) -> torch.Tensor:
        """lidar_agent.density_table on the device, at least cmax + 1 entries (a longer table has the same prefix)."""
        if self._bev_lut is None or self._bev_lut.numel() < cmax + 1:
            from .lidar_agent import density_table
            self._bev_lut = torch.from_numpy(density_table(cmax)).to(self.device)
        return self._bev_lut

    def alloc_bev(self, n: int, res: int) -> LidarBevResult:
        """Output buffers of run_lidar_bev for n samples at res x res."""
        d = self.device
        return LidarBevResult(0, n, res, torch.empty((n, res, res, 3), dtype=torch.uint8, device=d), torch.empty((n, res, res), dtype=torch.float32, device=d),
                              torch.empty((n, res, res), dtype=torch.uint8, device=d), torch.zeros(1, dtype=torch.int32, device=d))

    def run_lidar_bev(self, lr: LidarBatchResult, bev_res: int, bev_range: float, first: int = 0, n: Optional[int] = None,
                      out: Optional[LidarBevResult] = None) -> LidarBevResult:
        """The finished BEV of LiDARAgent._generate_multi_layer_bev (semantic with its overlays, height, density) for samples
        first .. first + n - 1 of a run_lidar result, stream-ordered after it (msc_keyframe_bev_batch, one call per
        BEV_WORKSPACE_PER_CALL bytes of workspace).  Nothing is synchronised; out.to_host() reads the results."""
        n = lr.n_samples - first if n is None else n
        if first < 0 or n < 0 or first + n > lr.n_samples:
            raise _capi.MscError("run_lidar_bev: samples [%d, %d) outside the batch of %d" % (first, first + n, lr.n_samples), _capi.MSC_ERR_BAD_ARGUMENT)
        res = int(bev_res)
        if out is None:
            out = self.alloc_bev(n, res)
        if out.n_samples != n or out.res != res:
            raise _capi.MscError("run_lidar_bev: the output buffers do not match the window", _capi.MSC_ERR_BAD_ARGUMENT)
        out.first = first
        out.status.zero_()
        if n == 0:
            return out
        from .lidar_agent import bev_stamp
        lut = self._density_table(lr.sample_rows if lr.sample_rows is not None else lr.row_capacity)
        stamp = self._stamp(("bev", res, float(bev_range)), lambda: bev_stamp(res, bev_range))
        per = int(self.lib.msc_keyframe_bev_batch_workspace_bytes(res, 1))
        if per == 0:
            raise _capi.MscError("run_lidar_bev: bev_res %d out of range" % res, _capi.MSC_ERR_BAD_ARGUMENT)
        step = max(1, min(n, 65535, BEV_WORKSPACE_PER_CALL // per))
        need = int(self.lib.msc_keyframe_bev_batch_workspace_bytes(res, step))
        ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        mp = make_params(GeomParams(bev_res=res, bev_range=float(bev_range)))
        rows = lr.struct()
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        for a in range(0, n, step):
            k = min(step, n - a)
            _capi.check(self.lib.msc_keyframe_bev_batch(C.byref(mp), C.byref(rows), lr.n_samples, first + a, k, lut.data_ptr(), lut.numel(),
                                                        stamp.data_ptr(), stamp.shape[0], out.semantic[a].data_ptr(), out.height[a].data_ptr(),
                                                        out.density[a].data_ptr(), out.status.data_ptr(), ws.data_ptr(), need, stream),
                        "msc_keyframe_bev_batch")
            self.kernel_launches += 3
        return out

    def run_cluster_views(self, rows: torch.Tensor, labels: torch.Tensor, views, max_view_points: Optional[int] = None,
                          out: Optional[ClusterViewsResult] = None) -> ClusterViewsResult:
        """The finished 4-view image of LiDARAgent._generate_cluster_visualization (discs, axes, titles) of every view, in one
        stream-ordered call per CLUSTER_VIEWS_WORKSPACE_PER_CALL bytes of workspace (msc_cluster_views_batch).  rows: f32 [*, 4] and
        labels: i32 [*] CUDA tensors (e.g. a LidarBatchResult's object and labels); views: (row_begin, row_end, label) triples, the
        points of a view being the rows of its range with its label, in row order.  The points of every view must be finite, as a
        LidarBatchResult's object rows are (the keyframe gate drops non-finite rows): the reference draws no point of a cluster whose
        mean is not finite, and nothing here checks for one (ops.cluster_views refuses such a cluster on the host).  max_view_points
        bounds the points of one view (default: the longest range); a larger view raises in to_host().  Nothing is synchronised."""
        v = np.ascontiguousarray(np.asarray(views, dtype=np.int64).reshape(-1, 3))
        n = v.shape[0]
        if not (isinstance(rows, torch.Tensor) and rows.is_cuda and rows.dtype == torch.float32 and rows.dim() == 2 and rows.shape[1] == 4
                and isinstance(labels, torch.Tensor) and labels.is_cuda and labels.dtype == torch.int32):
            raise _capi.MscError("run_cluster_views: rows must be f32 [*, 4] and labels i32 [*] CUDA tensors", _capi.MSC_ERR_BAD_ARGUMENT)
        if n and (v[:, 0].min() < 0 or (v[:, 1] <= v[:, 0]).any() or v[:, 1].max() > min(rows.shape[0], labels.numel())):
            raise _capi.MscError("run_cluster_views: a view's row range is empty, inverted or outside the rows", _capi.MSC_ERR_BAD_ARGUMENT)
        if max_view_points is None:
            max_view_points = int((v[:, 1] - v[:, 0]).max()) if n else 0
        if out is None:
            out = ClusterViewsResult(n, torch.empty((n, 512, 512, 3), dtype=torch.uint8, device=self.device),
                                     torch.zeros(1, dtype=torch.int32, device=self.device))
        if out.n_views != n:
            raise _capi.MscError("run_cluster_views: the output buffers do not match the views", _capi.MSC_ERR_BAD_ARGUMENT)
        out.status.zero_()
        if n == 0:
            return out
        from .lidar_agent import cluster_view_stamp
        stamp = self._stamp("cluster_view", cluster_view_stamp)
        per = int(self.lib.msc_cluster_views_batch_workspace_bytes(1, int(max_view_points)))
        if per == 0:
            raise _capi.MscError("run_cluster_views: max_view_points %d out of range" % max_view_points, _capi.MSC_ERR_BAD_ARGUMENT)
        step = max(1, min(n, 65535, CLUSTER_VIEWS_WORKSPACE_PER_CALL // per))
        need = int(self.lib.msc_cluster_views_batch_workspace_bytes(step, int(max_view_points)))
        ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        v32 = v.astype(np.int32)
        rows, labels = rows.contiguous(), labels.contiguous()
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        for a in range(0, n, step):
            k = min(step, n - a)
            _capi.check(self.lib.msc_cluster_views_batch(rows.data_ptr(), labels.data_ptr(), v32[a:a + k].ctypes.data, k, int(max_view_points),
                                                         stamp.data_ptr(), stamp.shape[0], out.images[a].data_ptr(), out.status.data_ptr(),
                                                         ws.data_ptr(), need, stream), "msc_cluster_views_batch")
            self.kernel_launches += 6
        return out

    def run_cluster_mosaics(self, views: ClusterViewsResult, groups) -> MosaicsResult:
        """The classifier mosaics lidar_agent.cluster_mosaic makes of views[first : first + count] for every (first, count) of `groups`
        (count 1..10), drawn from a run_cluster_views result on the device in one stream-ordered call (msc_cluster_mosaics): the views
        are copied into their cells, then each count's lidar_agent.mosaic_stamp ('#idx' labels, white empty cells) is written over them.
        Nothing is synchronised."""
        g = np.ascontiguousarray(np.asarray(groups, dtype=np.int64).reshape(-1, 2)).astype(np.int32)
        n = g.shape[0]
        if n and (g[:, 1].min() < 1 or g[:, 1].max() > 10 or g[:, 0].min() < 0 or (g[:, 0] + g[:, 1]).max() > views.n_views):
            raise _capi.MscError("run_cluster_mosaics: a group is outside 1..10 of the %d views" % views.n_views, _capi.MSC_ERR_BAD_ARGUMENT)
        shapes = [mosaic_shape(int(c)) for c in g[:, 1]]
        sizes = [int(np.prod(sh)) for sh in shapes]
        arena = torch.empty(max(sum(sizes), 16), dtype=torch.uint8, device=self.device)
        images, o = [], 0
        for sh, b in zip(shapes, sizes):
            images.append(arena[o:o + b].view(sh))
            o += b
        if n == 0:
            return MosaicsResult(g, images, arena)
        if "mosaic" not in self._stamps:
            from .lidar_agent import mosaic_stamp
            st = [mosaic_stamp(k) if k >= 2 else np.zeros((0, 2), np.uint32) for k in range(11)]
            self._mosaic_off = np.concatenate([[0, 0], np.cumsum([len(a) for a in st[1:]])]).astype(np.int32)
        stamps = self._stamp("mosaic", lambda: np.concatenate(st))
        need = int(self.lib.msc_cluster_mosaics_workspace_bytes(n))
        ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _capi.check(self.lib.msc_cluster_mosaics(views.images.data_ptr(), views.n_views, g.ctypes.data, n, stamps.data_ptr(),
                                                 self._mosaic_off.ctypes.data, arena.data_ptr(), ws.data_ptr(), need, stream), "msc_cluster_mosaics")
        self.kernel_launches += 2
        return MosaicsResult(g, images, arena)

    # ------------------------------------------------------------------ images -> PNG files (serialize.image_to_base64)
    def _png_descs(self, images, swap_rb):
        """msc_png_image descriptors of CUDA u8 images (H, W, 3) or (H, W) whose pixels are contiguous within a row (rows may be
        strided); swap_rb: one flag for all, or one per image."""
        n = len(images)
        swaps = [bool(swap_rb)] * n if isinstance(swap_rb, (bool, int, np.bool_)) else [bool(v) for v in swap_rb]
        if len(swaps) != n:
            raise _capi.MscError("run_png_encode: %d swap_rb flags for %d images" % (len(swaps), n), _capi.MSC_ERR_BAD_ARGUMENT)
        descs = (_capi.MscPngImage * max(n, 1))()
        shapes = []
        for i, im in enumerate(images):
            ok = isinstance(im, torch.Tensor) and im.is_cuda and im.dtype == torch.uint8 and im.device == self.device and im.dim() in (2, 3)
            if ok:
                c = 1 if im.dim() == 2 else int(im.shape[2])
                ok = c in (1, 3) and im.shape[0] > 0 and im.shape[1] > 0 and (im.dim() == 2 or im.stride(2) == 1) and im.stride(1) == c
            if not ok:
                raise _capi.MscError("run_png_encode: image %d must be a uint8 CUDA tensor (H, W, 3) or (H, W) on %s with contiguous rows"
                                     % (i, self.device), _capi.MSC_ERR_BAD_ARGUMENT)
            h, w = int(im.shape[0]), int(im.shape[1])
            descs[i] = _capi.MscPngImage(im.data_ptr(), im.stride(0) if h > 1 else w * c, h, w, c, int(swaps[i]))
            shapes.append((h, w, c))
        return descs, shapes

    def alloc_png(self, images, swap_rb=False, out_bytes: Optional[int] = None) -> PngBatchResult:
        """Buffers of run_png_encode for these images: the file arena (default: a quarter of the raw payload plus the framing of every
        file), offsets and status, and the workspace."""
        descs, shapes = self._png_descs(images, swap_rb)
        n = len(shapes)
        if out_bytes is None:
            out_bytes = sum(h * (1 + w * c) // 4 + PNG_FRAMING_BYTES for h, w, c in shapes)
        need = int(self.lib.msc_png_encode_workspace_bytes(n, descs))
        if need == 0 and n:
            raise _capi.MscError("alloc_png: these images cannot be encoded in one call", _capi.MSC_ERR_BAD_ARGUMENT)
        d = self.device
        return PngBatchResult(n, shapes, torch.zeros(n + 2, dtype=torch.int64, device=d), torch.empty(max(out_bytes, 1), dtype=torch.uint8, device=d),
                              torch.empty(max(need, 256), dtype=torch.uint8, device=d))

    def run_png_encode(self, images, swap_rb=False, out: Optional[PngBatchResult] = None) -> PngBatchResult:
        """PNG files of device images (a sequence of uint8 CUDA tensors (H, W, 3) RGB or (H, W) grey, shapes free, rows may be strided)
        in one stream-ordered call (msc_png_encode_batch): Pillow's IHDR, and an IDAT that inflates to the payload of Pillow's
        Image.fromarray(img).save(buf, "PNG").  swap_rb reads BGR images as RGB.  With `out` given nothing is allocated for the files;
        out.to_host() reads them."""
        if isinstance(images, torch.Tensor):
            images = list(images) if images.dim() == 4 else [images]
        descs, shapes = self._png_descs(images, swap_rb)
        n = len(shapes)
        if out is None:
            out = self.alloc_png(images, swap_rb)
        need = int(self.lib.msc_png_encode_workspace_bytes(n, descs))
        if out.shapes != shapes or out.workspace.numel() < need:
            raise _capi.MscError("run_png_encode: the output buffers do not match the images", _capi.MSC_ERR_BAD_ARGUMENT)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _capi.check(self.lib.msc_png_encode_batch(n, descs, out.arena.data_ptr(), out.arena.numel(), out.out_off.data_ptr(), out.small.data_ptr(),
                                                  out.workspace.data_ptr(), out.workspace.numel(), C.c_void_p(stream)), "msc_png_encode_batch")
        if n > 0:
            self.kernel_launches += 6
        return out

    # ------------------------------------------------------------------ camera frames -> JPEG files (CameraAgent._encode_image)
    def alloc_jpeg(self, n: int, h: int, w: int, out_bytes: Optional[int] = None) -> JpegBatchResult:
        """Buffers of run_jpeg_encode for n frames of h x w: the file arena (default: half the raw RGB bytes plus header and EOI per
        image), offsets and status, and the workspace."""
        if out_bytes is None:
            out_bytes = n * (h * w * 3 // 2 + JPEG_HEADER_BYTES)
        need = int(self.lib.msc_jpeg_encode_workspace_bytes(n, h, w, out_bytes))
        if need == 0:
            raise _capi.MscError("alloc_jpeg: %d frames of %d x %d cannot be encoded in one call" % (n, h, w), _capi.MSC_ERR_BAD_ARGUMENT)
        d = self.device
        return JpegBatchResult(n, h, w, torch.zeros(n + 2, dtype=torch.int64, device=d), torch.empty(max(out_bytes, 1), dtype=torch.uint8, device=d),
                               torch.empty(need, dtype=torch.uint8, device=d))

    def run_jpeg_encode(self, images: torch.Tensor, quality: int = 85, out: Optional[JpegBatchResult] = None) -> JpegBatchResult:
        """JPEG files of a device batch of RGB frames (uint8 [N, H, W, 3]), byte-identical to Pillow's save(..., "JPEG", quality=q), in
        one stream-ordered call (msc_jpeg_encode_batch).  With `out` given nothing is allocated; out.to_host() reads the files."""
        if not (isinstance(images, torch.Tensor) and images.is_cuda and images.dtype == torch.uint8 and images.dim() == 4 and images.shape[3] == 3):
            raise _capi.MscError("run_jpeg_encode: images must be a uint8 CUDA tensor [N, H, W, 3]", _capi.MSC_ERR_BAD_ARGUMENT)
        n, h, w = (int(v) for v in images.shape[:3])
        if out is None:
            out = self.alloc_jpeg(n, h, w)
        if (out.n_images, out.height, out.width) != (n, h, w):
            raise _capi.MscError("run_jpeg_encode: the output buffers do not match the batch", _capi.MSC_ERR_BAD_ARGUMENT)
        images = images.contiguous()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _capi.check(self.lib.msc_jpeg_encode_batch(n, h, w, int(quality), images.data_ptr(), out.arena.data_ptr(), out.arena.numel(),
                                                   out.out_off.data_ptr(), out.small.data_ptr(), out.workspace.data_ptr(), out.workspace.numel(),
                                                   C.c_void_p(stream)), "msc_jpeg_encode_batch")
        if n > 0:
            self.kernel_launches += 6
        return out

    # ------------------------------------------------------------------ camera files -> frames (NuScenesLoader._load_camera)
    def _jpeg_decode_chunks(self, staged) -> List[tuple]:
        """(first, count, workspace bytes) of every msc_jpeg_decode_batch call: consecutive files whose one-file workspaces sum to at most
        JPEG_DECODE_WORKSPACE_PER_CALL (an upper bound of the call's need: the per-call records are shared)."""
        base, size = C.addressof(staged.plans), C.sizeof(_capi.MscJpegPlan)
        n = len(staged)
        one = getattr(staged, "_ws_one", None)
        if one is None:
            one = staged._ws_one = [int(self.lib.msc_jpeg_decode_batch_workspace_bytes(1, base + k * size)) for k in range(n)]
        if 0 in one:
            raise _capi.MscError("run_jpeg_decode: file %d has no valid plan" % one.index(0), _capi.MSC_ERR_BAD_ARGUMENT)
        chunks, a = [], 0
        while a < n:
            k, acc = 1, one[a]
            while a + k < n and acc + one[a + k] <= JPEG_DECODE_WORKSPACE_PER_CALL:
                acc += one[a + k]
                k += 1
            chunks.append((a, k, int(self.lib.msc_jpeg_decode_batch_workspace_bytes(k, base + a * size))))
            a += k
        return chunks

    def alloc_jpeg_decode(self, staged) -> JpegDecodeResult:
        """Buffers of run_jpeg_decode for the files of an io.StagedCameras: coefficient and frame arenas, status words, the device copy
        of the staged bytes and the workspace of the largest call."""
        n = len(staged)
        shapes, coef_off, out_off = jpeg_decode_layout(staged)
        c = int(sum(int(staged.plans[k].desc.coef_elems) for k in range(n)))
        ws = max([need for _, _, need in self._jpeg_decode_chunks(staged)], default=256)
        dv = self.device
        return JpegDecodeResult(shapes, torch.empty(max(c, 8), dtype=torch.int16, device=dv), coef_off,
                                torch.empty(max(int(out_off[-1]), 1), dtype=torch.uint8, device=dv), out_off,
                                torch.zeros(max(n, 1), dtype=torch.int32, device=dv), torch.empty(max(staged.nbytes, 1), dtype=torch.uint8, device=dv),
                                torch.empty(ws, dtype=torch.uint8, device=dv))

    def run_jpeg_decode(self, staged, out: Optional[JpegDecodeResult] = None) -> JpegDecodeResult:
        """Decode the files of an io.StagedCameras on the device, bit-identical to np.array(Image.open(path)): one copy of the used part
        of the staged buffer, then one msc_jpeg_decode_batch call per JPEG_DECODE_WORKSPACE_PER_CALL bytes of workspace (unstuffing,
        Huffman decode, DC prediction, IDCT, upsampling and colour conversion all run there).  Nothing is synchronised; out.to_host() or
        out.check() reads the status words.  A given `out` must have been allocated for files of the same geometry (alloc_jpeg_decode on
        the same plans); any other raises MscError before anything is copied or launched."""
        if out is None:
            out = self.alloc_jpeg_decode(staged)
        n = len(staged)
        # the regions of `out` must be the ones these plans need: a buffer allocated for other files would be written out of bounds
        shapes, coef_off, out_off = jpeg_decode_layout(staged)
        coef_end = int(coef_off[-1]) + int(staged.plans[n - 1].desc.coef_elems) if n else 0
        if (list(out.shapes) != shapes or out.coef.dtype != torch.int16 or out.out.dtype != torch.uint8 or out.status.dtype != torch.int32
                or not np.array_equal(out.coef_off, coef_off) or not np.array_equal(out.out_off, out_off)
                or out.coef.numel() < coef_end or out.out.numel() < int(out_off[-1]) or out.status.numel() < n
                or out.files.numel() < staged.nbytes):
            raise _capi.MscError("run_jpeg_decode: the output buffers do not match the staged files", _capi.MSC_ERR_BAD_ARGUMENT)
        out.staged = staged
        if n == 0:
            return out
        chunks = self._jpeg_decode_chunks(staged)
        if max(need for _, _, need in chunks) > out.workspace.numel():
            raise _capi.MscError("run_jpeg_decode: the workspace is too small for these files", _capi.MSC_ERR_BAD_ARGUMENT)
        src = torch.from_numpy(staged.data[:staged.nbytes]) if staged._holder is None else staged._holder.view(torch.uint8).reshape(-1)[:staged.nbytes]
        out.files[:staged.nbytes].copy_(src, non_blocking=True)
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        base, size = C.addressof(staged.plans), C.sizeof(_capi.MscJpegPlan)
        file_off = np.ascontiguousarray(staged.file_off, np.int64)
        for a, k, _ in chunks:
            _capi.check(self.lib.msc_jpeg_decode_batch(k, base + a * size, out.files.data_ptr(), file_off[a:a + k].ctypes.data, out.coef.data_ptr(),
                                                       out.coef_off[a:a + k].ctypes.data, out.out.data_ptr(), out.out_off[a:a + k].ctypes.data,
                                                       out.status[a].data_ptr(), out.workspace.data_ptr(), out.workspace.numel(), stream),
                        "msc_jpeg_decode_batch")
            self.kernel_launches += 4
        return out

    # ------------------------------------------------------------------ batched pairwise relation tables ([EXT] e6)
    def alloc_relations(self, hb: HostBatch):
        """Ragged per-sample n_s x n_s tables in flat device arrays; returns (tensors dict, pair offsets on host)."""
        nb = np.diff(hb.sample_box_off).astype(np.int64)
        pair_off = np.zeros(hb.n_samples, np.int64)
        pair_off[1:] = np.cumsum(nb[:-1] ** 2)
        total = int((nb ** 2).sum())
        d = self.device
        return {"rect": torch.empty((hb.n_boxes, 6), dtype=torch.float64, device=d), "dist": torch.empty(total, dtype=torch.float32, device=d),
                "bearing": torch.empty(total, dtype=torch.float32, device=d), "category": torch.empty(total, dtype=torch.uint8, device=d),
                "overlap": torch.empty(total, dtype=torch.uint8, device=d), "pair_off": torch.from_numpy(pair_off).to(d)}, pair_off

    def run_relations(self, db: DeviceBatch, rel: Dict[str, torch.Tensor]) -> None:
        """Footprints of every box (loader's global frame, like the reference's annotation path) + one batched relation launch."""
        hb = db.host
        if hb.n_boxes == 0:
            return
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _capi.check(self.lib.msc_box_footprints(hb.n_boxes, db.tensors["boxes"].data_ptr(), None, rel["rect"].data_ptr(), stream), "msc_box_footprints")
        _capi.check(self.lib.msc_relation_table_batch(hb.n_samples, hb.max_boxes_per_sample, db.tensors["sample_box_off"].data_ptr(),
                                                      rel["pair_off"].data_ptr(), rel["rect"].data_ptr(), rel["dist"].data_ptr(), rel["bearing"].data_ptr(),
                                                      rel["category"].data_ptr(), rel["overlap"].data_ptr(), stream), "msc_relation_table_batch")
        self.kernel_launches += 2

    def process_samples(self, samples: Sequence[dict], params: Optional[GeomParams] = None) -> Dict[str, np.ndarray]:
        """Host-in / host-out convenience: pack, upload, run, download."""
        p = params or self.params
        hb = pack_batch(list(samples), n_cams=p.n_cams)
        res = self.run_fused(self.upload(hb), params=p)
        torch.cuda.synchronize(self.device)
        return res.to_host()
