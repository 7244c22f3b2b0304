"""Loader mirror (/root/reference/src/nuscenes_loader.py): same factory, same loader methods, same sample-dict keys; pose,
calibration and sweep data arrive only as ADDITIVE keys (`lidar_sweeps`, `ego_pose`, `lidar_calib`, `cameras`).

* MockNuScenesLoader reproduces the reference mock draw for draw (same NumPy global-RNG call order, nuscenes_loader.py:236-288),
  so a seeded run yields the identical sample.
* SyntheticNuScenesLoader serves nuScenes-shaped multi-sweep samples (msc_geom.synthetic) for batches and benchmarks.
* NuScenesLoader wraps the devkit when it is installed and adds the sweep / pose keys the multi-sweep path needs."""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np

from .geometry import pose7, ref_from_sweep
from .synthetic import CAMERA_CHANNELS, make_sample

try:  # the devkit is an optional, un-vendored dependency of the reference (requirements.txt:4)
    from nuscenes.nuscenes import NuScenes  # type: ignore
    from nuscenes.utils.data_classes import LidarPointCloud  # type: ignore
    NUSCENES_AVAILABLE = True
except ImportError:
    NUSCENES_AVAILABLE = False


class MockNuScenesLoader:
    def __init__(self, dataroot: str = None, version: str = "v1.0-mini"):
        self.camera_channels = list(CAMERA_CHANNELS)

    def get_scene_list(self) -> List[Dict]:
        return [{"token": "mock_scene_001", "name": "scene-0001", "description": "Mock scene with vehicles at intersection", "nbr_samples": 10,
                 "first_sample_token": "mock_sample_001"}]

    def load_sample(self, sample_token: str) -> Dict:
        images = [np.random.randint(0, 255, (900, 1600, 3), dtype=np.uint8) for _ in range(6)]
        point_cloud = np.random.randn(10000, 4).astype(np.float32)
        car = {"token": "mock_ann_001", "category_name": "vehicle.car", "translation": [10.0, 2.0, 0.5], "size": [2.0, 4.5, 1.5],
               "rotation": [1.0, 0.0, 0.0, 0.0], "velocity": [3.0, 0.5], "attribute_tokens": ["vehicle.moving"],
               "visibility_token": "60-80% visibility", "num_lidar_pts": 150, "num_radar_pts": 5}
        adult = {"token": "mock_ann_002", "category_name": "human.pedestrian.adult", "translation": [8.0, -3.0, 1.0], "size": [0.5, 0.5, 1.8],
                 "rotation": [1.0, 0.0, 0.0, 0.0], "velocity": [0.5, 0.2], "attribute_tokens": ["pedestrian.moving"],
                 "visibility_token": "80-100% visibility", "num_lidar_pts": 80, "num_radar_pts": 0}
        return {"sample_token": sample_token, "timestamp": 1532402927647951, "scene_description": "Mock driving scene", "scene_name": "scene-0001",
                "images": images, "camera_names": self.camera_channels, "point_cloud": point_cloud, "annotations": [car, adult],
                "metadata": {"location": "boston-seaport", "nbr_objects": 2}}

    def scene_sample_tokens(self, scene_token: str) -> List[str]:
        return [f"mock_sample_{i:03d}" for i in range(5)]

    def load_scene_samples(self, scene_token: str, max_samples: Optional[int] = None) -> List[Dict]:
        return [self.load_sample(f"mock_sample_{i:03d}") for i in range(min(max_samples or 5, 5))]

    def get_sample_by_scene_index(self, scene_idx: int, sample_idx: int = 0) -> Dict:
        return self.load_sample(f"mock_sample_{sample_idx:03d}")


class SyntheticNuScenesLoader:
    """nuScenes-shaped synthetic scenes: `n_scenes` x `samples_per_scene` samples of `n_sweeps` sweeps each."""

    def __init__(self, n_scenes: int = 10, samples_per_scene: int = 40, n_sweeps: int = 10, n_boxes=None, with_images: bool = False):
        self.camera_channels = list(CAMERA_CHANNELS)
        self.n_scenes, self.samples_per_scene, self.n_sweeps, self.n_boxes, self.with_images = n_scenes, samples_per_scene, n_sweeps, n_boxes, with_images

    def get_scene_list(self) -> List[Dict]:
        return [{"token": f"synth_scene_{s:04d}", "name": f"scene-s{s:04d}", "description": "Synthetic nuScenes-shaped scene",
                 "nbr_samples": self.samples_per_scene, "first_sample_token": f"synth_sample_{s * self.samples_per_scene:06d}"} for s in range(self.n_scenes)]

    def load_sample(self, sample_token: str) -> Dict:
        return make_sample(int(sample_token.rsplit("_", 1)[1]), n_sweeps=self.n_sweeps, n_boxes=self.n_boxes, with_images=self.with_images)

    def scene_sample_tokens(self, scene_token: str) -> List[str]:
        s = int(scene_token.rsplit("_", 1)[1])
        return [f"synth_sample_{s * self.samples_per_scene + i:06d}" for i in range(self.samples_per_scene)]

    def load_scene_samples(self, scene_token: str, max_samples: Optional[int] = None) -> List[Dict]:
        s = int(scene_token.rsplit("_", 1)[1])
        n = self.samples_per_scene if not max_samples else min(max_samples, self.samples_per_scene)
        return [self.load_sample(f"synth_sample_{s * self.samples_per_scene + i:06d}") for i in range(n)]

    def get_sample_by_scene_index(self, scene_idx: int, sample_idx: int = 0) -> Dict:
        return self.load_sample(f"synth_sample_{scene_idx * self.samples_per_scene + sample_idx:06d}")


class NuScenesLoader:
    """Real-data loader: the reference's keys (nuscenes_loader.py:88-101) plus the additive multi-sweep keys."""

    def __init__(self, dataroot: str, version: str = "v1.0-mini", n_sweeps: int = 10, lazy_sweeps: bool = False, engine=None):
        """lazy_sweeps: sweeps carry the .pcd.bin `path` instead of `points_raw` (and `point_cloud` / `images` are left out), so
        msc_geom.io.stage_batch reads the files straight into one pinned batch buffer -- the on-disk step of the batched path; each
        entry of `cameras` then carries its JPEG's `path` for msc_geom.io.stage_camera_files / msc_geom.ops.camera_frames.
        engine: a GeometryEngine; the six camera frames of a sample are then decoded by msc_geom.ops.decode_jpeg_batch (host Huffman
        decode in parallel, IDCT / upsampling / colour conversion on the device) -- the same bytes as the reference's
        np.array(Image.open(...)) (nuscenes_loader.py:136-144); files the decoder refuses (progressive, CMYK, PNG ...) go through PIL."""
        if not NUSCENES_AVAILABLE:
            raise ImportError("nuscenes-devkit is required. Install with: pip install nuscenes-devkit")
        from pathlib import Path
        self.dataroot, self.version, self.n_sweeps, self.lazy_sweeps = Path(dataroot), version, n_sweeps, lazy_sweeps
        self.engine = engine
        self.nusc = NuScenes(version=version, dataroot=str(dataroot), verbose=True)
        self.camera_channels = list(CAMERA_CHANNELS)

    def get_scene_list(self) -> List[Dict]:
        return [{k: s[k] for k in ("token", "name", "description", "nbr_samples", "first_sample_token")} for s in self.nusc.scene]

    def _pose7(self, rec) -> np.ndarray:
        return pose7(rec["translation"], rec["rotation"])

    def load_sample(self, sample_token: str) -> Dict:
        nusc = self.nusc
        sample = nusc.get("sample", sample_token)
        images, names, cameras, image_paths = [], [], [], []
        for ch in self.camera_channels:
            if ch in sample["data"]:
                sd = nusc.get("sample_data", sample["data"][ch])
                if not self.lazy_sweeps:
                    image_paths.append(self.dataroot / sd["filename"])
                names.append(sd["channel"])
                cs = nusc.get("calibrated_sensor", sd["calibrated_sensor_token"])
                cameras.append({"channel": ch, "ego_pose": self._pose7(nusc.get("ego_pose", sd["ego_pose_token"])), "calib": self._pose7(cs),
                                "intrinsic": np.asarray(cs["camera_intrinsic"], np.float64)})
                if self.lazy_sweeps:  # the frame itself is read by msc_geom.io.stage_camera_files
                    cameras[-1]["path"] = str(self.dataroot / sd["filename"])
        if image_paths:
            images = self._load_cameras(image_paths)
        ref_sd = nusc.get("sample_data", sample["data"]["LIDAR_TOP"])
        ref_pose = self._pose7(nusc.get("ego_pose", ref_sd["ego_pose_token"]))
        ref_cal = self._pose7(nusc.get("calibrated_sensor", ref_sd["calibrated_sensor_token"]))
        sweeps, sd = [], ref_sd
        for _ in range(self.n_sweeps):  # App. A.1: walk `prev` from the keyframe
            pose = self._pose7(nusc.get("ego_pose", sd["ego_pose_token"]))
            cal = self._pose7(nusc.get("calibrated_sensor", sd["calibrated_sensor_token"]))
            data = ({"path": str(self.dataroot / sd["filename"])} if self.lazy_sweeps
                    else {"points_raw": np.fromfile(str(self.dataroot / sd["filename"]), dtype=np.float32).reshape(-1, 5)})
            sweeps.append({**data, "ref_from_sensor": ref_from_sweep(ref_pose, ref_cal, pose, cal), "ego_pose": pose, "calib": cal,
                           "time_lag": 1e-6 * (ref_sd["timestamp"] - sd["timestamp"])})
            if sd["prev"] == "":
                break
            sd = nusc.get("sample_data", sd["prev"])
        annotations = []
        for tok in sample["anns"]:
            ann = nusc.get("sample_annotation", tok)
            annotations.append({"token": tok, "category_name": ann["category_name"], "instance_token": ann["instance_token"],
                                "translation": ann["translation"], "size": ann["size"], "rotation": ann["rotation"],
                                "velocity": nusc.box_velocity(tok), "attribute_tokens": [nusc.get("attribute", t)["name"] for t in ann["attribute_tokens"]],
                                "visibility_token": nusc.get("visibility", ann["visibility_token"])["description"],
                                "num_lidar_pts": ann["num_lidar_pts"], "num_radar_pts": ann["num_radar_pts"]})
        scene = nusc.get("scene", sample["scene_token"])
        return {"sample_token": sample_token, "timestamp": sample["timestamp"], "scene_description": scene["description"], "scene_name": scene["name"],
                "images": images, "camera_names": names, "point_cloud": None if self.lazy_sweeps else sweeps[0]["points_raw"][:, :4],
                "annotations": annotations,
                "metadata": {"location": nusc.get("log", scene["log_token"])["location"], "nbr_objects": len(annotations)},
                "lidar_sweeps": sweeps, "ego_pose": ref_pose, "lidar_calib": ref_cal, "cameras": cameras}

    def _load_cameras(self, paths) -> List[np.ndarray]:
        """The sample's camera frames (reference: `_load_camera`, one np.array(Image.open(path)) per channel)."""
        from PIL import Image
        if self.engine is not None:
            from . import ops
            from ._capi import MSC_ERR_UNSUPPORTED, MscError
            try:
                return ops.decode_jpeg_batch(self.engine, [np.fromfile(str(p), dtype=np.uint8) for p in paths])
            except MscError as e:
                # only a file flavour the decoder declares unsupported (progressive, 12-bit, CMYK ...: not nuScenes camera frames) goes
                # to the reference's decoder; a missing library, a corrupt stream or a failed launch is an error, not a detour
                if e.status != MSC_ERR_UNSUPPORTED:
                    raise
        return [np.array(Image.open(p)) for p in paths]

    def scene_sample_tokens(self, scene_token: str) -> List[str]:
        """Tokens of a scene's samples from the table links alone (the reference's evaluator loads every image and point cloud
        just to learn these, src/evaluation_framework.py:488-496)."""
        tok, out = self.nusc.get("scene", scene_token)["first_sample_token"], []
        while tok != "":
            out.append(tok)
            tok = self.nusc.get("sample", tok)["next"]
        return out

    def load_scene_samples(self, scene_token: str, max_samples: Optional[int] = None) -> List[Dict]:
        tok, out = self.nusc.get("scene", scene_token)["first_sample_token"], []
        while tok != "" and not (max_samples and len(out) >= max_samples):
            out.append(self.load_sample(tok))
            tok = self.nusc.get("sample", tok)["next"]
        return out

    def get_sample_by_scene_index(self, scene_idx: int, sample_idx: int = 0) -> Dict:
        samples = self.load_scene_samples(self.nusc.scene[scene_idx]["token"], max_samples=sample_idx + 1)
        return samples[sample_idx] if samples else None


def create_loader(dataroot: Optional[str] = None, version: str = "v1.0-mini", use_mock: bool = False):
    """Same selection rule as the reference factory (nuscenes_loader.py:301-314)."""
    if use_mock or not NUSCENES_AVAILABLE or dataroot is None:
        return MockNuScenesLoader(dataroot, version)
    return NuScenesLoader(dataroot, version)
