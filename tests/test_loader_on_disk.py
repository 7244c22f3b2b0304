"""Rows a1 / a2 / (f3) of SURVEY.md section 8 on an on-disk dataset: msc_geom.io.write_nuscenes_tree writes a v1.0-mini-shaped tree
(JSON tables + .pcd.bin + .jpg), tests/devkit_shim stands in for the un-vendored devkit's table access, and the REAL NuScenesLoader code
paths run against it -- this repo's, and (with MSC_REFERENCE_SRC set) the reference's own, unmodified, for a key-by-key comparison."""
import hashlib
import importlib
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM = os.path.join(HERE, "devkit_shim")
INTERFACE = os.path.join(HERE, "golden", "interface_golden.json")
REF_SRC = os.environ.get("MSC_REFERENCE_SRC", "")  # src/ of a checkout of the original project, which this repository does not carry


@pytest.fixture()
def devkit_shim():
    """Put the shim on sys.path for one test and reload the loader so its `try: import nuscenes` sees it; undo both afterwards."""
    import msc_geom.nuscenes_loader as nl
    sys.path.insert(0, SHIM)
    importlib.reload(nl)
    assert nl.NUSCENES_AVAILABLE
    yield nl
    sys.path.remove(SHIM)
    for m in [m for m in sys.modules if m == "nuscenes" or m.startswith("nuscenes.")]:
        del sys.modules[m]
    importlib.reload(nl)
    assert not nl.NUSCENES_AVAILABLE


def _scenes():
    from msc_geom.synthetic import make_sample
    rng = np.random.default_rng(3)
    scenes = []
    for si in range(2):
        sc = []
        for k in range(2):
            s = make_sample(500 + 10 * si + k, n_sweeps=3, n_boxes=5)
            for sw in s["lidar_sweeps"]:
                sw["points_raw"] = sw["points_raw"][: 3000 + 17 * k]          # small files, lengths that are not multiples of 4
            s["point_cloud"] = s["lidar_sweeps"][0]["points_raw"][:, :4]
            s["images"] = [rng.integers(0, 255, (45, 80, 3), dtype=np.uint8) for _ in s["cameras"]]
            s["scene_name"], s["scene_description"] = f"scene-{si:04d}", f"synthetic scene {si}"
            sc.append(s)
        scenes.append(sc)
    return scenes


def _digest(a):
    return [str(a.dtype), list(a.shape), list(a.strides), hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()]


def loader_record(loader):
    """What test_reference_loader_and_mirror_agree_on_the_same_tree compares between the reference's loader and the mirror, on the tree
    of _scenes(), as JSON: scene list, camera channels, and per sample the key order, the scalar fields, the annotation dicts and
    dtype / shape / strides / SHA-256 of the point cloud and of every camera frame (tests/golden/interface_golden.json records it)."""
    samples = []
    for sc in loader.get_scene_list():
        for s in loader.load_scene_samples(sc["token"]):
            rec = {"keys": list(s), "point_cloud": _digest(s["point_cloud"]), "images": [_digest(im) for im in s["images"]]}
            rec.update({k: s[k] for k in ("sample_token", "timestamp", "scene_description", "scene_name", "camera_names", "metadata")})
            rec["annotations"] = [{k: (np.asarray(v).tolist() if k == "velocity" else v) for k, v in a.items()} for a in s["annotations"]]
            samples.append(rec)
    return {"scene_list": loader.get_scene_list(), "camera_channels": list(loader.camera_channels), "samples": samples,
            "sample_1_1": loader.get_sample_by_scene_index(1, 1)["sample_token"]}


def test_loader_output_on_a_written_tree_equals_the_recorded_interface(tmp_path, devkit_shim):
    """The mirror's output on the tree of _scenes(), against the record of it: the values the reference comparison below checks, here
    on every run (NaN velocities compare equal)."""
    from msc_geom import io as mio
    mio.write_nuscenes_tree(str(tmp_path), _scenes())
    got = json.loads(json.dumps(loader_record(devkit_shim.create_loader(str(tmp_path), "v1.0-mini"))))   # the JSON form of the record
    want = json.load(open(INTERFACE))["loader"]
    assert set(got) == set(want) and len(got["samples"]) == len(want["samples"]) == 4
    for k in ("scene_list", "camera_channels", "sample_1_1"):
        assert got[k] == want[k], k
    for g, w in zip(got["samples"], want["samples"]):
        assert list(g) == list(w)
        for k in g:
            if k != "annotations":
                assert g[k] == w[k], (w["sample_token"], k)
        assert len(g["annotations"]) == len(w["annotations"])
        for a, b in zip(g["annotations"], w["annotations"]):
            assert list(a) == list(b)
            for k in a:
                assert np.array_equal(np.asarray(a[k], dtype=float), np.asarray(b[k], dtype=float), equal_nan=True) if k == "velocity" else a[k] == b[k], k


def test_real_loader_code_path_on_a_written_tree(tmp_path, devkit_shim):
    from msc_geom import io as mio
    from msc_geom.layout import pack_batch
    scenes = _scenes()
    sizes = mio.write_nuscenes_tree(str(tmp_path), scenes)
    assert sizes["scene"] == 2 and sizes["sample"] == 4 and sizes["sample_data"] == 4 * (3 + 6) and sizes["sample_annotation"] == 20
    loader = devkit_shim.create_loader(str(tmp_path), "v1.0-mini")
    assert type(loader).__name__ == "NuScenesLoader" and loader.n_sweeps == 10
    sl = loader.get_scene_list()
    assert [s["name"] for s in sl] == ["scene-0000", "scene-0001"] and sl[0]["nbr_samples"] == 2
    assert loader.scene_sample_tokens(sl[1]["token"]) == [s["sample_token"] for s in scenes[1]]     # token-only scan, no sensor files touched
    for si, sc in enumerate(scenes):
        got = loader.load_scene_samples(sl[si]["token"])
        assert len(got) == len(sc)
        for k, (g, s) in enumerate(zip(got, sc)):
            assert g["sample_token"] == s["sample_token"] and g["timestamp"] == s["timestamp"] and g["scene_name"] == s["scene_name"]
            assert g["camera_names"] == s["camera_names"] and g["metadata"] == {"location": "synthetic", "nbr_objects": 5}
            assert g["point_cloud"].shape == s["point_cloud"].shape and g["point_cloud"].strides[0] == 20    # the devkit's 20-byte-pitch view
            assert np.array_equal(g["point_cloud"], s["point_cloud"])
            # like the devkit's from_file_multisweep the walk over `prev` crosses keyframes: the second sample also sees the first one's sweeps
            assert len(g["lidar_sweeps"]) == 3 * (k + 1)
            for a, b in zip(g["lidar_sweeps"], s["lidar_sweeps"]):
                assert np.array_equal(a["points_raw"], b["points_raw"]) and np.array_equal(a["ref_from_sensor"], b["ref_from_sensor"])
                assert abs(a["time_lag"] - b["time_lag"]) < 1e-9
            assert np.array_equal(g["ego_pose"], s["ego_pose"]) and np.array_equal(g["lidar_calib"], s["lidar_calib"])
            for a, b in zip(g["cameras"], s["cameras"]):
                assert a["channel"] == b["channel"] and np.array_equal(a["intrinsic"], b["intrinsic"]) and np.array_equal(a["calib"], b["calib"])
            for a, b in zip(g["annotations"], s["annotations"]):
                for k in ("token", "category_name", "instance_token", "translation", "size", "rotation", "attribute_tokens", "visibility_token"):
                    assert a[k] == b[k], k
                assert np.isnan(a["velocity"]).all()                             # single-frame instances: the devkit's box_velocity gives NaN
            assert [im.shape for im in g["images"]] == [(45, 80, 3)] * 6
    # the on-disk step of the batched path: lazy sweeps (paths) -> files read straight into one (pooled) staging buffer
    lazy = devkit_shim.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=3, lazy_sweeps=True)
    flat = [s for sc in scenes for s in sc]
    lz = [lazy.load_sample(s["sample_token"]) for s in flat]
    assert all("path" in sw and "points_raw" not in sw for s in lz for sw in s["lidar_sweeps"]) and lz[0]["images"] == []
    hb_files = mio.stage_batch(lz, threads=4, pinned=False)
    hb_mem = pack_batch(flat)
    for k in ("points", "sweep_start", "sweep_count", "sweep_pose", "sample_sweep_off", "sample_box_off", "boxes", "ego_pose", "lidar_calib",
              "cam_ego_pose", "cam_calib", "cam_K"):
        assert np.array_equal(getattr(hb_files, k), getattr(hb_mem, k), equal_nan=True), k


@pytest.mark.skipif(not os.path.isdir(REF_SRC), reason="needs the original project's src/ directory in MSC_REFERENCE_SRC")
def test_reference_loader_and_mirror_agree_on_the_same_tree(tmp_path, devkit_shim):
    """The reference's own NuScenesLoader (src/nuscenes_loader.py:15-207), unmodified, on the written tree: every key of its sample dict
    equals the mirror's (which only ADDS keys)."""
    from msc_geom import io as mio
    mio.write_nuscenes_tree(str(tmp_path), _scenes())
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF_SRC)
    try:
        sys.modules.pop("nuscenes_loader", None)
        ref_mod = importlib.import_module("nuscenes_loader")
        assert ref_mod.NUSCENES_AVAILABLE
        ref = ref_mod.create_loader(str(tmp_path), "v1.0-mini")
        assert type(ref).__name__ == "NuScenesLoader"
        mine = devkit_shim.create_loader(str(tmp_path), "v1.0-mini")
        assert ref.get_scene_list() == mine.get_scene_list() and ref.camera_channels == mine.camera_channels
        for sc in ref.get_scene_list():
            for a, b in zip(ref.load_scene_samples(sc["token"]), mine.load_scene_samples(sc["token"])):
                assert set(a) <= set(b) and set(b) - set(a) == {"lidar_sweeps", "ego_pose", "lidar_calib", "cameras"}
                for k in ("sample_token", "timestamp", "scene_description", "scene_name", "camera_names", "metadata"):
                    assert a[k] == b[k], k
                assert a["point_cloud"].dtype == b["point_cloud"].dtype and a["point_cloud"].strides == b["point_cloud"].strides
                assert np.array_equal(a["point_cloud"], b["point_cloud"])
                assert len(a["images"]) == len(b["images"]) and all(np.array_equal(x, y) for x, y in zip(a["images"], b["images"]))
                assert len(a["annotations"]) == len(b["annotations"])
                for x, y in zip(a["annotations"], b["annotations"]):
                    assert list(x) == list(y)                                # same keys, same order
                    for k in x:
                        if k == "velocity":
                            assert np.array_equal(x[k], y[k], equal_nan=True)
                        else:
                            assert x[k] == y[k], k
        s0 = ref.get_sample_by_scene_index(1, 1)
        assert s0["sample_token"] == mine.get_sample_by_scene_index(1, 1)["sample_token"]
    finally:
        sys.path.remove(REF_SRC)
        sys.modules.pop("nuscenes_loader", None)
