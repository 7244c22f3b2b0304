"""Evidence serialisation into prompts -- SURVEY.md section 8(f) rank 4, the step right after the geometric path.

Host-side mirror of the strings the reference builds from the evidence before it calls its LLM:
  * SceneGraphAgent._generate_scene_graph's `object_summary` and user prompt
    (/root/reference/src/agents/content_transform/scenegraph_agent.py:327-366),
  * LiDARAgent._image_to_base64 (lidar_agent.py:819-832),
plus the JSON block that carries the [EXT] evidence (per-box point counts, nearest distances, camera visibility, pairwise
relations), which the reference has no slot for except the `context` argument (camera_agent.py:43-47, scenegraph_agent.py:365-366).
Exact string equality with the reference is pinned by tests/golden/prompt_golden.json (made by running the reference).
"""
from __future__ import annotations

import base64
import json
from io import BytesIO
from typing import Any, Dict, List, Optional, Sequence

import numpy as np

_CATEGORY_LINES = (("Vehicles", "vehicles"), ("Cyclists", "cyclists"), ("Pedestrians", "pedestrians"), ("Barriers", "barriers"),
                   ("Traffic cones", "traffic_cones"), ("Construction", "construction"))
_ZONE_LINES = (("Front close (<10m)", "front_close"), ("Front medium (10-30m)", "front_medium"), ("Left close (<10m)", "left_close"),
               ("Right close (<10m)", "right_close"))
_DETAIL_KEYS = ("id", "category", "position", "distance", "direction", "state", "visibility")


def object_summary(categorized: Dict[str, List[Dict]], spatial_zones: Dict[str, List[Dict]], annotations: Sequence[Dict]) -> str:
    """scenegraph_agent.py:327-355: counts per category and zone, then the first five vehicles and pedestrians as JSON."""
    def detail(obj: Dict) -> Dict[str, Any]:
        d = {k: obj[k] for k in _DETAIL_KEYS}
        d["distance"] = round(obj["distance"], 1)
        return d

    n = len(annotations)
    lines = ["", f"Total objects: {n}", "", "By category:"]
    lines += [f"- {label}: {len(categorized[key])}" for label, key in _CATEGORY_LINES]
    lines += ["", "Spatial distribution:"]
    lines += [f"- {label}: {len(spatial_zones.get(key, []))}" for label, key in _ZONE_LINES]
    sample = [detail(o) for o in categorized["vehicles"][:5] + categorized["pedestrians"][:5]]
    lines += ["", "Object details:", json.dumps(sample, indent=2), f"... (showing sample, {n} total)", ""]
    return "\n".join(lines)


def scene_graph_user_prompt(categorized: Dict[str, List[Dict]], spatial_zones: Dict[str, List[Dict]], annotations: Sequence[Dict],
                            context: Optional[Dict] = None) -> str:
    """scenegraph_agent.py:357-366: the user message; `context` is JSON-dumped and cut at 500 characters like the reference does."""
    prompt = ("Build a hierarchical scene graph from this driving scene:\n\n" + object_summary(categorized, spatial_zones, annotations)
              + "\n\nCreate a complete scene graph with all hierarchical levels filled.")
    if context:
        prompt += f"\n\nAdditional context from other sensors:\n{json.dumps(context, indent=2)[:500]}"
    return prompt


def image_to_base64(img: np.ndarray) -> str:
    """lidar_agent.py:819-832: uint8 conversion, BGR -> RGB, PNG through Pillow, base64."""
    from PIL import Image
    if img.dtype != np.uint8:
        img = (img * 255).astype(np.uint8)
    if img.ndim == 3 and img.shape[2] == 3:
        img = np.ascontiguousarray(img[:, :, ::-1])  # cv2.cvtColor(img, cv2.COLOR_BGR2RGB) is a channel reversal
    buf = BytesIO()
    Image.fromarray(img).save(buf, format="PNG")
    return base64.b64encode(buf.getvalue()).decode()


def jpeg_base64(img: np.ndarray) -> str:
    """camera_agent.py:128-137: uint8 conversion, JPEG quality 85 through Pillow (no channel swap: camera images are RGB), base64."""
    from PIL import Image
    if img.dtype != np.uint8:
        img = (img * 255).astype(np.uint8)
    buf = BytesIO()
    Image.fromarray(img).save(buf, format="JPEG", quality=85)
    return base64.b64encode(buf.getvalue()).decode()


def ext_evidence(annotations: Sequence[Dict], box_count: np.ndarray, box_nearest: np.ndarray, box_centroid: np.ndarray,
                 proj_visible: np.ndarray, camera_names: Sequence[str], relations: Optional[Dict[str, Any]] = None,
                 max_pairs: int = 20, camera_support: Optional[np.ndarray] = None, cluster_match: Optional[np.ndarray] = None) -> Dict[str, Any]:
    """[EXT] evidence of one sample (rows e3, e5, e6 of SURVEY.md section 8a) as a JSON-serialisable dict: the `context` a caller
    hands to CameraAgent.process / SceneGraphAgent.process.  Floats are rounded the way the reference rounds distances (1 decimal).
    camera_support: the sample's box_support [B, C, 4] of msc_camera_depth_batch (row e7); adds per object "lidar_in_camera" with the
    block counts of every camera the box is visible in.  cluster_match: the sample's box table [B, 5] of msc_cluster_match_batch; adds per
    object "lidar_cluster" with the object rows inside the box and the LiDAR clusters they belong to, for boxes that hold a cluster."""
    objs = []
    for i, a in enumerate(annotations):
        n = int(box_count[i])
        cams = [camera_names[c] for c in range(len(camera_names)) if proj_visible[i, c]]
        objs.append({"id": f"obj_{i}", "category": str(a.get("category_name", "unknown")), "lidar_points": n,
                     "nearest_point_m": None if n == 0 else round(float(box_nearest[i]), 1),
                     "centroid": None if n == 0 else [round(float(v), 1) for v in box_centroid[i]], "visible_in": cams})
        if camera_support is not None:
            objs[-1]["lidar_in_camera"] = {camera_names[c]: {"blocks": int(camera_support[i, c, 0]), "blocks_with_returns": int(camera_support[i, c, 1]),
                                                             "on_object": int(camera_support[i, c, 3]), "occluded": int(camera_support[i, c, 2])}
                                           for c in range(len(camera_names)) if camera_support[i, c, 0]}
        if cluster_match is not None and int(cluster_match[i, 2]) > 0:
            objs[-1]["lidar_cluster"] = {"rows": int(cluster_match[i, 0]), "clusters": int(cluster_match[i, 2])}
    out: Dict[str, Any] = {"objects": objs}
    if relations is not None:
        labels = relations.get("labels", ("ahead", "left", "behind", "right"))
        dist, cat, ov = relations["dist"], relations["category"], relations["overlap"]
        n = dist.shape[0]
        pairs = sorted(((float(dist[i, j]), i, j) for i in range(n) for j in range(n) if i != j))[:max_pairs]
        out["nearest_pairs"] = [{"from": f"obj_{i}", "to": f"obj_{j}", "distance_m": round(d, 1), "relation": labels[int(cat[i, j])],
                                 "footprints_overlap": bool(ov[i, j])} for d, i, j in pairs]
    return out
