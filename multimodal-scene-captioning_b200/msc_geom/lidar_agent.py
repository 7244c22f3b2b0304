"""LiDARAgent -- host-side mirror of the reference agent's LOCAL half
(/root/reference/src/agents/content_transform/lidar_agent.py), with the numeric work on the GPU.

Same constructor, attribute names, method names, argument meaning and return shapes as the reference
(SURVEY.md section 8(b)), so the three geometry methods the reference's scripts call directly
(src/export_sample_data.py:59-65, src/generate_detailed_logs.py:213-215) and `process()` are drop-ins.
What stays on the host, and why:
  * the cluster LIST ORDER follows CPython set iteration over the labels, like the reference (lidar_agent.py:154-159);
    DBSCAN itself runs on the device with scikit-learn's exact labelling (csrc/dbscan.cu).
  * the cv2 overlays drawn after the raster (lidar_agent.py:599-634) and the log1p density normalisation, which is
    evaluated with NumPy's own float32 log1p through a count -> value table so the uint8 layer is bit-identical.  process_batch
    draws both on the device for the whole batch, from the same table and from stamps of these same cv2 calls (overlay_stamp).
  * every remote LLM call: injected as callables (`llm`, `cluster_classifier`); absent callables yield the
    reference's own fallbacks ('unknown' clusters are dropped, lidar_agent.py:228).
"""
from __future__ import annotations

import base64
import json
from dataclasses import dataclass
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import ops
from .engine import DeviceBatch, GeometryEngine
from .layout import GeomParams, pack_batch

CLUSTER_IMAGES_PER_CALL = 1024  # cluster images process_batch draws per device call and holds on the host (768 KiB each)
DIRECTION_LABELS = ("front_right", "front", "front_left", "left", "back_left", "back", "back_right", "right")


@dataclass
class DetectedObject:
    """Same fields as the reference dataclass (lidar_agent.py:18-27)."""
    category: str
    position: np.ndarray
    dimensions: np.ndarray
    num_points: int
    distance: float
    direction: str
    confidence: float


def direction_label(position_2d) -> str:
    """8-way label of lidar_agent.py:506-530: 45-degree bins starting at 337.5, in the reference's (rotated) label order."""
    x, y = position_2d
    angle = (np.arctan2(y, x) * 180 / np.pi + 360) % 360
    if angle >= 337.5 or angle < 22.5:
        return DIRECTION_LABELS[0]
    lo = 22.5
    for label in DIRECTION_LABELS[1:7]:
        if lo <= angle < lo + 45.0:
            return label
        lo += 45.0
    return DIRECTION_LABELS[7]


def density_table(cmax: int) -> np.ndarray:
    """log1p(c) for c = 0..cmax with NumPy's own float32 log1p (lidar_agent.py:563): the BEV density of a cell of c rows, on the host and
    through msc_keyframe_bev_batch.  NumPy may pick a CPU-dependent SIMD log1p, so the table is always computed here, never on the device."""
    return np.log1p(np.arange(cmax + 1, dtype=np.float32))


def finish_bev_layers(count: np.ndarray, height: np.ndarray, semantic: np.ndarray, res: int, bev_range) -> Dict[str, np.ndarray]:
    """Host half of _generate_multi_layer_bev: density normalisation (lidar_agent.py:563-564), ego cross, vertical
    flips, range rings and labels (:599-634).  `count`/`height`/`semantic` are the unflipped GPU raster layers."""
    import cv2
    cmax = int(count.max()) if count.size else 0
    lut = density_table(cmax)
    dens = lut[count.astype(np.int64)]
    density = (dens / dens.max() * 255).astype(np.uint8) if cmax > 0 else dens.astype(np.uint8)
    vis = np.ascontiguousarray(semantic)
    c, arm = res // 2, 15
    green = (0, 255, 0)
    cv2.line(vis, (c - arm, c), (c + arm, c), green, 3)
    cv2.line(vis, (c, c - arm), (c, c + arm), green, 3)
    vis, height, density = (cv2.flip(np.ascontiguousarray(a), 0) for a in (vis, height, density))
    for metres in (10, 20, 30, 40):
        radius = int(metres / (2 * bev_range) * res)
        cv2.circle(vis, (c, c), radius, (100, 100, 100), 1)
        cv2.putText(vis, f"{metres}m", (c + 5, c - radius + 15), cv2.FONT_HERSHEY_SIMPLEX, 0.4, (150, 150, 150), 1)
    for text, org in (("FRONT", (c - 25, 20)), ("BACK", (c - 20, res - 10)), ("L", (10, c + 5)), ("R", (res - 20, c + 5))):
        cv2.putText(vis, text, org, cv2.FONT_HERSHEY_SIMPLEX, 0.6, (200, 200, 200), 2)
    return {"semantic": vis, "height": height, "density": density}


def finish_cluster_view(grid: np.ndarray, img_size: int = 256) -> np.ndarray:
    """Host half of _generate_cluster_visualization: axes and titles (lidar_agent.py:299-313, :353-354) on top of the GPU
    disc raster.  They sit well inside their quadrant, a disc bleeds at most two pixels over a quadrant border, so drawing
    them after all discs gives the reference's image."""
    import cv2
    grid = np.ascontiguousarray(grid)
    half = img_size // 2
    for qx, qy, title in ((0, 0, "Top (XY)"), (1, 0, "Side (XZ)"), (0, 1, "Front (YZ)"), (1, 1, "3D View")):
        ox, oy = qx * img_size, qy * img_size
        if (qx, qy) != (1, 1):
            cv2.line(grid, (ox + half, oy + half), (ox + half + 30, oy + half), (0, 0, 255), 2)   # x axis, red
            cv2.line(grid, (ox + half, oy + half), (ox + half, oy + half - 30), (0, 255, 0), 2)   # y axis, green
        cv2.putText(grid, title, (ox + 10, oy + 20), cv2.FONT_HERSHEY_SIMPLEX, 0.5, (0, 0, 0), 1)
    return grid


def overlay_stamp(draw: Callable[[np.ndarray], np.ndarray], h: int, w: int) -> np.ndarray:
    """The pixels an opaque overlay sets, as u32 [m, 2] = (pixel y * w + x, B | G << 8 | R << 16): what `draw(canvas)` changes on an all-0
    or an all-255 BGR canvas of h x w, with the colour it leaves there.  cv2's line / circle / putText with the default LINE_8 are opaque
    (pixels and colours do not depend on the canvas), so writing the stamp over any raster equals drawing on it."""
    lo, hi = draw(np.zeros((h, w, 3), np.uint8)), draw(np.full((h, w, 3), 255, np.uint8))
    mask = (lo != 0).any(-1) | (hi != 255).any(-1)
    if not np.array_equal(lo[mask], hi[mask]):
        raise ValueError("overlay_stamp: the overlay depends on the canvas")
    px = np.flatnonzero(mask.ravel())
    c = lo.reshape(-1, 3)[px].astype(np.uint32)
    return np.stack([px.astype(np.uint32), c[:, 0] | (c[:, 1] << 8) | (c[:, 2] << 16)], 1)


def bev_stamp(res: int, bev_range) -> np.ndarray:
    """The overlays of finish_bev_layers (ego cross, rings, labels) on a res x res BEV, as an overlay_stamp."""
    zero = np.zeros((res, res), np.uint32)
    return overlay_stamp(lambda canvas: finish_bev_layers(zero, zero.view(np.float32), canvas, res, bev_range)["semantic"], res, res)


def cluster_view_stamp() -> np.ndarray:
    """The axes and titles of finish_cluster_view on a 512 x 512 cluster image, as an overlay_stamp."""
    return overlay_stamp(finish_cluster_view, 512, 512)


def cluster_mosaic(images: List[np.ndarray]) -> np.ndarray:
    """The batch image of _classify_batch_with_llm (lidar_agent.py:366-386): up to three columns, '#idx' labels."""
    import cv2
    if len(images) == 1:
        return images[0]
    cols = min(3, len(images))
    rows = (len(images) + cols - 1) // cols
    h, w = images[0].shape[:2]
    sheet = np.full((rows * h, cols * w, 3), 255, dtype=np.uint8)
    for idx, img in enumerate(images):
        r, c = divmod(idx, cols)
        sheet[r * h:(r + 1) * h, c * w:(c + 1) * w] = img
        cv2.putText(sheet, f"#{idx}", (c * w + 10, r * h + 50), cv2.FONT_HERSHEY_SIMPLEX, 1.5, (255, 0, 0), 3)
    return sheet


def mosaic_stamp(count: int) -> np.ndarray:
    """The '#idx' labels and the white empty cells cluster_mosaic draws on a mosaic of `count` (2..10) views, as an overlay_stamp: what
    cluster_mosaic of the canvas's own 512 x 512 cells changes.  Written over the views copied into their cells, it gives the mosaic."""
    rows, cols = (count + 2) // 3, min(3, count)

    def draw(canvas):
        return cluster_mosaic([canvas[r * 512:(r + 1) * 512, c * 512:(c + 1) * 512] for r, c in (divmod(i, cols) for i in range(count))])
    return overlay_stamp(draw, rows * 512, cols * 512)


def set_order(cluster_first, noise_first: int) -> List[int]:
    """The cluster labels (noise excluded) in the order `s = set(labels); s.discard(-1)` iterates them (lidar_agent.py:154-159), from
    each label's first row alone: cluster_first[k] is the smallest index of a row labelled k (a sequence over k = 0..K-1, or a dict
    label -> row), noise_first that of the first noise row (-1: none).  CPython lays a set out from the sequence of NEW keys inserted, so
    set(labels) iterates like the set of the distinct labels inserted in first-appearance order -- noise included, since -1 takes a slot
    before it is discarded.  O(K log K), with no pass over the labels."""
    items = cluster_first.items() if isinstance(cluster_first, dict) else enumerate(cluster_first)
    firsts = [(int(f), int(k)) for k, f in items]
    if noise_first >= 0:
        firsts.append((int(noise_first), -1))
    firsts.sort()
    uniq = set(label for _, label in firsts)
    uniq.discard(-1)
    return list(uniq)


def annotation_match(order: List[int], clusters: np.ndarray, cluster_match: np.ndarray, box_match: np.ndarray,
                     annotations: Optional[Sequence[dict]] = None) -> Dict[str, List[dict]]:
    """The "annotation_match" of one sample (LiDARAgent.process_batch(match_annotations=True)) from its run_lidar cluster table
    `clusters` (K, 11), its run_cluster_match tables cluster_match (K, 3) and box_match (B, 5) and the classifier's cluster order:
      clusters:    per cluster of `order`, in that order: index (its position in `order`), num_points, annotation ("obj_<j>": the
                   annotation j holding most of its rows; None: no row in any box), category (that annotation's category_name when the
                   annotation dicts are given, else None) and points_in_annotation (its rows inside annotation j);
      annotations: per annotation j: id "obj_<j>", rows (object rows inside, noise included), clusters (clusters with a row inside) and
                   best_cluster (the index in `clusters` of the cluster with most rows inside; None when there is none or it is not in
                   the classifier's order)."""
    index_of = {int(l): i for i, l in enumerate(order)}
    cl = []
    for i, l in enumerate(order):
        b, pts = int(cluster_match[l, 0]), int(cluster_match[l, 1])
        cat = str(annotations[b].get("category_name", "unknown")) if annotations is not None and b >= 0 else None
        cl.append({"index": i, "num_points": int(clusters[l, 10]), "annotation": f"obj_{b}" if b >= 0 else None, "category": cat,
                   "points_in_annotation": pts})
    anns = [{"id": f"obj_{j}", "rows": int(r[0]), "clusters": int(r[2]), "best_cluster": index_of.get(int(r[3]))} for j, r in enumerate(box_match)]
    return {"clusters": cl, "annotations": anns}


class LiDARAgent:
    def __init__(self, client, model: str, agent_name: str, engine: Optional[GeometryEngine] = None,
                 llm: Optional[Callable[..., str]] = None, cluster_classifier: Optional[Callable[..., List[dict]]] = None):
        self.client, self.model, self.agent_name = client, model, agent_name
        self.dbscan_eps = 0.5          # lidar_agent.py:44
        self.dbscan_min_samples = 10   # :45
        self.bev_resolution = 800      # :48
        self.bev_range = 50            # :49
        self.engine = engine or GeometryEngine()
        self.llm = llm
        self.cluster_classifier = cluster_classifier

    # ------------------------------------------------------------------ remote half (injected)
    def call_llm(self, messages, temperature: float = 0.7, **kw) -> str:
        if self.llm is None:
            return ""
        return self.llm(messages, temperature=temperature, **kw)

    # ------------------------------------------------------------------ local geometry (GPU)
    def _params(self, ground_threshold: float = -1.4) -> GeomParams:
        return GeomParams(range_max=float(self.bev_range), bev_range=float(self.bev_range), bev_res=int(self.bev_resolution),
                          ground_z=float(ground_threshold))

    def _preprocess_point_cloud(self, pc: np.ndarray) -> np.ndarray:
        return ops.keyframe_filter_split(self.engine, pc, self._params())[0]

    def _segment_ground(self, pc: np.ndarray, ground_threshold: float = -1.4) -> Tuple[np.ndarray, np.ndarray]:
        _, ground, obj = ops.keyframe_filter_split(self.engine, pc, self._params(ground_threshold), split_only=True)
        return ground, obj

    def _generate_multi_layer_bev(self, ground_points: np.ndarray, object_points: np.ndarray) -> Dict[str, np.ndarray]:
        res, r = int(self.bev_resolution), self.bev_range
        count, height, sem = ops.keyframe_bev_layers(self.engine, ground_points, object_points, res, float(r))
        return finish_bev_layers(count, height, sem, res, r)

    def _generate_cluster_visualization(self, points: np.ndarray, img_size: int = 256) -> np.ndarray:
        """One cluster -> 512x512 4-view image (lidar_agent.py:241-356)."""
        if img_size != 256:
            raise ValueError("the device raster is built for the reference's img_size = 256")
        return finish_cluster_view(ops.cluster_views(self.engine, points, [np.arange(len(points))])[0])

    def _cluster_visualizations(self, object_points: np.ndarray, labels: np.ndarray, order: List[int]) -> List[np.ndarray]:
        """All clusters of a cloud in one launch (the reference loops over clusters, lidar_agent.py:198-209)."""
        discs = ops.cluster_views(self.engine, object_points, [np.nonzero(labels == l)[0] for l in order])
        return [finish_cluster_view(d) for d in discs]

    def _cluster_metadata(self, object_points: np.ndarray, labels: np.ndarray, order: List[int]) -> List[dict]:
        n_clusters = int(labels.max()) + 1 if labels.size else 0
        return self._metadata_of(ops.cluster_aabb(self.engine, object_points, labels, n_clusters), order)

    @staticmethod
    def _metadata_of(table: np.ndarray, order: List[int]) -> List[dict]:
        """Cluster metadata (lidar_agent.py:198-209) of the clusters in `order` from their msc_cluster_aabb rows."""
        meta = []
        for i, lab in enumerate(order):
            row = table[lab]
            mn, mx, center = row[0:3], row[3:6], row[6:9]
            meta.append({"index": i, "center": center.copy(), "dimensions": mx - mn, "distance": row[9], "direction": direction_label(center[:2]),
                         "num_points": int(row[10])})
        return meta

    def _detect_objects_3d(self, object_points: np.ndarray) -> List[DetectedObject]:
        """lidar_agent.py:134-239 with the local work on the device: DBSCAN (scikit-learn's labelling), per-cluster boxes, and the
        4-view images of ALL clusters in one launch; the classifier sees what the reference's sees -- per batch of ten, the cluster
        images and their metadata (`_classify_batch_with_llm(cluster_images, cluster_metadata)`, :358)."""
        if len(object_points) < self.dbscan_min_samples:
            return []
        labels = ops.dbscan(self.engine, object_points, self.dbscan_eps, self.dbscan_min_samples)
        uniq = set(labels)
        uniq.discard(-1)
        order = [int(l) for l in uniq if int((labels == l).sum()) >= 5]  # set-iteration order, like lidar_agent.py:154-165
        if not order:
            return []
        labels = labels.astype(np.int32)
        meta = self._cluster_metadata(object_points, labels, order)
        images = self._cluster_visualizations(object_points, labels, order)
        return self._classified_objects(meta, lambda a, b: images[a:b])

    def _classified_objects(self, meta: List[dict], images_of: Callable[[int, int], Any],
                            classify: Optional[Callable[[Any, List[dict]], List[dict]]] = None) -> List[DetectedObject]:
        """The classifier loop of lidar_agent.py:189-239; images_of(a, b) gives the images of clusters a..b-1 of `meta`, which
        classify(images, metadata) (default: _classify_batch_with_llm) classifies."""
        classify = classify or self._classify_batch_with_llm
        out: List[DetectedObject] = []
        for start in range(0, len(meta), 10):  # the reference classifies in batches of 10 (:189)
            batch = meta[start:start + 10]
            cls = classify(images_of(start, start + len(batch)), batch)
            for m, c in zip(batch, cls):
                if c["category"] != "unknown" and c["confidence"] > 0.3:
                    out.append(DetectedObject(c["category"], m["center"], m["dimensions"], m["num_points"], m["distance"], m["direction"],
                                              c["confidence"]))
        return out

    def _classify_batch_with_llm(self, cluster_images: List[np.ndarray], cluster_metadata: List[dict]) -> List[dict]:
        """The remote half of lidar_agent.py:358-504, injected: `cluster_classifier(images, mosaic, metadata)` gets the batch's cluster
        images, the mosaic the reference would send (:366-386) and the metadata.  Without one every cluster takes the reference's
        parse-failure default (:503)."""
        if self.cluster_classifier is None:
            return [{"category": "unknown", "confidence": 0.5} for _ in cluster_metadata]
        return self.cluster_classifier(cluster_images, cluster_mosaic(cluster_images), cluster_metadata)

    # ------------------------------------------------------------------ evidence -> features / report (host, tiny)
    def _extract_semantic_features(self, detected_objects: List[DetectedObject], ground_points: np.ndarray, object_points: np.ndarray) -> Dict[str, Any]:
        counts: Dict[str, int] = {}
        by_dir = {d: 0 for d in ("front", "back", "left", "right", "front_left", "front_right", "back_left", "back_right")}
        close = medium = far = vehicles = 0
        for o in detected_objects:
            counts[o.category] = counts.get(o.category, 0) + 1
            by_dir[o.direction] += 1
            if o.distance < 10:
                close += 1
            elif o.distance < 30:
                medium += 1
            else:
                far += 1
            vehicles += o.category in ("car", "truck", "bus")
        total = len(ground_points) + len(object_points)
        ratio = len(object_points) / total if total > 0 else 0
        return {
            "total_objects": len(detected_objects), "object_counts": counts, "objects_by_direction": by_dir,
            "distance_distribution": {"close": close, "medium": medium, "far": far},
            "scene_characteristics": {"object_point_ratio": float(ratio),
                                      "traffic_density": "heavy" if vehicles > 10 else "moderate" if vehicles > 5 else "light",
                                      "total_points": total},
            "nearest_object": min(detected_objects, key=lambda o: o.distance) if detected_objects else None,
        }

    def _generate_structured_report(self, semantic_features: Dict[str, Any], detected_objects: List[DetectedObject]) -> str:
        f = semantic_features
        lines = ["=== LiDAR Scene Analysis ===\n", f"Total detected objects: {f['total_objects']}"]
        if f["object_counts"]:
            lines.append("\nObject Distribution:")
            lines += [f"  - {n} {cat}(s)" for cat, n in sorted(f["object_counts"].items())]
        lines.append("\nSpatial Distribution:")
        for direction, n in f["objects_by_direction"].items():
            if n > 0:
                cats = ", ".join(set(o.category for o in detected_objects if o.direction == direction))
                lines.append(f"  - {direction}: {n} objects ({cats})")
        d = f["distance_distribution"]
        lines += ["\nDistance Distribution:", f"  - Close (<10m): {d['close']} objects", f"  - Medium (10-30m): {d['medium']} objects",
                  f"  - Far (>30m): {d['far']} objects"]
        near = f["nearest_object"]
        if near:
            lines += ["\nNearest Object:", f"  - Type: {near.category}", f"  - Distance: {near.distance:.1f}m", f"  - Direction: {near.direction}"]
        sc = f["scene_characteristics"]
        lines += ["\nScene Characteristics:", f"  - Traffic density: {sc['traffic_density']}", f"  - Object point ratio: {sc['object_point_ratio']:.2%}"]
        return "\n".join(lines)

    @staticmethod
    def _object_to_dict(obj: DetectedObject) -> Dict[str, Any]:
        return {"category": obj.category, "position": obj.position.tolist(), "dimensions": obj.dimensions.tolist(), "num_points": obj.num_points,
                "distance": float(obj.distance), "direction": obj.direction, "confidence": float(obj.confidence)}

    # ------------------------------------------------------------------ entry point (lidar_agent.py:51-101)
    def process(self, point_cloud: np.ndarray, context: Optional[Dict] = None) -> Dict[str, Any]:
        kept, ground, obj = ops.keyframe_filter_split(self.engine, point_cloud, self._params())
        detected = self._detect_objects_3d(obj)
        bev = self._generate_multi_layer_bev(ground, obj)
        return self._result(detected, ground, obj, bev, context)

    def process_batch(self, samples: Optional[Sequence[dict]] = None, device_batch: Optional[DeviceBatch] = None,
                      contexts: Optional[Sequence[Optional[Dict]]] = None, match_annotations: bool = False,
                      annotations: Optional[Sequence[Sequence[dict]]] = None, png: bool = False) -> List[Dict[str, Any]]:
        """[process(sample["point_cloud"], context) for each sample], with the filter, the ground split, DBSCAN and the cluster boxes of
        every sample's keyframe (sweep 0) in one device pass (GeometryEngine.run_lidar).  `device_batch` (e.g. engine.upload of
        io.stage_batch over lazy-loader samples, whose point_cloud is None) is used as it is; otherwise `samples` are packed and uploaded.
        The classifier sees the same images, mosaics and metadata in the same order as process's; the 800 x 800 BEV, which only the
        scene interpretation reads, is drawn only when an llm is injected (GeometryEngine.run_lidar_bev, enqueued behind run_lidar), and
        cluster images only when a classifier is (GeometryEngine.run_cluster_views, CLUSTER_IMAGES_PER_CALL clusters at a time).
        match_annotations=True adds to each result the key "annotation_match" (lidar_agent.annotation_match): which annotated box each
        cluster of the classifier's order lies in and which clusters each box holds (GeometryEngine.run_cluster_match, enqueued behind
        run_lidar).  Categories come from the samples' annotation dicts, or from `annotations` (one list per sample) for a device_batch.
        png=True hands each callable what goes on the wire, encoded on the device (ops.encode_png_batch) so that only PNG bytes cross PCIe:
        the llm gets bev_png=<base64 of the BEV's PNG> instead of bev_semantic=<array>, and the classifier is called
        cluster_classifier(None, <base64 of the mosaic's PNG>, metadata) (GeometryEngine.run_cluster_mosaics on whole groups of ten)."""
        eng = self.engine
        if device_batch is None:
            if samples is None:
                raise ValueError("process_batch needs samples or a device_batch")
            device_batch = eng.upload(pack_batch(list(samples), n_cams=eng.params.n_cams))
        res = eng.run_lidar(device_batch, params=self._params(), eps=self.dbscan_eps, min_samples=self.dbscan_min_samples)
        match = eng.run_cluster_match(res, device_batch) if match_annotations else None
        bev = eng.run_lidar_bev(res, int(self.bev_resolution), float(self.bev_range)) if self.llm is not None else None
        per = res.to_host()
        matches = match.to_host() if match is not None else None
        if annotations is None and samples is not None:
            annotations = [s.get("annotations", []) for s in samples]
        if bev is None:
            bevs = [None] * len(per)
        elif png:
            bev.check()
            bevs = [{"png": base64.b64encode(f).decode("ascii")} for f in ops.encode_png_batch(eng, list(bev.semantic), swap_rb=True)]
        else:
            bevs = bev.to_host(("semantic",))
        orders = []
        for r in per:
            table = r["clusters"]
            orders.append([l for l in set_order(r["cluster_first"], r["noise_first"]) if int(table[l, 10]) >= 5]
                          if len(r["object"]) >= self.dbscan_min_samples else [])  # the guard of _detect_objects_3d
        images = None
        if self.cluster_classifier is not None:
            images = self._batch_cluster_mosaics(res, per, orders) if png else self._batch_cluster_images(res, per, orders)
        # without a classifier every path takes _classify_batch_with_llm's default
        classify = (lambda mosaic, meta: self.cluster_classifier(None, mosaic, meta)) if png and images is not None else None
        contexts = list(contexts) if contexts is not None else [None] * len(per)
        out, base = [], 0
        for s, (r, order) in enumerate(zip(per, orders)):
            detected: List[DetectedObject] = []
            if order:
                images_of = (lambda a, b, o=base: images(o + a, o + b)) if images is not None else (lambda a, b: [])
                detected = self._classified_objects(self._metadata_of(r["clusters"], order), images_of, classify)
            base += len(order)
            out.append(self._result(detected, r["ground"], r["object"], bevs[s], contexts[s]))
            if matches is not None:
                out[-1]["annotation_match"] = annotation_match(order, r["clusters"], matches[s]["cluster_match"], matches[s]["box_match"],
                                                               annotations[s] if annotations is not None else None)
        return out

    def _batch_cluster_images(self, res, per: List[Dict[str, Any]], orders: List[List[int]]) -> Callable[[int, int], List[np.ndarray]]:
        """images(a, b): the 4-view images of clusters a..b-1 of all samples' orders laid end to end, drawn on the device
        CLUSTER_IMAGES_PER_CALL at a time as they are asked for (in increasing order)."""
        views = np.array([(r["object_off"], r["object_off"] + len(r["object"]), l) for r, order in zip(per, orders) for l in order],
                         np.int64).reshape(-1, 3)
        sizes = np.array([int(r["clusters"][l, 10]) for r, order in zip(per, orders) for l in order], np.int64)
        k, held = CLUSTER_IMAGES_PER_CALL, {}

        def images(a: int, b: int) -> List[np.ndarray]:
            got = []
            for i in range(a, b):
                c = i // k
                if c not in held:
                    held.clear()
                    held[c] = self.engine.run_cluster_views(res.object, res.labels, views[c * k:(c + 1) * k],
                                                            max_view_points=int(sizes[c * k:(c + 1) * k].max())).to_host()
                got.append(held[c][i - c * k])
            return got
        return images

    def _batch_cluster_mosaics(self, res, per: List[Dict[str, Any]], orders: List[List[int]]) -> Callable[[int, int], Optional[str]]:
        """mosaic(a, b): the base64 PNG of the classifier mosaic of clusters a..b-1 of all samples' orders laid end to end (a group of
        at most ten of one sample), drawn and encoded on the device for whole groups, at most CLUSTER_IMAGES_PER_CALL views at a time, as
        they are asked for (in increasing order).  Only the PNG files are copied to the host."""
        views = np.array([(r["object_off"], r["object_off"] + len(r["object"]), l) for r, order in zip(per, orders) for l in order],
                         np.int64).reshape(-1, 3)
        sizes = np.array([int(r["clusters"][l, 10]) for r, order in zip(per, orders) for l in order], np.int64)
        groups, base = [], 0
        for order in orders:
            groups += [(base + a, min(10, len(order) - a)) for a in range(0, len(order), 10)]
            base += len(order)
        chunks, g0 = [], 0  # whole groups, at most CLUSTER_IMAGES_PER_CALL views (at least one group) per chunk
        while g0 < len(groups):
            g1 = g0 + 1
            while g1 < len(groups) and groups[g1][0] + groups[g1][1] - groups[g0][0] <= CLUSTER_IMAGES_PER_CALL:
                g1 += 1
            chunks.append((g0, g1))
            g0 = g1
        chunk_of = {groups[g][0]: c for c, (a, b) in enumerate(chunks) for g in range(a, b)}
        held: Dict[int, Dict[int, str]] = {}

        def mosaic(a: int, b: int) -> Optional[str]:
            c = chunk_of[a]
            if c not in held:
                held.clear()
                g0, g1 = chunks[c]
                v0, v1 = groups[g0][0], groups[g1 - 1][0] + groups[g1 - 1][1]
                vr = self.engine.run_cluster_views(res.object, res.labels, views[v0:v1], max_view_points=int(sizes[v0:v1].max()))
                mos = self.engine.run_cluster_mosaics(vr, [(f - v0, n) for f, n in groups[g0:g1]])
                vr.check()
                files = ops.encode_png_batch(self.engine, mos.images, swap_rb=True)
                held[c] = {groups[g][0]: base64.b64encode(f).decode("ascii") for g, f in zip(range(g0, g1), files)}
            return held[c][a]
        return mosaic

    def _result(self, detected: List[DetectedObject], ground: np.ndarray, obj: np.ndarray, bev: Optional[Dict[str, np.ndarray]],
                context: Optional[Dict]) -> Dict[str, Any]:
        features = self._extract_semantic_features(detected, ground, obj)
        report = self._generate_structured_report(features, detected)
        observations = self._scene_interpretation(report, bev, context)
        return {"agent": self.agent_name, "modality": "lidar", "detected_objects": [self._object_to_dict(o) for o in detected],
                "semantic_features": features, "structured_report": report, "observations": observations,
                "bev_metadata": {"num_objects": len(detected), "ground_points": len(ground), "object_points": len(obj)}}

    def _scene_interpretation(self, report: str, bev: Dict[str, np.ndarray], context: Optional[Dict]) -> str:
        if self.llm is None:
            return ""
        prompt = "Analyze this driving scene from LiDAR data:\n\n" + report
        if context:
            prompt += "\n\nAdditional context from other sensors:\n" + json.dumps(context, indent=2)
        if "png" in bev:
            return self.call_llm([{"role": "user", "content": prompt}], temperature=0.4, bev_png=bev["png"])
        return self.call_llm([{"role": "user", "content": prompt}], temperature=0.4, bev_semantic=bev["semantic"])


def create_lidar_agent(client, model: str, **kw) -> LiDARAgent:
    return LiDARAgent(client, model, "LiDARAgent", **kw)
