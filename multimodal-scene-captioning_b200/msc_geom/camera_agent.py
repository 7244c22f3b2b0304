"""Camera-side evidence.  The reference's CameraAgent does no geometry (camera_agent.py:12-127 is base64 + one VLM call);
its `process(images, camera_names, context=None)` JSON-dumps `context` into the prompt (:43-47), which is the natural carrier
for the [EXT] box -> camera projection evidence built here (devkit get_sample_data + view_points + box_in_image, App. A.3)."""
from __future__ import annotations

import base64
import json
from typing import Any, Callable, Dict, List, Optional

import numpy as np
import torch

from . import ops
from .engine import GeometryEngine
from .layout import DepthParams, GeomParams, boxes_from_annotations


def projection_evidence(engine: GeometryEngine, sample: Dict[str, Any], image_size=(1600, 900)) -> Dict[str, Any]:
    """Per camera: which annotations are visible and their clipped 2D extents.  Needs the additive `cameras` key
    (ego_pose, calib, intrinsic per camera); returns {} for plain reference-style samples."""
    cams = sample.get("cameras") or []
    anns = sample.get("annotations") or []
    if not cams or not anns:
        return {}
    boxes = boxes_from_annotations(anns)
    pose = np.stack([np.asarray(c.get("ego_pose", sample.get("ego_pose")), np.float64) for c in cams])
    calib = np.stack([np.asarray(c["calib"], np.float64) for c in cams])
    K = np.stack([np.asarray(c["intrinsic"], np.float64).reshape(9) for c in cams])
    vis, ext = ops.project_boxes(engine, boxes, pose, calib, K, image_size[0], image_size[1])
    out: Dict[str, Any] = {}
    for ci, c in enumerate(cams):
        rows = [{"annotation": int(i), "category": anns[i].get("category_name", "unknown"), "bbox": [round(float(v), 1) for v in ext[i, ci]]}
                for i in np.nonzero(vis[:, ci])[0]]
        out[c.get("channel", f"CAM_{ci}")] = {"visible_objects": len(rows), "objects": rows}
    return out


def lidar_evidence(engine: GeometryEngine, sample: Dict[str, Any], dp: Optional[DepthParams] = None, image_size=(1600, 900)) -> Dict[str, Any]:
    """[EXT] what LiDAR sees in each camera (devkit map_pointcloud_to_image over the sample's multi-sweep cloud, ops.camera_depth):
    per camera the number of returns that land in the image and, per visible annotation, how many ds x ds pixel blocks its projected
    box covers, how many of them hold returns, in how many the nearest return lies on the box (`on_object`) and in how many something
    nearer hides it (`occluded`).  Needs the additive `cameras` key; returns {} for plain reference-style samples."""
    cams = sample.get("cameras") or []
    if not cams:
        return {}
    anns = sample.get("annotations") or []
    res = ops.camera_depth(engine, sample, dp, GeomParams(image_w=image_size[0], image_h=image_size[1], n_cams=len(cams)))
    sup = res["box_support"]
    out: Dict[str, Any] = {}
    for ci, c in enumerate(cams):
        rows = [{"annotation": int(i), "category": anns[i].get("category_name", "unknown"), "blocks": int(sup[i, ci, 0]),
                 "blocks_with_returns": int(sup[i, ci, 1]), "on_object": int(sup[i, ci, 3]), "occluded": int(sup[i, ci, 2])}
                for i in np.nonzero(sup[:, ci, 0])[0]]
        out[c.get("channel", f"CAM_{ci}")] = {"lidar_returns": int(res["cam_points"][ci]), "objects": rows}
    return out


def evidence_context(engine: GeometryEngine, sample: Dict[str, Any], image_size=(1600, 900), lidar: bool = False) -> Dict[str, Any]:
    """The `context` argument for CameraAgent.process: the projection evidence under one key, JSON-serialisable.  lidar=True adds
    lidar_evidence under "lidar_in_camera"."""
    ev = projection_evidence(engine, sample, image_size)
    out = {"box_projection": ev} if ev else {}
    if lidar:
        lev = lidar_evidence(engine, sample, image_size=image_size)
        if lev:
            out["lidar_in_camera"] = lev
    return out


def split_camera_sections(response: str, camera_names: List[str]) -> Dict[str, str]:
    """Per-camera sections of one multi-camera reply (camera_agent.py:75-117): a section runs from the first mention of the camera's
    name (or the name with spaces) to the first later mention of any following camera; no mention of any camera at all -> every camera
    gets the whole reply; a camera that is not mentioned gets the reference's placeholder."""
    low = response.lower()
    forms = lambda name: (name.lower(), name.replace("_", " ").lower())
    if not any(name.lower() in low for name in camera_names):
        return {name: response for name in camera_names}
    out = {}
    for i, name in enumerate(camera_names):
        start = next((low.find(f) for f in forms(name) if low.find(f) != -1), -1)
        if start == -1:
            out[name] = f"(Analysis for {name} not clearly separated in response)"
            continue
        end = len(response)
        for later in camera_names[i + 1:]:
            for f in forms(later):
                k = low.find(f, start + 1)
                if k != -1 and k < end:
                    end = k
                    break
        out[name] = response[start:end].strip()
    return out


class CameraAgent:
    """Mirror of the reference's CameraAgent boundary (camera_agent.py:9-127): same `process(images, camera_names, context=None)`
    signature and result keys.  The agent has no local geometry of its own -- it base64-encodes the images and makes ONE VLM call --
    so the mirror's job is the carrier: `context` is where the [EXT] box -> camera evidence enters the prompt, rendered exactly like the
    reference renders any context (:43-47).  The VLM call is the injected `llm(messages, temperature=...)`; without one the reply is
    empty and every camera gets it, like the reference's unparsed-reply branch."""

    def __init__(self, client, model: str, agent_name: str, engine: Optional[GeometryEngine] = None, llm: Optional[Callable[..., str]] = None,
                 lidar: bool = False):
        self.client, self.model, self.agent_name = client, model, agent_name
        self.engine = engine
        self.lidar = lidar  # opt-in: process(sample=...) also puts lidar_evidence into the context
        self.llm = llm

    def call_llm(self, messages, temperature: float = 0.7, **kw) -> str:
        return "" if self.llm is None else self.llm(messages, temperature=temperature, **kw)

    @staticmethod
    def context_block(context: Optional[Dict]) -> Optional[Dict[str, str]]:
        """The text part the reference puts in front of the images when `context` is truthy (camera_agent.py:42-47)."""
        if not context:
            return None
        return {"type": "text", "text": f"Context from other sensors:\n{json.dumps(context, indent=2)}\n\n"}

    def device_jpegs(self, images: List[Any]) -> Dict[int, str]:
        """Base64 JPEG of every (H, W, 3) frame of `images` (after the reference's uint8 conversion), encoded in one device call per frame
        shape (ops.encode_jpeg_batch), keyed by position.  Other frames -- grayscale, RGBA -- are left to serialize.jpeg_base64."""
        picked, where = [], []
        for k, img in enumerate(images):
            if isinstance(img, torch.Tensor) and img.is_cuda:
                if img.dtype == torch.uint8 and img.dim() == 3 and img.shape[2] == 3:
                    picked.append(img)
                    where.append(k)
                continue
            a = np.asarray(img)
            if a.dtype != np.uint8:
                a = (a * 255).astype(np.uint8)
            if a.ndim == 3 and a.shape[2] == 3:
                picked.append(a)
                where.append(k)
        files = ops.encode_jpeg_batch(self.engine, picked, quality=85) if picked else []
        return {k: base64.b64encode(f).decode() for k, f in zip(where, files)}

    def user_content(self, images: List[np.ndarray], camera_names: List[str], context: Optional[Dict] = None) -> List[Dict[str, Any]]:
        """The reference's user message: the context block, the instruction, then every camera's name and base64 JPEG.  With an
        engine, the (H, W, 3) frames are JPEG-encoded on the device in one batch, with the same bytes as Pillow's; `images` may then also
        hold CUDA tensors (e.g. ops.decode_jpeg_batch(..., to_host=False)), so no raw frame crosses PCIe."""
        from . import serialize
        content = []
        block = self.context_block(context)
        if block:
            content.append(block)
        content.append({"type": "text", "text": f"Analyze all {len(camera_names)} camera views. For each view, provide detailed observations:\n\n"})
        frames = list(zip(images, camera_names))
        encoded = self.device_jpegs([img for img, _ in frames]) if self.engine is not None else {}
        for k, (img, name) in enumerate(frames):
            if k in encoded:
                b64 = encoded[k]
            else:
                b64 = serialize.jpeg_base64(img.cpu().numpy() if self.engine is not None and isinstance(img, torch.Tensor) else img)
            content.append({"type": "text", "text": f"Camera: {name}"})
            content.append({"type": "image_url", "image_url": {"url": f"data:image/jpeg;base64,{b64}", "detail": "low"}})
        return content

    def process(self, images: List[np.ndarray], camera_names: List[str], context: Optional[Dict] = None, sample: Optional[Dict] = None) -> Dict[str, Any]:
        """`sample` (additive): a loader sample with the `cameras` key; its projection evidence is merged into `context` (for an agent
        made with lidar=True also what LiDAR sees in each camera, lidar_evidence).  The parameter list stays the reference's."""
        if sample is not None and self.engine is not None:
            context = {**(context or {}), **evidence_context(self.engine, sample, lidar=self.lidar)}
        messages = [{"role": "user", "content": self.user_content(images, camera_names, context)}]
        response = self.call_llm(messages, temperature=0.3)
        return {"agent": self.agent_name, "modality": "camera", "camera_views": camera_names,
                "observations": split_camera_sections(response, camera_names), "full_response": response}
