"""Time msc_cluster_match_batch (which annotated box each LiDAR cluster lies in) on the benchmark's batch: 592 samples of BASELINE config 3
(37 distinct synthetic samples with 60 boxes each, tiled on the device like bench.py), behind one run_lidar of the same batch, which is
timed too for comparison.  Also times the per-sample path (ops.cluster_match: one-sample batches, host in / host out) and a NumPy
restatement (f64 devkit points_in_box, then the counts and argmaxes) on a subset, and counts the samples whose outputs differ.

    python tools/bench_cluster_match.py [--samples 592] [--calls 20] [--warmup 3] [--subset 37]

Device calls are timed with CUDA events on the current stream, median over --calls after --warmup; results stay on the device (to_host is
not in the timed window).  The per-sample loop and the NumPy restatement run over the first --subset samples once, timed with a host
clock.  NumPy's f64 membership may differ from the f32 contract for rows within a few micrometres of a face, so its differing samples are
reported, not treated as errors.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "multimodal-scene-captioning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from msc_geom import ops  # noqa: E402
from msc_geom.engine import GeometryEngine  # noqa: E402
from msc_geom.layout import GeomParams, pack_batch  # noqa: E402
from msc_geom.synthetic import make_sample  # noqa: E402
from tools.bench_lidar_batch import card, timed  # noqa: E402


def _quat_R(q):
    w, x, y, z = np.asarray(q, np.float64) / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def numpy_match(obj, labels, K, boxes, ego_pose, lidar_calib):
    """The cluster and box tables from a devkit-style f64 points_in_box (ties: the smaller index / label)."""
    member = np.zeros((len(obj), len(boxes)), bool)
    pts = obj[:, :3].astype(np.float64)
    for b, box in enumerate(boxes):
        c, R = box[:3].astype(np.float64), _quat_R(box[6:10])
        for pose in (ego_pose, lidar_calib):
            P = _quat_R(pose[3:7])
            c, R = P.T @ (c - pose[:3]), P.T @ R
        w, l, h = box[3:6]
        p1 = R @ np.array([l / 2, w / 2, h / 2]) + c
        i, j, k = -l * R[:, 0], -w * R[:, 1], -h * R[:, 2]
        v = pts - p1
        iv, jv, kv = v @ i, v @ j, v @ k
        member[:, b] = (0 <= iv) & (iv <= i @ i) & (0 <= jv) & (jv <= j @ j) & (0 <= kv) & (kv <= k @ k)
    cnt = np.stack([member[labels == q].sum(0) for q in range(K)], 1) if K else np.zeros((len(boxes), 0), np.int64)
    box_t = np.stack([member.sum(0), member[labels >= 0].sum(0), (cnt > 0).sum(1),
                      np.where(cnt.max(1, initial=0) > 0, cnt.argmax(1) if K else -1, -1), cnt.max(1, initial=0)], 1)
    cl_t = (np.stack([np.where(cnt.max(0, initial=0) > 0, cnt.argmax(0) if len(boxes) else -1, -1), cnt.max(0, initial=0),
                      [int(member[labels == q].any(1).sum()) for q in range(K)]], 1) if K else np.zeros((0, 3), np.int64))
    return cl_t, box_t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=592)
    ap.add_argument("--unique", type=int, default=37)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--subset", type=int, default=37)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cluster_match needs a CUDA device")
    torch.cuda.set_device(0)
    eng = GeometryEngine(0)
    p = GeomParams(bev_res=800)  # LiDARAgent._params()
    n_u = max(1, min(args.unique, args.samples))
    samples = [make_sample(i, n_sweeps=10, n_boxes=60) for i in range(n_u)]
    db = eng.upload_tiled(pack_batch(samples), (args.samples + n_u - 1) // n_u, args.samples)
    hb = db.host
    lr = eng.alloc_lidar(hb)
    lidar_ms = timed(lambda: eng.run_lidar(db, lr, p), args.calls, args.warmup)
    m = eng.alloc_cluster_match(lr, hb)
    match_ms = timed(lambda: eng.run_cluster_match(lr, db, m), args.calls, args.warmup)
    per, got = lr.to_host(), m.to_host()

    sub = min(args.subset, hb.n_samples)
    ops.cluster_match(eng, samples[0], params=p)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    loop = [ops.cluster_match(eng, samples[s % n_u], params=p) for s in range(sub)]
    loop_s = time.perf_counter() - t0
    loop_diff = sum(not (np.array_equal(a["cluster_match"], g["cluster_match"]) and np.array_equal(a["box_match"], g["box_match"]))
                    for a, g in zip(loop, got))
    t0 = time.perf_counter()
    ref = []
    for s in range(sub):
        b0, b1 = int(hb.sample_box_off[s]), int(hb.sample_box_off[s + 1])
        ref.append(numpy_match(per[s]["object"], per[s]["labels"], len(per[s]["clusters"]), hb.boxes[b0:b1], hb.ego_pose[s], hb.lidar_calib[s]))
    numpy_s = time.perf_counter() - t0
    numpy_diff = sum(not (np.array_equal(cl, g["cluster_match"]) and np.array_equal(bx, g["box_match"])) for (cl, bx), g in zip(ref, got))
    res = {"gpu": None, "power_limit": None, "samples": hb.n_samples, "boxes": hb.n_boxes,
           "object_rows": int(sum(len(r["object"]) for r in per)), "clusters": int(sum(len(r["clusters"]) for r in per)),
           "clusters_matched": int(sum(int((g["cluster_match"][:, 0] >= 0).sum()) for g in got)),
           "cluster_match_ms_per_call": round(match_ms, 4), "lidar_batch_ms_per_call": round(lidar_ms, 4),
           "subset": sub, "per_sample_loop_ms_per_sample": round(loop_s * 1e3 / sub, 4), "samples_differing_from_loop": loop_diff,
           "numpy_ms_per_sample": round(numpy_s * 1e3 / sub, 4), "samples_differing_from_numpy_f64": numpy_diff}
    res["gpu"], res["power_limit"] = card()
    print(json.dumps(res))
    if loop_diff:
        raise SystemExit("the batch differs from the per-sample path on %d samples" % loop_diff)


if __name__ == "__main__":
    main()
