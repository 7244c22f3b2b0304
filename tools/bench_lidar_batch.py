"""Time msc_lidar_batch (the reference's keyframe evidence for a whole batch: filter + ground split, DBSCAN, cluster boxes) on the
benchmark's batch: 592 samples of BASELINE config 3 (37 distinct synthetic samples tiled on the device like bench.py; only each sample's
keyframe, sweep 0 with 34,720 rows, is read), against the per-sample loop of the latency path over the same keyframes.

    python tools/bench_lidar_batch.py [--samples 592] [--calls 20] [--warmup 3] [--eps 0.5] [--min-samples 10]

The batched call is timed with CUDA events on the current stream, median over --calls after --warmup; it stays on the device (to_host is
not in the timed window).  The per-sample loop is ops.keyframe_filter_split + ops.dbscan + ops.cluster_aabb on host arrays (host in,
host out, one host synchronisation per DBSCAN call), timed with a host clock over all samples once after one warm-up sample, and its
outputs are compared with the batch's sample by sample.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
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


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = "unknown (%s)" % type(e).__name__
    return name, pl


def timed(fn, calls: int, warmup: int):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def per_sample(eng, pc, p, eps, min_samples):
    _, ground, obj = ops.keyframe_filter_split(eng, pc, p)
    labels = ops.dbscan(eng, obj[:, :3], eps, min_samples) if len(obj) else np.zeros(0, np.int64)
    n = int(labels.max()) + 1 if labels.size else 0
    return ground, obj, labels, ops.cluster_aabb(eng, obj, labels.astype(np.int32), n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=592)
    ap.add_argument("--unique", type=int, default=37)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--eps", type=float, default=0.5)
    ap.add_argument("--min-samples", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lidar_batch needs a CUDA device")
    torch.cuda.set_device(0)
    eng = GeometryEngine(0)
    p = GeomParams(bev_res=800)  # LiDARAgent._params()
    n_u = max(1, min(args.unique, args.samples))
    samples = [make_sample(i, n_sweeps=10, n_boxes=60) for i in range(n_u)]
    db = eng.upload_tiled(pack_batch(samples), (args.samples + n_u - 1) // n_u, args.samples)
    hb = db.host
    out = eng.alloc_lidar(hb)
    ms = timed(lambda: eng.run_lidar(db, out, p, args.eps, args.min_samples), args.calls, args.warmup)
    got = out.to_host()

    keyframes = [s["lidar_sweeps"][0]["points_raw"][:, :4] for s in samples]  # 20-byte pitch view, like the devkit loader
    per_sample(eng, keyframes[0], p, args.eps, args.min_samples)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ref = [per_sample(eng, keyframes[i % n_u], p, args.eps, args.min_samples) for i in range(hb.n_samples)]
    loop_s = time.perf_counter() - t0
    mismatches = 0
    for g, (ground, obj, labels, table) in zip(got, ref):
        same = (np.array_equal(g["ground"], ground) and np.array_equal(g["object"], obj) and np.array_equal(g["labels"], labels)
                and np.array_equal(g["clusters"], table))
        mismatches += not same
    res = {"gpu": None, "power_limit": None, "samples": hb.n_samples, "keyframe_rows": out.row_capacity,
           "object_rows": int(sum(len(g["object"]) for g in got)), "clusters": int(sum(len(g["clusters"]) for g in got)),
           "batch_ms_per_call": round(ms, 4), "batch_samples_per_s": round(hb.n_samples / (ms * 1e-3), 1),
           "per_sample_loop_ms_per_sample": round(loop_s * 1e3 / hb.n_samples, 4), "per_sample_loop_samples_per_s": round(hb.n_samples / loop_s, 1),
           "speedup_vs_loop": round(loop_s * 1e3 / ms, 2), "samples_differing_from_loop": mismatches}
    res["gpu"], res["power_limit"] = card()
    print(json.dumps(res))
    if mismatches:
        raise SystemExit("the batch differs from the per-sample path on %d samples" % mismatches)


if __name__ == "__main__":
    main()
