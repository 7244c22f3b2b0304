"""Time the LiDAR agent's batched images -- msc_keyframe_bev_batch (GeometryEngine.run_lidar_bev: the finished 800 x 800 BEV of every
sample) and msc_cluster_views_batch (GeometryEngine.run_cluster_views: the finished 4-view image of every cluster of at least 5 points)
-- on the benchmark's batch: 592 samples of BASELINE config 3 (37 distinct synthetic samples tiled on the device like bench.py), against
the per-sample loop they replace in LiDARAgent.process_batch.

    python tools/bench_lidar_images.py [--samples 592] [--calls 10] [--warmup 2]

The batched calls are timed with CUDA events on the current stream, median over --calls after --warmup, once with the results kept on
the device and once with the copy to the host that process_batch makes (BEV: the semantic layer; cluster images: CLUSTER_IMAGES_PER_CALL
at a time).  The per-sample loop (ops.keyframe_bev_layers + finish_bev_layers per sample; agent._cluster_visualizations per sample) is
timed with a host clock over all samples once after one warm-up sample.  process_batch runs end to end with a stub llm and classifier.
Every batched image is compared with the loop's image of the same sample (the batch repeats the distinct samples, so the loop's images of
the distinct ones are the reference); the tool exits non-zero if any differs.  The card's name and power limit are read in the same run."""
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

from msc_geom import lidar_agent, ops  # noqa: E402
from msc_geom.engine import GeometryEngine  # noqa: E402
from msc_geom.layout import pack_batch  # noqa: E402
from msc_geom.lidar_agent import LiDARAgent, finish_bev_layers, set_order  # noqa: E402
from msc_geom.synthetic import make_sample  # noqa: E402
from tools.bench_lidar_batch import card, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=592)
    ap.add_argument("--unique", type=int, default=37)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lidar_images needs a CUDA device")
    torch.cuda.set_device(0)
    eng = GeometryEngine(0)
    agent = LiDARAgent(object(), "m", "LiDARAgent", engine=eng)
    res_px, rng = int(agent.bev_resolution), float(agent.bev_range)
    n_u = max(1, min(args.unique, args.samples))
    samples = [make_sample(i, n_sweeps=10, n_boxes=60) for i in range(n_u)]
    db = eng.upload_tiled(pack_batch(samples), (args.samples + n_u - 1) // n_u, args.samples)
    lr = eng.run_lidar(db, params=agent._params(), eps=agent.dbscan_eps, min_samples=agent.dbscan_min_samples)
    per = lr.to_host()
    S = len(per)
    orders = [[l for l in set_order(r["cluster_first"], r["noise_first"]) if int(r["clusters"][l, 10]) >= 5]
              if len(r["object"]) >= agent.dbscan_min_samples else [] for r in per]
    views = np.array([(r["object_off"], r["object_off"] + len(r["object"]), l) for r, o in zip(per, orders) for l in o], np.int64).reshape(-1, 3)
    sizes = np.array([int(r["clusters"][l, 10]) for r, o in zip(per, orders) for l in o], np.int64)
    max_pts = int(sizes.max()) if sizes.size else 0

    # ---------------------------------------------------------------- batched, on the device
    bev = eng.alloc_bev(S, res_px)
    bev_ms = timed(lambda: eng.run_lidar_bev(lr, res_px, rng, out=bev), args.calls, args.warmup)
    bev_copy_ms = timed(lambda: eng.run_lidar_bev(lr, res_px, rng, out=bev).semantic.cpu(), args.calls, args.warmup)
    got_bev = bev.to_host()
    views_out = eng.run_cluster_views(lr.object, lr.labels, views, max_view_points=max_pts)
    views_ms = timed(lambda: eng.run_cluster_views(lr.object, lr.labels, views, max_view_points=max_pts, out=views_out), args.calls, args.warmup)
    k = lidar_agent.CLUSTER_IMAGES_PER_CALL

    def views_to_host():
        for a in range(0, len(views), k):
            eng.run_cluster_views(lr.object, lr.labels, views[a:a + k], max_view_points=int(sizes[a:a + k].max())).to_host()
    views_copy_ms = timed(views_to_host, max(1, args.calls // 4), 1)

    # ---------------------------------------------------------------- the per-sample loop process_batch ran before
    def bev_loop(s):
        r = per[s]
        return finish_bev_layers(*ops.keyframe_bev_layers(eng, r["ground"], r["object"], res_px, rng), res_px, rng)

    def views_loop(s):
        r = per[s]
        return agent._cluster_visualizations(r["object"], r["labels"].astype(np.int32), orders[s]) if orders[s] else []
    bev_loop(0); views_loop(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(S):
        bev_loop(s)
    bev_loop_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    for s in range(S):
        views_loop(s)
    views_loop_s = time.perf_counter() - t0

    # ---------------------------------------------------------------- process_batch end to end, stub llm and classifier
    stub = LiDARAgent(object(), "m", "LiDARAgent", engine=eng, llm=lambda *a, **kw: "",
                      cluster_classifier=lambda images, mosaic, meta: [{"category": "car", "confidence": 0.9} for _ in meta])
    stub.process_batch(device_batch=db)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    stub.process_batch(device_batch=db)
    torch.cuda.synchronize()
    process_batch_s = time.perf_counter() - t0

    # ---------------------------------------------------------------- every image against the loop's
    bev_diff = views_diff = 0
    ref_bev = [bev_loop(u) for u in range(min(n_u, S))]
    for s in range(S):
        want = ref_bev[s % n_u]
        bev_diff += not all(np.array_equal(got_bev[s][key], want[key]) for key in ("semantic", "height", "density"))
    ref_views = [views_loop(u) for u in range(min(n_u, S))]
    owner = [(s, j) for s in range(S) for j in range(len(orders[s]))]
    if int(views_out.status.cpu()[0]):
        raise SystemExit("msc_cluster_views_batch reported a view above max_view_points")
    for a in range(0, len(views), k):
        imgs = views_out.images[a:a + k].cpu().numpy()
        views_diff += sum(not np.array_equal(img, ref_views[owner[a + j][0] % n_u][owner[a + j][1]]) for j, img in enumerate(imgs))

    out = {"gpu": None, "power_limit": None, "samples": S, "clusters_drawn": int(len(views)), "largest_cluster": max_pts,
           "bev_batch_ms": round(bev_ms, 3), "bev_batch_with_semantic_copy_ms": round(bev_copy_ms, 3),
           "cluster_views_batch_ms": round(views_ms, 3), "cluster_views_batch_with_copy_ms": round(views_copy_ms, 3),
           "bev_per_sample_loop_ms": round(bev_loop_s * 1e3, 1), "cluster_views_per_sample_loop_ms": round(views_loop_s * 1e3, 1),
           "bev_speedup_vs_loop": round(bev_loop_s * 1e3 / bev_copy_ms, 2),
           "cluster_views_speedup_vs_loop": round(views_loop_s * 1e3 / views_copy_ms, 2) if views_copy_ms else None,
           "process_batch_stub_llm_and_classifier_ms": round(process_batch_s * 1e3, 1),
           "bev_images_differing_from_loop": int(bev_diff), "cluster_images_differing_from_loop": int(views_diff)}
    out["gpu"], out["power_limit"] = card()
    print(json.dumps(out))
    if bev_diff or views_diff:
        raise SystemExit("the batched images differ from the per-sample path: %d BEVs, %d cluster images" % (bev_diff, views_diff))


if __name__ == "__main__":
    main()
