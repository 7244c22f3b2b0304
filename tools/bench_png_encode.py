"""Time the device PNG encode of the LiDAR agent's images (msc_png_encode_batch / GeometryEngine.run_png_encode) on the benchmark's batch:
592 samples of BASELINE config 3 (37 distinct synthetic samples tiled on the device like bench.py), against Pillow on all host cores over
the same images.

    python tools/bench_png_encode.py [--samples 592] [--calls 10] [--warmup 2]

Two device workloads, each one run_png_encode call timed with CUDA events (median over --calls after --warmup, files kept on the device):
the 800 x 800 semantic BEV of every sample (swap_rb, read in place), and the classifier mosaic of every group of ten clusters
(run_cluster_mosaics over run_cluster_views of every cluster of at least 5 points).  Pillow encodes the same images (BGR -> RGB on the
host beforehand, not timed) in a process pool of os.cpu_count() workers; its wall time is taken once.  Every device file is checked: it
inflates to Pillow's payload.  process_batch runs end to end with stub callables twice -- png=True, and png=False followed by
serialize.image_to_base64 of every BEV and mosaic it handed over -- each timed with a host clock once after a warm-up.  The card's name and
power limit are read in the same run."""
import argparse
import base64
import json
import os
import sys
import time
import zlib
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "multimodal-scene-captioning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from msc_geom import serialize  # noqa: E402
from msc_geom.engine import GeometryEngine  # noqa: E402
from msc_geom.layout import pack_batch  # noqa: E402
from msc_geom.lidar_agent import LiDARAgent, set_order  # noqa: E402
from msc_geom.synthetic import make_sample  # noqa: E402
from tools.bench_lidar_batch import card, timed  # noqa: E402

_HOST = []  # images the pool's workers encode (inherited at fork)


def _pillow(k: int) -> bytes:
    import io
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(_HOST[k]).save(buf, "PNG")
    return buf.getvalue()


def _payload(data: bytes) -> bytes:
    i, idat = 8, []
    while i < len(data):
        n = int.from_bytes(data[i:i + 4], "big")
        if data[i + 4:i + 8] == b"IDAT":
            idat.append(data[i + 8:i + 8 + n])
        i += 12 + n
    return zlib.decompress(b"".join(idat))


def pillow_all_cores(imgs):
    _HOST[:] = imgs
    with ProcessPoolExecutor(os.cpu_count()) as ex:
        list(ex.map(_pillow, range(min(len(imgs), os.cpu_count())), chunksize=1))  # start the workers
        t0 = time.perf_counter()
        files = list(ex.map(_pillow, range(len(imgs)), chunksize=1))
        return time.perf_counter() - t0, files


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=592)
    ap.add_argument("--unique", type=int, default=37)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_png_encode needs a CUDA device")
    torch.cuda.set_device(0)
    eng = GeometryEngine(0)
    agent = LiDARAgent(object(), "m", "LiDARAgent", engine=eng)
    res_px, rng = int(agent.bev_resolution), float(agent.bev_range)
    n_u = max(1, min(args.unique, args.samples))
    samples = [make_sample(i, n_sweeps=10, n_boxes=60) for i in range(n_u)]
    db = eng.upload_tiled(pack_batch(samples), (args.samples + n_u - 1) // n_u, args.samples)
    lr = eng.run_lidar(db, params=agent._params(), eps=agent.dbscan_eps, min_samples=agent.dbscan_min_samples)
    per = lr.to_host()
    orders = [[l for l in set_order(r["cluster_first"], r["noise_first"]) if int(r["clusters"][l, 10]) >= 5]
              if len(r["object"]) >= agent.dbscan_min_samples else [] for r in per]
    views = np.array([(r["object_off"], r["object_off"] + len(r["object"]), l) for r, o in zip(per, orders) for l in o], np.int64).reshape(-1, 3)
    groups, base = [], 0
    for o in orders:
        groups += [(base + a, min(10, len(o) - a)) for a in range(0, len(o), 10)]
        base += len(o)

    bev = eng.run_lidar_bev(lr, res_px, rng)
    bev.check()
    vr = eng.run_cluster_views(lr.object, lr.labels, views)
    vr.check()
    mos = eng.run_cluster_mosaics(vr, groups)
    bev_imgs, mos_imgs = list(bev.semantic), mos.images
    bev_out, mos_out = eng.alloc_png(bev_imgs, True), eng.alloc_png(mos_imgs, True)
    bev_ms = timed(lambda: eng.run_png_encode(bev_imgs, True, out=bev_out), args.calls, args.warmup)
    mos_ms = timed(lambda: eng.run_png_encode(mos_imgs, True, out=mos_out), args.calls, args.warmup)
    dev_files = bev_out.to_host() + mos_out.to_host()
    del vr

    host = [np.ascontiguousarray(t.cpu().numpy()[..., ::-1]) for t in bev_imgs] + [np.ascontiguousarray(t.cpu().numpy()[..., ::-1]) for t in mos_imgs]
    raw_bytes = sum(im.shape[0] * (1 + im.shape[1] * 3) for im in host)
    pil_bev_s, pil_bev = pillow_all_cores(host[:len(bev_imgs)])
    pil_mos_s, pil_mos = pillow_all_cores(host[len(bev_imgs):])
    pil_files = pil_bev + pil_mos
    _HOST[:] = []
    bad = sum(_payload(d) != _payload(p) for d, p in zip(dev_files, pil_files))
    del host

    # process_batch with stub callables: png=True against png=False plus image_to_base64 of every payload
    def run(png):
        payloads = []
        stub = LiDARAgent(object(), "m", "LiDARAgent", engine=eng, llm=lambda *a, **kw: payloads.append(kw.get("bev_png", kw.get("bev_semantic"))) or "",
                          cluster_classifier=lambda images, mosaic, meta: payloads.append(mosaic) or [{"category": "car", "confidence": 0.9} for _ in meta])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        stub.process_batch(device_batch=db, png=png)
        if not png:
            payloads = [serialize.image_to_base64(p) for p in payloads]
        torch.cuda.synchronize()
        return time.perf_counter() - t0, payloads
    run(True)
    png_s, png_payloads = run(True)
    run(False)
    arr_s, arr_payloads = run(False)
    bad_wire = sum(_payload(base64.b64decode(a)) != _payload(base64.b64decode(b)) for a, b in zip(png_payloads, arr_payloads))
    bad_wire += len(png_payloads) != len(arr_payloads)

    dev_b, pil_b = [len(f) for f in dev_files], [len(f) for f in pil_files]
    out = {"gpu": None, "power_limit": None, "samples": len(per), "host_cpus": os.cpu_count(), "bevs": len(bev_imgs), "mosaics": len(mos_imgs),
           "clusters": int(len(views)), "raw_payload_mb": round(raw_bytes / 1e6, 1),
           "device_bev_encode_ms": round(bev_ms, 3), "device_mosaic_encode_ms": round(mos_ms, 3),
           "pillow_all_cores_bev_ms": round(pil_bev_s * 1e3, 1), "pillow_all_cores_mosaic_ms": round(pil_mos_s * 1e3, 1),
           "device_speedup_vs_pillow_all_cores": round((pil_bev_s + pil_mos_s) * 1e3 / (bev_ms + mos_ms), 2),
           "size_ratio_total": round(sum(dev_b) / sum(pil_b), 4), "size_ratio_worst": round(max(d / p for d, p in zip(dev_b, pil_b)), 4),
           "size_ratio_bev": round(sum(dev_b[:len(bev_imgs)]) / sum(pil_b[:len(bev_imgs)]), 4),
           "size_ratio_mosaic": round(sum(dev_b[len(bev_imgs):]) / max(1, sum(pil_b[len(bev_imgs):])), 4),
           "device_png_mb": round(sum(dev_b) / 1e6, 2), "pillow_png_mb": round(sum(pil_b) / 1e6, 2),
           "process_batch_png_ms": round(png_s * 1e3, 1), "process_batch_arrays_plus_image_to_base64_ms": round(arr_s * 1e3, 1),
           "files_with_a_payload_differing_from_pillow": int(bad), "wire_payloads_differing": int(bad_wire)}
    out["gpu"], out["power_limit"] = card()
    print(json.dumps(out))
    if bad or bad_wire:
        raise SystemExit("device files differ from Pillow's payload: %d files, %d wire payloads" % (bad, bad_wire))


if __name__ == "__main__":
    main()
