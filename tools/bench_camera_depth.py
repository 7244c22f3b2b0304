"""Time msc_camera_depth_batch ([EXT] row e7) on the benchmark's batch: 592 samples of BASELINE config 3 (10 sweeps x 34,720 points,
60 boxes, 6 cameras), built like bench.py (distinct samples tiled on the device, ~4.1 GB of rows), downsample 8, with and without the
per-box support; the streaming kernel of the fused pass is timed in the same run for scale.

    python tools/bench_camera_depth.py [--samples 592] [--calls 30] [--warmup 5] [--profile DIR]

Times are CUDA events around each call on the current stream, median over --calls after --warmup.  The algorithmic bytes are what the
pass must move at least once: 20 B per point row, per sweep its pose (96 B) + start / count (8 B), per sample the offsets and poses
(ego, lidar calib, per camera ego pose, calib and K), the depth maps and cam_points written, and with support the boxes read (80 B) and
16 B per (box, camera) written.  --profile DIR adds a torch.profiler table of the three kernels (fill / depth / support) in DIR."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "multimodal-scene-captioning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from msc_geom import _capi  # noqa: E402
from msc_geom.engine import GeometryEngine  # noqa: E402
from msc_geom.layout import DepthParams, GeomParams, pack_batch  # noqa: E402
from msc_geom.synthetic import make_sample  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = "unknown (%s)" % type(e).__name__
    return name, pl


def algorithmic_bytes(hb, p: GeomParams, dp: DepthParams, support: bool) -> int:
    S, Cn, B = hb.n_samples, p.n_cams, hb.n_boxes
    hbk, wbk = dp.block_shape(p.image_w, p.image_h)
    n_sweeps = int(hb.sweep_start.shape[0])
    b = 20 * hb.n_points + (96 + 8) * n_sweeps
    b += S * (4 + 56 + 56 + Cn * (56 + 56 + 72))
    b += S * Cn * (hbk * wbk * 4 + 4)
    if support:
        b += B * 80 + S * 4 + 16 * B * Cn
    return int(b)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=592)
    ap.add_argument("--unique", type=int, default=37)
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--downsample", type=int, default=8)
    ap.add_argument("--profile", default=None, metavar="DIR")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_camera_depth needs a CUDA device")
    torch.cuda.set_device(0)
    eng = GeometryEngine(0)
    p, dp = GeomParams(), DepthParams(downsample=args.downsample)
    n_u = max(1, min(args.unique, args.samples))
    hb_u = pack_batch([make_sample(i, n_sweeps=10, n_boxes=60) for i in range(n_u)])
    db = eng.upload_tiled(hb_u, (args.samples + n_u - 1) // n_u, args.samples)
    hb = db.host
    out_s = eng.alloc_depth(hb, dp, p, box_support=True)
    out_n = eng.alloc_depth(hb, dp, p, box_support=False)
    fused = eng.alloc_result(hb, p)

    res = {"gpu": None, "power_limit": None, "samples": hb.n_samples, "points": hb.n_points, "boxes": hb.n_boxes, "downsample": dp.downsample}
    for tag, out, sup in (("with_support", out_s, True), ("depth_only", out_n, False)):
        ms = timed(lambda: eng.run_camera_depth(db, out, dp, p), args.calls, args.warmup)
        nb = algorithmic_bytes(hb, p, dp, sup)
        res[tag] = {"ms_per_step": round(ms, 4), "samples_per_s": round(hb.n_samples / (ms * 1e-3), 1), "algorithmic_bytes": nb,
                    "algorithmic_GB_per_s": round(nb / (ms * 1e-3) / 1e9, 1)}
    # the fused pass's streaming kernel in the same run, for scale (CUDA events recorded by the library around that kernel alone)
    _capi.set_option("time_kernel", 1)
    step_ms = timed(lambda: eng.run_fused(db, fused), args.calls, args.warmup)
    kt = _capi.kernel_times(args.calls)
    _capi.set_option("time_kernel", 0)
    res["fused_step_ms"] = round(step_ms, 4)
    res["streaming_kernel_ms"] = round(float(np.median(kt)), 4)
    res["depth_over_streaming_kernel"] = round(res["with_support"]["ms_per_step"] / res["streaming_kernel_ms"], 3)
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.profile, exist_ok=True)
        for _ in range(3):
            eng.run_camera_depth(db, out_s, dp, p)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(10):
                eng.run_camera_depth(db, out_s, dp, p)
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=12)
        with open(os.path.join(args.profile, "camera_depth_profile.txt"), "w") as f:
            f.write(table)
        print(table)
    res["gpu"], res["power_limit"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
