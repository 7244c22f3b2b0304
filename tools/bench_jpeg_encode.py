"""Time msc_jpeg_encode_batch (camera frames -> JPEG files, byte-identical to Pillow's save(..., "JPEG", quality=85)) on camera-like
1600 x 900 frames, against Pillow on every host core over the same frames.

    python tools/bench_jpeg_encode.py [--frames 3552] [--unique 64] [--chunk 592] [--calls 10] [--warmup 2] [--quality 85]

Frames: --unique seeded frames (smooth structure + texture + hard edges + noise, like the frames of tests/test_gpu_parity.py), uploaded
once and tiled on the device to --frames (distinct memory, identical content); 3552 = 592 samples x 6 cameras, the benchmark's batch.
Device timings are CUDA-event medians over --calls after --warmup, files staying on the device (to_host is not in the timed window):
  - one sample: 6 frames in one call (its 26 MB of input fits the 126 MB L2, so later calls read it from there);
  - the batch: --frames frames in calls of --chunk frames (15 GB of input, far beyond the L2; each call's workspace reserves the
    worst-case scan of its frames, 7.1 MB per frame, 4.2 GB for 592).
Bandwidth counts raw RGB read plus JPEG bytes written, against the B200's 7.7 TB/s.  Pillow runs on a thread pool of os.cpu_count()
threads (it releases the GIL while encoding), host clock over all frames once; its files are the reference every device file is
compared with, byte for byte, in the same run.  End to end: CameraAgent.user_content for one sample from device frames (one device call,
one copy back, base64) against the engine-less agent on host frames (Pillow, one core), host clock, median of --calls.  The card's name
and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from io import BytesIO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "multimodal-scene-captioning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from PIL import Image  # noqa: E402

from msc_geom.camera_agent import CameraAgent  # noqa: E402
from msc_geom.engine import GeometryEngine  # noqa: E402

CAMS = ["CAM_FRONT", "CAM_FRONT_LEFT", "CAM_FRONT_RIGHT", "CAM_BACK", "CAM_BACK_LEFT", "CAM_BACK_RIGHT"]
HBM_BYTES_PER_S = 7.7e12


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = "unknown (%s)" % type(e).__name__
    return name, pl


def frames(n, h=900, w=1600, seed=0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    out = []
    for k in range(n):
        a, b = rng.uniform(11, 31, 2)
        base = np.stack([127 + 120 * np.sin(xx / a + yy / b + k), 127 + 100 * np.cos(xx / (a / 3) + k) * np.sin(yy / b),
                         255.0 * ((xx // (7 + k % 11) + yy // (5 + k % 7)) % 2)], -1)
        out.append(np.clip(base + rng.normal(0, 6 + k % 20, (h, w, 3)), 0, 255).astype(np.uint8))
    return out


def pil_jpeg(img, q):
    buf = BytesIO()
    Image.fromarray(img).save(buf, format="JPEG", quality=q)
    return buf.getvalue()


def timed(fn, calls, warmup):
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
    ap.add_argument("--frames", type=int, default=3552)
    ap.add_argument("--unique", type=int, default=64)
    ap.add_argument("--chunk", type=int, default=592)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--quality", type=int, default=85)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_jpeg_encode needs a CUDA device")
    torch.cuda.set_device(0)
    eng = GeometryEngine(0)
    q, N = args.quality, args.frames
    uniq = frames(min(args.unique, N))
    U = len(uniq)
    H, W = uniq[0].shape[:2]
    dev_u = torch.from_numpy(np.stack(uniq)).to(eng.device)
    batch = dev_u[torch.arange(N, device=eng.device) % U].contiguous()

    # one sample: 6 frames, one call
    sample = batch[:6].contiguous()
    out6 = eng.alloc_jpeg(6, H, W)
    ms6 = timed(lambda: eng.run_jpeg_encode(sample, q, out6), args.calls, args.warmup)
    files6 = out6.to_host()

    # the batch, in calls of --chunk frames
    views = [batch[a:a + args.chunk] for a in range(0, N, args.chunk)]
    outs = {}  # one set of buffers per call size, reused by the calls of that size
    for v in views:
        if v.shape[0] not in outs:
            outs[v.shape[0]] = eng.alloc_jpeg(v.shape[0], H, W)

    def run_batch():
        for v in views:
            eng.run_jpeg_encode(v, q, outs[v.shape[0]])
    msN = timed(run_batch, args.calls, args.warmup)
    files = [f for v in views for f in eng.run_jpeg_encode(v, q, outs[v.shape[0]]).to_host()]

    # Pillow on every core over the same frames: the baseline and the reference bytes
    threads = os.cpu_count() or 1
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as pool:
        ref = list(pool.map(lambda i: pil_jpeg(uniq[i % U], q), range(N)))
    pil_s = time.perf_counter() - t0
    differ = sum(f != r for f, r in zip(files, ref)) + sum(f != ref[i] for i, f in enumerate(files6))

    # end to end, one sample: device frames -> base64 strings, against the engine-less agent on host frames
    fast, plain = CameraAgent(None, "m", "camera", engine=eng), CameraAgent(None, "m", "camera")
    host6 = [uniq[i % U] for i in range(6)]
    dev6 = [sample[i] for i in range(6)]
    same_strings = fast.user_content(dev6, CAMS) == plain.user_content(host6, CAMS)
    e2e, e2e_pil = [], []
    for _ in range(args.calls):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fast.user_content(dev6, CAMS)
        e2e.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        plain.user_content(host6, CAMS)
        e2e_pil.append(time.perf_counter() - t0)

    raw = N * H * W * 3
    jpeg_bytes = sum(len(f) for f in files)
    res = {"gpu": None, "power_limit": None, "quality": q, "height": H, "width": W, "unique_frames": U,
           "sample_frames": 6, "sample_ms_per_call": round(ms6, 4), "sample_frames_per_s": round(6 / (ms6 * 1e-3), 1),
           "batch_frames": N, "frames_per_call": args.chunk, "batch_ms": round(msN, 3), "batch_frames_per_s": round(N / (msN * 1e-3), 1),
           "batch_gb_per_s": round((raw + jpeg_bytes) / (msN * 1e-3) / 1e9, 1),
           "batch_share_of_hbm_bandwidth": round((raw + jpeg_bytes) / (msN * 1e-3) / HBM_BYTES_PER_S, 4),
           "mean_file_bytes": int(jpeg_bytes / N), "pillow_threads": threads, "pillow_s": round(pil_s, 3),
           "pillow_frames_per_s": round(N / pil_s, 1), "speedup_vs_pillow_all_cores": round(pil_s * 1e3 / msN, 2),
           "files_differing_from_pillow": int(differ), "e2e_sample_device_ms": round(float(np.median(e2e)) * 1e3, 3),
           "e2e_sample_pillow_one_core_ms": round(float(np.median(e2e_pil)) * 1e3, 3), "e2e_strings_equal": bool(same_strings)}
    res["gpu"], res["power_limit"] = card()
    print(json.dumps(res))
    if differ or not same_strings:
        raise SystemExit("%d files differ from Pillow's; strings equal: %s" % (differ, same_strings))


if __name__ == "__main__":
    main()
