"""Time msc_jpeg_decode_batch (camera JPEGs -> frames, every stage on the device, bit-identical to np.array(Image.open(...))) on
1600 x 900 files, against the per-sample device decoder with host Huffman decode (ops.decode_jpeg_batch) and Pillow, over the same files.

    python tools/bench_jpeg_decode.py [--frames 3552] [--unique 64] [--chunk 592] [--calls 10] [--warmup 2] [--threads 16] [--profile DIR]

Files: --unique seeded frames from tools/bench_jpeg_encode.py's generator, saved by Pillow at quality 90 (4:2:0), the quality
io.write_nuscenes_tree uses.  Real nuScenes camera files are not in this repository, so their sizes and entropy may differ.  The batch
is --frames files (592 samples x 6 cameras), the unique files repeated, staged once into pinned memory and decoded in calls of --chunk
files; each timed call includes its one host-to-device copy of the staged bytes.  Device times are CUDA-event medians over --calls
after --warmup.  ops.decode_jpeg_batch (host Huffman decode on --threads threads) and Pillow (--threads threads) run once over the same
files, host clock.  Every device frame of the batch is compared with Pillow's.  --profile writes a torch.profiler kernel table of one
batch call to DIR.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from io import BytesIO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "multimodal-scene-captioning_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from PIL import Image  # noqa: E402

from bench_jpeg_encode import card, frames  # noqa: E402
from msc_geom import io as mio  # noqa: E402
from msc_geom import ops  # noqa: E402
from msc_geom.engine import GeometryEngine  # noqa: E402


def timed(fn, calls, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(calls):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=3552)
    ap.add_argument("--unique", type=int, default=64)
    ap.add_argument("--chunk", type=int, default=592)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    eng = GeometryEngine(0)
    which = [k % a.unique for k in range(a.frames)]
    groups = [which[i:i + a.chunk] for i in range(0, a.frames, a.chunk)]
    with tempfile.TemporaryDirectory(prefix="bench_jpeg_decode_") as tmp:  # the files are only read while staging
        paths = []
        for k, img in enumerate(frames(a.unique)):
            paths.append(os.path.join(tmp, "f%03d.jpg" % k))
            Image.fromarray(img).save(paths[-1], "JPEG", quality=90)
        datas = [open(p, "rb").read() for p in paths]
        staged = [mio.stage_camera_files([{"cameras": [{"path": paths[k]} for k in g]}]) for g in groups]
        one = mio.stage_camera_files([{"cameras": [{"path": paths[k]} for k in range(6)]}])
    pil = [np.array(Image.open(BytesIO(d))) for d in datas]
    outs = [eng.alloc_jpeg_decode(s) for s in staged]
    comp_bytes = sum(len(datas[k]) for k in which)

    def batch():
        for s, o in zip(staged, outs):
            eng.run_jpeg_decode(s, o)
    t_batch = timed(batch, a.calls, a.warmup)
    equal = 0
    for g, o in zip(groups, outs):
        equal += sum(int(np.array_equal(f, pil[k])) for f, k in zip(o.to_host(), g))
    one_out = eng.alloc_jpeg_decode(one)
    t_one = timed(lambda: eng.run_jpeg_decode(one, one_out), a.calls, a.warmup)
    # the per-sample device decoder (host Huffman decode) and Pillow, over the same files, host clock
    ops.decode_jpeg_batch(eng, datas[:6], threads=a.threads)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for g in groups:
        ops.decode_jpeg_batch(eng, [datas[k] for k in g], threads=a.threads, to_host=False)
    torch.cuda.synchronize()
    t_hostdec = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    with ThreadPoolExecutor(a.threads) as ex:
        list(ex.map(lambda k: np.array(Image.open(BytesIO(datas[k]))), which))
    t_pil = (time.perf_counter() - t0) * 1e3
    name, pl = card()
    res = {"card": name, "power_limit": pl, "frames": a.frames, "chunk": a.chunk, "unique_files": a.unique,
           "compressed_mb_per_frame": comp_bytes / a.frames / 1e6,
           "batch_ms": t_batch, "batch_frames_per_s": a.frames / t_batch * 1e3, "batch_compressed_gb_per_s": comp_bytes / t_batch / 1e6,
           "one_sample_ms": t_one, "decode_jpeg_batch_host_huffman_ms": t_hostdec, "pil_ms": t_pil, "threads": a.threads,
           "frames_equal_to_pil": equal}
    print(json.dumps(res))
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(a.profile, exist_ok=True)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            eng.run_jpeg_decode(staged[0], outs[0])
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=20)
        open(os.path.join(a.profile, "jpeg_decode_kernels.txt"), "w").write(table)
        print(table)


if __name__ == "__main__":
    main()
