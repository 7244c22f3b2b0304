"""Kernel sweep of the fused path on one config-3 batch: every variant is checked bit for bit against the first one listed (config 7,
the previous-generation kernel, itself checked against the oracle by tests/test_gpu_parity.py), then timed with CUDA events.
usage: python tools/sweep_configs.py [config[:split]...]   (env: SWEEP_UNIQUE, SWEEP_REPS, SWEEP_ITERS)"""
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "multimodal-scene-captioning_b200")); sys.path.insert(0, ROOT)
import numpy as np
import torch
from msc_geom.synthetic import make_sample
from msc_geom.layout import pack_batch, tile_batch
from msc_geom.engine import GeometryEngine
from msc_geom import _capi

configs = [tuple(int(v) for v in a.split(":")) for a in sys.argv[1:]] or [(7,), (10,)]
n_unique = int(os.environ.get("SWEEP_UNIQUE", "8")); reps = int(os.environ.get("SWEEP_REPS", "74")); iters = int(os.environ.get("SWEEP_ITERS", "10"))
eng = GeometryEngine()
t0 = time.time()
hb = tile_batch(pack_batch([make_sample(i) for i in range(n_unique)]), reps)
db = eng.upload(hb)
print("batch", hb.n_samples, "samples", hb.n_points, "points, built in %.1f s" % (time.time() - t0), flush=True)
ref = None
rows = []
for cs in configs:
    cfg, split = cs[0], (cs[1] if len(cs) > 1 else 0)
    _capi.set_option("standard", 1)
    if cfg >= 100:  # 102 / 104: stream4.cu with 2 / 4 points per lane; 112: 2 points per lane without the compile-time-constant instantiation
        _capi.set_option("ppt", cfg % 10)
        _capi.set_option("standard", 0 if (cfg // 10) % 10 == 1 else 1)
        cfg = 10
    _capi.set_option("config", cfg)
    _capi.set_option("grid", split)  # (second field of a spec: CTAs of the stream4.cu launch, 0 = auto)
    out = eng.alloc_result(hb)
    try:
        eng.run_fused(db, out)
        torch.cuda.synchronize()
    except Exception as e:  # noqa: BLE001
        print("config", cfg, "FAILED:", e, flush=True)
        continue
    got = out.to_host()
    if ref is None:
        ref = got
        same = "reference"
    else:
        bad = [k for k in ref if not np.array_equal(ref[k][..., :13] if k == "stats" else ref[k], got[k][..., :13] if k == "stats" else got[k], equal_nan=True)]
        same = "IDENTICAL" if not bad else "MISMATCH " + ",".join("%s(%d)" % (k, int((ref[k] != got[k]).sum())) for k in bad)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        eng.run_fused(db, out)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(iters):
        eng.run_fused(db, out)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / iters
    _capi.set_option("time_kernel", 1)
    for _ in range(iters):
        eng.run_fused(db, out)
    torch.cuda.synchronize()
    kt = _capi.kernel_times(iters)
    _capi.set_option("time_kernel", 0)
    row = {"config": cfg, "ppt": _capi.get_option("ppt"), "standard": _capi.get_option("last_standard"), "grid": _capi.get_option("last_grid"), "ms": round(ms, 4), "kernel_ms": round(sum(kt) / len(kt), 4), "samples_per_s": round(hb.n_samples / ms * 1e3), "vs_first": same,
           "window": _capi.get_option("last_window"), "threads": _capi.get_option("threads"), "tile_pts": _capi.get_option("tile_pts")}
    rows.append(row)
    print(json.dumps(row), flush=True)
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "sweep_configs.json"), "w"), indent=1)
