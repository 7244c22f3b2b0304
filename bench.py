#!/usr/bin/env python
"""bench.py -- LiDAR samples/sec of the fused geometric-evidence path (10-sweep, in-box + BEV + proj).

One "step" = one pass of the hot path over one batch of synthetic nuScenes-shaped samples
(BASELINE.json configs[2] shape: 10 sweeps x 34,720 points, 60 boxes, 6 cameras, 200x200 BEV at 0.5 m).
Weak scaling: every rank processes `--samples-per-gpu` samples; `value` is the whole-job aggregate.

    python bench.py [--gpus N --steps K --warmup W]          (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                     (the CPU oracle port on the host cores)
    python bench.py --dump-outputs DIR ...                   (+ the results of the last timed step as DIR/<name>.npy)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "multimodal-scene-captioning_b200"))
sys.path.insert(0, ROOT)

import numpy as np

METRIC = "lidar_samples_per_sec_10sweep_inbox_bev_proj"
UNIT = "samples/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--samples-per-gpu", type=int, default=592, help="batch per rank (4 per SM); inputs ~4.1 GB >> L2")
    ap.add_argument("--unique", type=int, default=37, help="distinct synthetic samples generated per rank, tiled to the batch")
    ap.add_argument("--workload", default="config3", choices=["config3", "config2", "mini", "mini404", "trainval"],
                    help="config3: 10 sweeps, 60 boxes (weak scaling, the metric's config); config2: single keyframes; mini: 10 sweeps, 60-120 "
                         "boxes; mini404: BASELINE config 4, 404 samples sharded over the ranks (strong scaling); trainval: BASELINE config 5, "
                         "34,149 samples sharded over the ranks + a 200-annotation relation table per sample (needs 8 GPUs)")
    ap.add_argument("--total-samples", type=int, default=0, help="override the total of the strong-scaling workloads (testing)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short measurements of BASELINE configs 2, 4 and 5")
    ap.add_argument("--fov", type=int, default=1)
    ap.add_argument("--window", type=int, default=0)
    ap.add_argument("--config", type=int, default=0, help="streaming kernel: 0 = auto, 10 = stream4.cu, 7 = fused_stream.cu")
    ap.add_argument("--grid", type=int, default=0, help="stream4.cu: CTAs of the launch (0 = auto)")
    ap.add_argument("--ppt", type=int, default=0, help="stream4.cu: points per lane, 2 or 4 (0 = the library's default)")
    ap.add_argument("--cull-shift", type=int, default=-1)
    ap.add_argument("--gather", default="fused", choices=["fused", "peer", "nccl"],
                    help="how the small result tables of the shards reach every GPU: fused = written into peer memory by the kernels that produce "
                         "them (no gather step), peer = copy-engine pushes after the step, nccl = one all_gather_into_tensor after the step")
    ap.add_argument("--cpu-samples", type=int, default=0, help="samples in the bounded CPU sample (0 = 4 x cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="GPU arm (--impl b200) only: after the timed steps, write what the last step computed as DIR/<name>.npy (finite "
                         "float32 / float64, at most 64 MB; rank 0's shard when N > 1), so that two builds can be compared output for output "
                         "on the same seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the GPU path (--impl b200)")
    return args


def workload_kwargs(name):
    if name == "config2":
        return dict(n_sweeps=1, n_boxes=60), "config2: 1 keyframe x 34,720 pts, 60 boxes, 6 cams, BEV 200x200"
    if name == "mini":
        return dict(n_sweeps=10, n_boxes="mini"), "config4-shape: 10 sweeps x 34,720 pts, 60-120 boxes, 6 cams, BEV 200x200"
    if name == "mini404":
        return dict(n_sweeps=10, n_boxes="mini"), "config4: 404 samples x 10 sweeps x 34,720 pts, 60-120 boxes, sharded over the ranks"
    if name == "trainval":
        return dict(n_sweeps=10, n_boxes=60), "config5: 34,149 samples x 10 sweeps x 34,720 pts, 60 boxes + 200-annotation relation table, sharded"
    return dict(n_sweeps=10, n_boxes=60), "config3: 10 sweeps x 34,720 pts (347,200), 60 boxes, 6 cams, BEV 200x200 @0.5m"


def algorithmic_bytes(hb, params) -> int:
    """DESIGN.md section 5: bytes the path must move once -- raw rows in, result tables out."""
    G = params.bev_res * params.bev_res
    C = params.n_cams
    n_sweeps = int(hb.sweep_count.shape[0])
    return int(20 * hb.n_points + 96 * n_sweeps + (80 + 20 + 17 * C) * hb.n_boxes + hb.n_samples * (12 * G + 64 + 56 * 2 + C * (56 * 2 + 72)))


class ClockSampler:
    """Polls SM clock and throttle reasons through NVML while the timed regions run."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self._stop, self._t = [], set(), None, threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        if self.nv is not None:
            self._stop.clear()
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        if self._t is not None:
            self._stop.set()
            self._t.join()
            self._t = None

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def cpu_oracle_throughput(hb, params, n_samples: int, threads: int):
    """Time the scalar oracle (tests/oracle_bridge.py -> oracle/libmsc_oracle.so) on the host cores.
    ctypes releases the GIL, so a thread pool uses `threads` cores."""
    from concurrent.futures import ThreadPoolExecutor
    from tests.oracle_bridge import oracle_fused
    idx = [i % hb.n_samples for i in range(n_samples)]
    oracle_fused(hb, 0, params)  # warm-up (page-in, lazy build)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda i: oracle_fused(hb, i, params), idx))
    dt = time.perf_counter() - t0
    return n_samples / dt, dt


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLES = 16  # samples whose BEV grids (and relation tables) are written: ~1 MB each, the whole batch's grids would be far larger


def dump_outputs(path, out, rel=None):
    """Write one step's results as path/<name>.npy: the per-box and per-sample tables of the whole batch, the BEV grids of a fixed
    seeded sample of it (bev_sample_index) and, with `rel` = (relation batch, its device tables), the footprints and pairwise
    relation tables of the same samples.  Tables that would not fit the size limit next to the grids are cut to the sampled samples
    as well (table_sample_index).  Integers are written as float64 (exact for uint32), floats as they are, and every value is finite:
    box_nearest of a box without member points, +inf in the result, is written as -1."""
    import torch
    got = out.to_host()
    keep = np.sort(np.random.default_rng(0).choice(out.n_samples, min(out.n_samples, DUMP_SAMPLES), replace=False))

    def rows_of(off, samples):
        return np.concatenate([np.arange(off[i], off[i + 1]) for i in samples] + [np.zeros(0, np.int64)])

    arrays = {"bev_sample_index": keep}
    arrays.update({k: got[k][keep] for k in ("bev_count", "bev_isum_q", "bev_intensity_sum", "bev_height")})
    if rel is not None:
        rel_db, tabs = rel
        box_off = rel_db.host.sample_box_off.astype(np.int64)
        pair_off = np.concatenate([[0], np.cumsum(np.diff(box_off) ** 2)])  # the n x n tables of the samples, back to back
        rows, pairs = rows_of(box_off, keep), rows_of(pair_off, keep)
        for k, idx in (("rect", rows), ("dist", pairs), ("bearing", pairs), ("category", pairs), ("overlap", pairs)):
            arrays["relation_" + k] = tabs[k][torch.from_numpy(idx).to(tabs[k].device)].cpu().numpy()
    tables = {k: got[k] for k in ("box_count", "box_nearest", "box_centroid", "proj_visible", "proj_extent", "stats")}
    # +inf marks a box without member points (include/msc_geom.h); a distance is never negative, so -1 stands for it without loss
    tables["box_nearest"] = np.where(np.isposinf(tables["box_nearest"]), np.float32(-1), tables["box_nearest"])
    if 8 * sum(a.size for a in list(arrays.values()) + list(tables.values())) > DUMP_LIMIT_BYTES:
        rows = rows_of(got["sample_box_off"].astype(np.int64), keep)
        tables = {k: v[keep] if k == "stats" else v[rows] for k, v in tables.items()}
        arrays["table_sample_index"] = keep
    arrays.update(tables)
    arrays = {k: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64) for k, a in arrays.items()}
    bad = [k for k, a in arrays.items() if not np.isfinite(a).all()]
    if bad:  # the path writes no other NaN / inf: one here is a defect, and a dump must not hide it
        raise ValueError("--dump-outputs: non-finite values in " + ", ".join(bad))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    from msc_geom.dist import shard_range
    from msc_geom.layout import GeomParams, pack_batch, tile_batch, truncate_batch
    from msc_geom.synthetic import make_sample

    params = GeomParams()
    wkw, wname = workload_kwargs(args.workload)
    cores = os.cpu_count() or 1

    # ---------------------------------------------------------------- reference arm: CPU oracle port, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return 0
        n_unique = min(args.unique, 8)
        hb = pack_batch([make_sample(i, **wkw) for i in range(n_unique)])
        per_step = args.cpu_samples or 4 * cores
        for _ in range(max(args.warmup, 1) if args.warmup else 0):
            cpu_oracle_throughput(hb, params, max(cores, 2), cores)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_oracle_throughput(hb, params, per_step, cores)
        dt = time.perf_counter() - t0
        val = args.steps * per_step / dt
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
                "config": {"workload": wname, "samples_per_step": per_step},
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": f"{per_step} samples per step x {args.steps} steps, scalar C oracle, {cores} threads"},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- B200 arm
    import torch
    import torch.distributed as dist
    from msc_geom import _capi
    from msc_geom.dist import FusedTableGather, make_table_gather, bind_to_gpu_numa
    from msc_geom.engine import GeometryEngine

    numa = bind_to_gpu_numa(local_rank)  # before any pinned allocation: staging buffers and copy threads stay on the GPU's socket
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = GeometryEngine(local_rank, params)
    _capi.set_option("fov", args.fov)
    _capi.set_option("window", args.window)
    _capi.set_option("config", args.config)
    _capi.set_option("cull_shift", args.cull_shift)
    _capi.set_option("grid", args.grid)
    if args.ppt:
        _capi.set_option("ppt", args.ppt)
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def run_device_resident(workload: str, steps: int, warmup: int, samples_per_gpu: int, total_override: int = 0, sampler=None, dump=None):
        """`steps` timed passes of the hot path over one HBM-resident batch of `workload`, sharded over the ranks; tables gathered with
        one overlapped collective per step; `dump`: directory for the results of the last step (rank 0).  Returns the measurement and
        the pieces the caller reuses (distinct-sample batch, engine state)."""
        wkw_, wname_ = workload_kwargs(workload)
        strong = {"mini404": 404, "trainval": 34149}.get(workload, 0)
        if strong:
            strong = total_override or strong
            lo, hi = shard_range(strong, rank, world)
            S = hi - lo
        else:
            S = samples_per_gpu
        n_unique = max(1, min(args.unique, S))
        reps = (S + n_unique - 1) // n_unique
        base = rank * 100000
        hb_u = pack_batch([make_sample(base + i, **wkw_) for i in range(n_unique)])
        db = eng.upload_tiled(hb_u, reps, S)  # one host copy of the distinct samples, replicated on the device
        hb = db.host
        S = hb.n_samples
        rel_db = rel = None
        if workload == "trainval":  # + pairwise relation table over 200 annotations per sample (BASELINE config 5)
            ann_u = [{"point_cloud": np.zeros((0, 4), np.float32), "annotations": make_sample(base + 50000 + i, n_sweeps=1, n_boxes=200)["annotations"]}
                     for i in range(n_unique)]
            rel_db = eng.upload_tiled(pack_batch(ann_u), reps, S)
            rel, _ = eng.alloc_relations(rel_db.host)
        _, arena_bytes = eng.table_layout(S, hb.n_boxes, params.n_cams)
        arena_bytes = int(max_over_ranks(float(arena_bytes)))  # ragged shards: every rank gathers the size of the largest
        # only the small tables cross GPUs (BEV grids stay sharded).  Default: the kernels that produce a table entry store it into every
        # GPU's gathered buffer themselves (P2P stores into peer-mapped memory); alternatives for comparison: copy-engine pushes, NCCL
        gat, gat_how, reps_c = None, "none (1 GPU)", [None, None]
        if world > 1 and args.gather == "fused":
            try:
                gat = FusedTableGather(arena_bytes, eng.device)
                outs = [gat.result(eng, hb, k) for k in range(2)]
                reps_c = [gat.replicas(eng, hb, k) for k in range(2)]
                gat_how = "fused into the producing kernels: P2P stores into every GPU's gathered tables (symmetric memory), no gather step"
            except Exception as e:  # noqa: BLE001 -- no symmetric memory on this platform / build
                gat, gat_how = None, "symmetric memory unavailable (%s)" % type(e).__name__
        if world > 1 and gat is None:
            outs = [eng.alloc_result(hb, arena_bytes=arena_bytes) for _ in range(2)]
            gat, how2 = make_table_gather(arena_bytes, eng.device, prefer_peer=args.gather != "nccl")
            gat_how = how2 if gat_how.startswith("none") else how2 + "; " + gat_how
        if world == 1:
            outs = [eng.alloc_result(hb, arena_bytes=arena_bytes)]

        def step(k):
            out = outs[k % len(outs)]
            if gat is not None and gat.done[k % 2] is not None:
                stream.wait_event(gat.done[k % 2])  # the gather that read this arena two steps ago is done
            eng.run_fused(db, out, replicas=reps_c[k % 2])
            if gat is not None:
                gat.launch(out.table_arena)

        for k in range(max(warmup, 3)):
            step(k)
        if gat is not None:
            gat.wait()
        barrier()
        _capi.set_option("time_kernel", 1)  # CUDA events around the streaming kernel alone, recorded by the library on this stream
        launches0 = eng.kernel_launches
        call_events, rel_events = [], []
        if sampler is not None:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        host_t0 = time.perf_counter()
        for k in range(steps):
            ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ka.record(stream)
            step(k)
            kb.record(stream)
            call_events.append((ka, kb))
            if rel_db is not None:
                kc = torch.cuda.Event(enable_timing=True)
                eng.run_relations(rel_db, rel)
                kc.record(stream)
                rel_events.append((kb, kc))
        host_enqueue_ms = (time.perf_counter() - host_t0) * 1e3 / steps  # host time to queue one step (no synchronisation inside the loop)
        if gat is not None:
            gat.wait()
        e1.record(stream)
        barrier()
        if sampler is not None:
            sampler.stop()
        elapsed_ms = max_over_ranks(e0.elapsed_time(e1))
        call_ms = sum(a.elapsed_time(b) for a, b in call_events) / len(call_events)
        own = _capi.kernel_times(min(steps, 64))
        _capi.set_option("time_kernel", 0)
        kernel_ms_here = (sum(own) / len(own)) if own else call_ms
        per_rank_kernel_ms = [kernel_ms_here]
        if world > 1:  # ranks stream different synthetic samples: the step ends with the slowest one
            t = torch.tensor([kernel_ms_here], device="cuda", dtype=torch.float64)
            allr = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allr, t)
            per_rank_kernel_ms = [round(float(x.item()), 4) for x in allr]
        total = strong if strong else world * S
        m = {"workload": wname_, "scaling": "strong" if strong else "weak", "total_samples": total, "samples_this_rank": S,
             "value": total * steps / (elapsed_ms * 1e-3), "unit": UNIT, "ms_per_step": elapsed_ms / steps, "steps": steps,
             "call_ms": call_ms, "kernel_ms": (sum(own) / len(own)) if own else call_ms, "host_enqueue_ms": host_enqueue_ms, "per_rank_kernel_ms": per_rank_kernel_ms, "gpu_launches": eng.kernel_launches - launches0,
             "kernel_config": _capi.get_option("last_config"), "table_gather": gat_how + (" (one per step, double-buffered)" if world > 1 else ""),
             "grid": _capi.get_option("last_grid"), "bev_window_cells": _capi.get_option("last_window"),
             "tile_pts": _capi.get_option("tile_pts"), "threads": _capi.get_option("threads"), "table_arena_bytes": arena_bytes,
             "points_per_step_this_rank": hb.n_points, "algorithmic_bytes": algorithmic_bytes(hb, params), "n_unique": n_unique, "reps": reps}
        if rel_events:
            m["relation_table_ms"] = sum(a.elapsed_time(b) for a, b in rel_events) / len(rel_events)
            m["relation_table_bytes"] = int(hb.n_samples * (40 * 200 + 10 * 200 * 200))
        if dump and rank == 0:
            dump_outputs(dump, outs[(steps - 1) % len(outs)], (rel_db, rel) if rel_db is not None else None)
        return m, hb_u, reps

    # ---------------------------------------------------------------- the metric: BASELINE config 3, weak scaling, inputs resident in HBM
    sampler = ClockSampler(local_rank)
    main, hb_u, reps = run_device_resident(args.workload, args.steps, args.warmup, args.samples_per_gpu, args.total_samples, sampler,
                                           args.dump_outputs)
    strong_total = main["total_samples"] if main["scaling"] == "strong" else 0

    # ---------------------------------------------------------------- end to end: pinned host buffers in, host tables + BEV out
    e2e = None
    if not args.no_e2e and not strong_total:
        # one chunk = one copy of the distinct-sample set (loader-format flat buffers) in a pinned input arena: ONE H2D copy per chunk
        # into a preallocated device arena, the fused call, then three D2H copies (table arena, two BEV layers); three slots / streams so
        # H2D, kernel and D2H of neighbouring chunks overlap.  Nothing is allocated inside the timed region.
        n_slots = 3
        arenas = [eng.input_arena(hb_u) for _ in range(n_slots)]
        for a in arenas:
            a.load(hb_u)
        streams = [torch.cuda.Stream() for _ in range(n_slots)]
        outs = [eng.alloc_result(hb_u) for _ in range(n_slots)]
        host_out = [[torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in (o.table_arena, o.bev_ci, o.bev_height)] for o in outs]
        h2d = arenas[0].nbytes * reps
        d2h = sum(int(t.numel() * t.element_size()) for t in host_out[0]) * reps

        def e2e_step():
            for ci in range(reps):
                slot = ci % n_slots
                with torch.cuda.stream(streams[slot]):
                    dbc = arenas[slot].upload(non_blocking=True)
                    eng.run_fused(dbc, outs[slot])
                    for src, dst in zip((outs[slot].table_arena, outs[slot].bev_ci, outs[slot].bev_height), host_out[slot]):
                        dst.copy_(src, non_blocking=True)
            for s in streams:
                s.synchronize()

        e2e_step()
        barrier()
        sampler.start()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        dt_rank = time.perf_counter() - t0
        barrier()
        sampler.stop()
        dt = max_over_ranks(dt_rank)
        n_e2e = reps * hb_u.n_samples
        rates = [h2d * args.e2e_steps / dt_rank / 1e9]
        if world > 1:
            t = torch.tensor(rates, device="cuda", dtype=torch.float64)
            allr = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allr, t)
            rates = [float(x.item()) for x in allr]
        e2e = {"value": world * n_e2e * args.e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "h2d_copies_per_chunk": 1, "d2h_copies_per_chunk": 3, "chunks_per_step": reps, "per_rank_h2d_gbs": [round(r, 2) for r in rates],
               "numa": numa}

    # ---------------------------------------------------------------- the other BASELINE configs, one short measurement each
    extras = []
    if not args.no_extra and args.workload == "config3":
        try:
            m, _, _ = run_device_resident("mini404", 20, 3, 0)   # config 4: 404 samples, 60-120 boxes, strong scaling over the ranks
            extras.append(m)
            if world == 1:
                m, _, _ = run_device_resident("config2", 20, 3, 1)    # config 2 as written: ONE keyframe on one GPU (latency; the sample is split over CTAs)
                m["latency_us_per_call"] = 1e3 * m["call_ms"]
                extras.append(m)
                m, _, _ = run_device_resident("config2", 20, 3, 592)  # ... and a batch of keyframes (throughput)
                extras.append(m)
            if world == 8:
                m, _, _ = run_device_resident("trainval", 5, 3, 0)   # config 5: 34,149 samples + 200-annotation relation tables, 8 GPUs
                extras.append(m)
        except Exception as e:  # noqa: BLE001 -- an extra must not take the headline down with it
            extras.append({"error": repr(e)})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---------------------------------------------------------------- roofline + CPU baseline (rank 0)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    kavg_ms, abytes = main["kernel_ms"], main["algorithmic_bytes"]
    achieved = abytes / (kavg_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "fused_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    kname = "stream4_kernel" if main["kernel_config"] == 10 else "stream_evidence_kernel"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": "profiles/fused_traffic.json (one ncu --set full capture of the same launch shape, not this run)",
                "kernel": kname, "kernel_ms": kavg_ms, "call_ms": main["call_ms"], "host_enqueue_ms": main["host_enqueue_ms"], "per_rank_kernel_ms": main["per_rank_kernel_ms"], "algorithmic_bytes_per_launch": abytes, "peak_source": peak_src}
    cpu = None
    if not args.no_cpu and world == 1:
        n_cpu = args.cpu_samples or 16 * cores  # ~2 s wall on 16 threads = ~30 s of CPU work on the bounded sample
        v, dt = cpu_oracle_throughput(hb_u, params, n_cpu, cores)
        v1, _ = cpu_oracle_throughput(hb_u, params, 8, 1)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "value_1_thread": v1,
               "sample": f"{n_cpu} samples of the same workload, scalar C oracle (oracle/c/msc_oracle.c), {cores} threads, {dt:.1f} s wall"}
        ref_py = os.path.join(ROOT, "profiles", "r2_cpu_baseline_reference_python.json")
        if os.path.exists(ref_py):  # the reference's own Python functions, timed where /root/reference exists (tools/cpu_baseline_reference.py)
            try:
                cpu["reference_python"] = json.load(open(ref_py))
            except Exception:
                pass
    line = {"metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": main["scaling"], "vs_baseline": None,
            "dtype": "f32+f64", "data": f"synthetic ({main['n_unique']} distinct seeded samples per rank tiled x{main['reps']}, distinct memory)",
            "config": {"workload": main["workload"], "samples_per_gpu": main["samples_this_rank"], "total_samples": main["total_samples"],
                       "points_per_step_per_gpu": main["points_per_step_this_rank"],
                       "l2_policy": "inputs (%.2f GB of raw rows per step) larger than L2; no explicit flush" % (main["points_per_step_this_rank"] * 20 / 1e9),
                       "fov_counts": bool(args.fov), "bev_window_cells": main["bev_window_cells"], "tile_pts": main["tile_pts"],
                       "threads": main["threads"], "kernel_config": main["kernel_config"], "grid": main["grid"],
                       "table_gather": main["table_gather"],
                       "table_arena_bytes": main["table_arena_bytes"]},
            "e2e": e2e, "gpu_launches": main["gpu_launches"], "clocks": sampler.summary(), "roofline": roofline, "cpu_baseline": cpu,
            "extra_workloads": extras}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
