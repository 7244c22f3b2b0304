"""bench.py --impl reference runs on CPU and prints one JSON line with the contract's keys; --dump-outputs writes what the timed
path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TABLES = ("box_count", "box_nearest", "box_centroid", "proj_visible", "proj_extent", "stats")
BEV = ("bev_count", "bev_isum_q", "bev_intensity_sum", "bev_height")


def _load_dir(path):
    return {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path)) if f.endswith(".npy")}


def _box_rows(off, samples):
    return np.concatenate([np.arange(off[i], off[i + 1]) for i in samples])


def _dumped(k, a):
    """What --dump-outputs writes for result array `a`: +inf in box_nearest (a box without member points) as -1."""
    return np.where(np.isposinf(a), np.float32(-1), a) if k == "box_nearest" else a


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-samples", "2", "--unique", "2", "--workload", "config2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun (N > 1) rank 0 alone runs and prints the reference arm; every other rank exits 0 without work or output."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29999")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip() == ""


def _fake_result(S, R, n_cams, seed):
    """A BatchResult on host tensors with random contents, shaped like one step of the fused path; every third box has no member
    point (count 0, nearest +inf, centroid 0)."""
    import torch
    from msc_geom.engine import BatchResult
    rng = np.random.default_rng(seed)
    off = np.concatenate([[0], np.cumsum(rng.integers(0, 5, S))]).astype(np.int32)
    B = int(off[-1])
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    count, nearest, centroid = rng.integers(1, 1 << 31, B, dtype=np.int32), rng.random(B, dtype=np.float32), rng.random((B, 3), dtype=np.float32)
    count[::3], nearest[::3], centroid[::3] = 0, np.inf, 0
    return BatchResult(S, n_cams, R, 8, off, t(count), t(nearest), t(centroid), t(rng.integers(0, 2, (B, n_cams), dtype=np.uint8)),
                       t(rng.random((B, n_cams, 4), dtype=np.float32)), t(rng.integers(0, 1 << 31, (S, R, R, 2), dtype=np.int32)),
                       t(rng.random((S, R, R), dtype=np.float32)), t(rng.integers(0, 1 << 31, (S, 16), dtype=np.int32)))


def test_dump_outputs_writes_exact_float_arrays_within_the_limit(tmp_path, monkeypatch):
    import bench
    out = _fake_result(40, 8, 6, 0)
    host = out.to_host()
    bench.dump_outputs(str(tmp_path / "a"), out)
    bench.dump_outputs(str(tmp_path / "b"), out)
    a, b = _load_dir(str(tmp_path / "a")), _load_dir(str(tmp_path / "b"))
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)                 # the sample of the BEV grids is fixed
    assert set(a) == {"bev_sample_index", *BEV, *TABLES}
    assert all(v.dtype in (np.float32, np.float64) and np.isfinite(v).all() for v in a.values())
    assert np.isinf(host["box_nearest"]).any() and np.array_equal(a["box_nearest"] == -1, host["box_count"] == 0)
    keep = a["bev_sample_index"].astype(np.int64)
    assert len(keep) == bench.DUMP_SAMPLES and np.array_equal(keep, np.unique(keep)) and keep.max() < 40
    for k in TABLES:                                                                        # uint32 values survive float64 exactly
        assert np.array_equal(a[k], _dumped(k, host[k])), k
    for k in BEV:
        assert np.array_equal(a[k], host[k][keep]), k

    # with relation tables (footprint rows per box, n x n pair tables per sample): those of the same samples
    import torch
    from types import SimpleNamespace
    rng = np.random.default_rng(1)
    roff = np.concatenate([[0], np.cumsum(rng.integers(0, 4, 40))])
    poff = np.concatenate([[0], np.cumsum(np.diff(roff) ** 2)])
    tabs = {"rect": torch.rand(int(roff[-1]), 6, dtype=torch.float64), "dist": torch.rand(int(poff[-1])), "bearing": torch.rand(int(poff[-1])),
            "category": torch.randint(0, 4, (int(poff[-1]),), dtype=torch.uint8), "overlap": torch.randint(0, 2, (int(poff[-1]),), dtype=torch.uint8)}
    bench.dump_outputs(str(tmp_path / "r"), out, (SimpleNamespace(host=SimpleNamespace(sample_box_off=roff)), tabs))
    r = _load_dir(str(tmp_path / "r"))
    assert np.array_equal(r["relation_rect"], tabs["rect"].numpy()[_box_rows(roff, keep)])
    for k in ("dist", "bearing", "category", "overlap"):
        assert np.array_equal(r["relation_" + k], tabs[k].numpy()[_box_rows(poff, keep)]), k

    # a limit that holds the grids and the tables of the sampled samples, but not the whole tables: those are cut to the same samples
    rows = _box_rows(host["sample_box_off"], keep)
    cut = {**{k: _dumped(k, host[k][rows]) for k in TABLES[:-1]}, "stats": host["stats"][keep]}
    limit = 8 * (sum(a[k].size for k in BEV) + 2 * len(keep) + sum(v.size for v in cut.values()))
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", limit)
    bench.dump_outputs(str(tmp_path / "c"), out)
    c = _load_dir(str(tmp_path / "c"))
    assert set(c) == set(a) | {"table_sample_index"} and np.array_equal(c["table_sample_index"], keep)
    for k in TABLES:
        assert np.array_equal(c[k], cut[k]), k
    assert sum(v.nbytes for v in c.values()) <= limit

    # any other NaN / inf is a defect of the path: refused, nothing written
    out.box_centroid[1, 0] = float("nan")
    with pytest.raises(ValueError, match="box_centroid"):
        bench.dump_outputs(str(tmp_path / "d"), out)
    assert not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_bench_dump_outputs_equal_the_oracle(tmp_path):
    """The tables and BEV grids bench.py writes after its timed steps are those of the CPU oracle on the same seeded samples, whatever
    the number of steps; the launches of the timed region grow with --steps."""
    from msc_geom.layout import GeomParams, pack_batch
    from msc_geom.synthetic import make_sample
    from tests.oracle_bridge import oracle_fused
    n_unique, S = 3, 7
    lines, dumps = {}, {}
    for steps in (2, 5):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0", "--samples-per-gpu", str(S),
                              "--unique", str(n_unique), "--no-e2e", "--no-cpu", "--no-extra", "--dump-outputs", str(tmp_path / str(steps))],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines[steps] = json.loads(out.stdout.strip().splitlines()[-1])
        dumps[steps] = _load_dir(str(tmp_path / str(steps)))
    assert lines[2]["gpu_launches"] > 0 and 2 * lines[5]["gpu_launches"] == 5 * lines[2]["gpu_launches"]   # counted inside the timed loop
    assert set(dumps[2]) == set(dumps[5]) and all(np.array_equal(dumps[2][k], dumps[5][k]) for k in dumps[2])
    d = dumps[5]
    assert sum(v.nbytes for v in d.values()) <= 64 << 20 and "table_sample_index" not in d
    assert all(np.isfinite(v).all() for v in d.values())
    assert np.array_equal(d["bev_sample_index"], np.arange(S))                              # fewer samples than the sample size: all of them
    hb = pack_batch([make_sample(i, n_sweeps=10, n_boxes=60) for i in range(n_unique)])   # the batch is these samples, tiled
    params = GeomParams()
    b = 0
    for i in range(S):
        ref = oracle_fused(hb, i % n_unique, params)
        nb = len(ref["box_count"])
        for k in TABLES[:-1]:
            assert np.array_equal(d[k][b:b + nb], _dumped(k, ref[k]).astype(d[k].dtype)), (i, k)
        for k in ("bev_count", "bev_isum_q", "bev_height"):
            assert np.array_equal(d[k][i], ref[k].astype(d[k].dtype)), (i, k)
        assert np.array_equal(d["stats"][i][:13], ref["stats"][:13].astype(np.float64)), i
        b += nb
    assert b == len(d["box_count"])
