"""PNG files of the LiDAR agent's images encoded on the device (msc_png_encode_batch / GeometryEngine.run_png_encode /
ops.encode_png_batch) and the classifier mosaics drawn there (msc_cluster_mosaics / GeometryEngine.run_cluster_mosaics).  A file must
have Pillow's IHDR and an IDAT that inflates to exactly Pillow's payload (its filter choice, restated below); its deflate stream is the
encoder's own, within size bars against Pillow's files."""
import base64
import ctypes as C
import io
import json
import os
import struct
import zlib

import numpy as np
import pytest
from PIL import Image

from msc_geom import _capi
from msc_geom.lidar_agent import cluster_mosaic, mosaic_stamp

GOLDEN_KEYFRAMES = ("mock", "edge", "synth", "empty", "flatobj")


def chunks(data: bytes):
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    i, out = 8, []
    while i < len(data):
        n, = struct.unpack(">I", data[i:i + 4])
        out.append((data[i + 4:i + 8], data[i + 8:i + 8 + n], struct.unpack(">I", data[i + 8 + n:i + 12 + n])[0]))
        i += 12 + n
    assert i == len(data)
    return out


def pillow_png(img: np.ndarray) -> bytes:
    buf = io.BytesIO()
    Image.fromarray(img).save(buf, "PNG")
    return buf.getvalue()


def inflated_idat(data: bytes) -> bytes:
    return zlib.decompress(b"".join(d for t, d, _ in chunks(data) if t == b"IDAT"))


def filtered_rows(img: np.ndarray) -> bytes:
    """Pillow's IDAT payload (ZipEncode.c), restated: per row a filter byte and the filtered row; None, Up, Sub, Paeth tried in that order,
    cost sum(v < 128 ? v : 256 - v), a candidate taken only when strictly cheaper, the search stopped at cost 0, Average never."""
    h = img.shape[0]
    bpp = 1 if img.ndim == 2 else img.shape[2]
    x = img.reshape(h, -1).astype(np.int32)
    prev, out = np.zeros(x.shape[1], np.int32), []
    z = np.zeros(bpp, np.int32)
    for y in range(h):
        r = x[y]
        a, b, c = np.concatenate([z, r[:-bpp]]), prev, np.concatenate([z, prev[:-bpp]])
        p = a + b - c
        pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
        paeth = np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))
        best = cost = None
        for ftype, f in ((0, r), (2, r - b), (1, r - a), (4, r - paeth)):
            v = f & 255
            s = int(np.where(v < 128, v, 256 - v).sum())
            if cost is None or s < cost:
                best, cost, bv = ftype, s, v
            if cost == 0:
                break
        out.append(bytes([best]) + bv.astype(np.uint8).tobytes())
        prev = r
    return b"".join(out)


def stored_bound(h, w, c):
    raw = h * (1 + w * c)
    return 57 + 6 + raw + 5 * -(-raw // 65535)


def _random_images():
    rng = np.random.default_rng(7)
    grad = (np.add.outer(np.arange(64), np.arange(80))[..., None] * [1, 2, 3] % 256).astype(np.uint8)
    sparse = np.zeros((120, 90, 3), np.uint8)
    sparse[::7, ::5] = (80, 80, 120)
    noisy = np.full((50, 70, 3), 255, np.uint8)
    m = rng.random((50, 70)) < 0.1
    noisy[m] = rng.integers(0, 256, (int(m.sum()), 3))
    return {"rgb_37x53": rng.integers(0, 256, (37, 53, 3), np.uint8), "grey_40x41": rng.integers(0, 256, (40, 41), np.uint8), "gradient": grad,
            "grey_gradient": grad[..., 1].copy(), "sparse": sparse, "white": np.full((30, 30, 3), 255, np.uint8), "noise_on_white": noisy,
            "flat_grey": np.full((9, 700), 17, np.uint8)}


def _golden_corpus(golden_dir):
    """The agent-image goldens: BEVs (semantic as RGB, density), cluster views and the reference mosaic, as Pillow sees them."""
    out = {}
    for name in GOLDEN_KEYFRAMES:
        g = np.load(os.path.join(golden_dir, f"keyframe_{name}.npz"))
        out[f"bev_{name}"] = np.ascontiguousarray(g["semantic"][..., ::-1])
        out[f"density_{name}"] = g["density"]
    v = np.load(os.path.join(golden_dir, "cluster_views.npz"))
    for k in range(int(v["n"])):
        out[f"view_{k}"] = np.ascontiguousarray(v[f"img_{k}"][..., ::-1])
    out["mosaic"] = np.ascontiguousarray(v["mosaic"][..., ::-1])
    return out


# ---------------------------------------------------------------------------------------------------------------------------- CPU
def test_filter_restatement_equals_pillow(golden_dir):
    imgs = dict(_random_images())
    imgs.update(_golden_corpus(golden_dir))
    for name, img in imgs.items():
        data = pillow_png(img)
        assert [t for t, _, _ in chunks(data)][0] == b"IHDR", name
        assert inflated_idat(data) == filtered_rows(img), name


@pytest.mark.parametrize("count", range(1, 11))
def test_views_plus_mosaic_stamp_equal_cluster_mosaic(count):
    rng = np.random.default_rng(count)
    views = [rng.integers(0, 256, (512, 512, 3), np.uint8) for _ in range(count)]
    want = cluster_mosaic(views)
    if count == 1:
        assert want is views[0]
        return
    rows, cols = (count + 2) // 3, min(3, count)
    got = np.zeros((rows * 512, cols * 512, 3), np.uint8)
    for i, v in enumerate(views):
        r, c = divmod(i, cols)
        got[r * 512:(r + 1) * 512, c * 512:(c + 1) * 512] = v
    st = mosaic_stamp(count)
    flat = got.reshape(-1, 3)
    px, col = st[:, 0].astype(np.int64), st[:, 1]
    flat[px] = np.stack([col & 255, (col >> 8) & 255, (col >> 16) & 255], 1).astype(np.uint8)
    assert np.array_equal(got, want)
    empty = rows * cols - count
    assert len(st) >= empty * 512 * 512


def test_argument_refusals_without_a_device():
    """Bad arguments are refused with MSC_ERR_BAD_ARGUMENT before anything is launched (without a device a launch fails otherwise)."""
    lib = _capi.load()
    p = 1 << 20  # a 256-byte aligned address that is never dereferenced

    def descs(*imgs):
        a = (_capi.MscPngImage * len(imgs))()
        for i, (h, w, c, sw, pitch, px) in enumerate(imgs):
            a[i] = _capi.MscPngImage(px, pitch, h, w, c, sw)
        return a

    good = (20, 30, 3, 0, 90, p)
    need = int(lib.msc_png_encode_workspace_bytes(2, descs(good, (5, 7, 1, 0, 7, p))))
    assert need >= 20 * 91 * 5
    bad = [(20, 30, 2, 0, 90, p), (20, 30, 4, 0, 120, p), (20, 30, 1, 1, 90, p), (0, 30, 3, 0, 90, p), (20, 0, 3, 0, 90, p),
           (65536, 30, 3, 0, 90, p), (20, 65536, 3, 0, 196608, p), (20, 30, 3, 0, 89, p), (20, 30, 3, 0, 90, None),
           (65535, 65535, 1, 0, 65535, p)]  # raw >= 2^31
    for b in bad:
        d = descs(good, b)
        assert lib.msc_png_encode_workspace_bytes(2, d) == 0, b
        assert lib.msc_png_encode_batch(2, d, p, 1 << 20, p, p, p, 1 << 40, None) == _capi.MSC_ERR_BAD_ARGUMENT, b
    assert lib.msc_png_encode_workspace_bytes(-1, descs(good)) == 0
    d = descs(good)
    one = int(lib.msc_png_encode_workspace_bytes(1, d))
    for args in ((None, p, p, p), (p, None, p, p), (p, p, None, p), (p, p, p, None)):
        out, off, st, ws = args
        assert lib.msc_png_encode_batch(1, d, out, 1 << 20, off, st, ws, one, None) == _capi.MSC_ERR_BAD_ARGUMENT, args
    assert lib.msc_png_encode_batch(1, None, p, 1 << 20, p, p, p, one, None) == _capi.MSC_ERR_BAD_ARGUMENT
    assert lib.msc_png_encode_batch(1, d, p, 1 << 20, p, p, p, one - 1, None) == _capi.MSC_ERR_BAD_ARGUMENT
    assert lib.msc_png_encode_batch(1, d, p, 1 << 20, p, p, p + 16, one, None) == _capi.MSC_ERR_BAD_ARGUMENT
    assert lib.msc_png_encode_batch(-1, d, p, 1 << 20, p, p, p, one, None) == _capi.MSC_ERR_BAD_ARGUMENT
    assert lib.msc_png_encode_batch(0, None, None, 0, None, None, None, 0, None) == 0

    # mosaics: counts outside 1..10, a group past the views, NULL buffers, a short workspace
    mneed = int(lib.msc_cluster_mosaics_workspace_bytes(2))
    assert mneed >= 256 and lib.msc_cluster_mosaics_workspace_bytes(-1) == 0
    off = np.zeros(12, np.int32)

    def mosaics(groups, n_views=12, views=p, out=p, ws=p, ws_bytes=mneed):
        g = np.ascontiguousarray(np.array(groups, np.int32).reshape(-1, 2))
        return lib.msc_cluster_mosaics(views, n_views, g.ctypes.data, len(g), p, off.ctypes.data, out, ws, ws_bytes, None)

    for kw in ({"groups": ((0, 0), (0, 1))}, {"groups": ((0, 11), (0, 1))}, {"groups": ((5, 8), (0, 1))}, {"groups": ((-1, 2), (0, 1))},
               {"groups": ((0, 2), (0, 1)), "views": None}, {"groups": ((0, 2), (0, 1)), "out": None}, {"groups": ((0, 2), (0, 1)), "ws": None},
               {"groups": ((0, 2), (0, 1)), "ws_bytes": mneed - 1}):
        assert mosaics(**kw) == _capi.MSC_ERR_BAD_ARGUMENT, kw
    assert lib.msc_cluster_mosaics(None, 0, None, 0, None, None, None, None, 0, None) == 0


# ---------------------------------------------------------------------------------------------------------------------------- GPU
def check_file(data: bytes, img: np.ndarray, what=""):
    """Every property of a device file: chunk sequence, CRCs, Pillow's IHDR, Pillow's inflated payload, the pixels, the stored bound."""
    cs = chunks(data)
    types = [t for t, _, _ in cs]
    assert types[0] == b"IHDR" and types[-1] == b"IEND" and set(types[1:-1]) == {b"IDAT"}, (what, types)
    for t, d, crc in cs:
        assert zlib.crc32(t + d) == crc, (what, t)
    ref = pillow_png(img)
    assert cs[0][1] == chunks(ref)[0][1], what
    z = b"".join(d for t, d, _ in cs if t == b"IDAT")
    assert z[:2] == b"\x78\x9c", what
    assert zlib.decompress(z) == inflated_idat(ref), what
    assert np.array_equal(np.array(Image.open(io.BytesIO(data))), img), what
    h, w = img.shape[:2]
    assert len(data) <= stored_bound(h, w, 1 if img.ndim == 2 else 3), (what, len(data))


def _edge_images():
    rng = np.random.default_rng(11)
    return {"1x1": rng.integers(0, 256, (1, 1, 3), np.uint8), "1x40000": rng.integers(0, 256, (1, 40000, 3), np.uint8),
            "40000x1": rng.integers(0, 256, (40000, 1), np.uint8), "3x3": rng.integers(0, 256, (3, 3, 3), np.uint8),
            "1x40000_smooth": np.repeat((np.arange(40000) // 300 % 256).astype(np.uint8)[None, :, None], 3, 2),
            "constant": np.full((300, 500, 3), 93, np.uint8), "noise": rng.integers(0, 256, (300, 400, 3), np.uint8),
            "wide_stride": np.tile((np.arange(11000) % 7 * 30).astype(np.uint8)[None, :, None], (40, 1, 3)),
            "grey_noise": rng.integers(0, 256, (257, 300), np.uint8)}


@pytest.mark.gpu
def test_device_files_on_shapes_and_edges(engine, golden_dir):
    from msc_geom import ops
    imgs = dict(_random_images())
    imgs.update(_edge_images())
    imgs.update(_golden_corpus(golden_dir))
    names = list(imgs)
    files = ops.encode_png_batch(engine, [imgs[k] for k in names])
    for k, f in zip(names, files):
        check_file(f, imgs[k], k)
    noise = files[names.index("noise")]
    assert len(noise) == stored_bound(300, 400, 3)  # incompressible: stored blocks


@pytest.mark.gpu
def test_strided_rows_and_swap_rb(engine):
    import torch
    rng = np.random.default_rng(5)
    big = rng.integers(0, 256, (60, 90, 3), np.uint8)
    big[:, 40:] = big[:, 40:41]
    dev = torch.from_numpy(big).to(engine.device)
    sub = dev[5:50, 7:70]  # strided rows
    bgr = dev[:, :, :]
    grey = torch.from_numpy(np.ascontiguousarray(big[..., 1])).to(engine.device)
    imgs = [sub, bgr, grey[3:40, 10:30]]
    out = engine.alloc_png(imgs, out_bytes=stored_bound(45, 63, 3) + stored_bound(60, 90, 3) + stored_bound(37, 20, 1))  # noise: stored
    res = engine.run_png_encode(imgs, swap_rb=[False, True, False], out=out).to_host()
    check_file(res[0], np.ascontiguousarray(big[5:50, 7:70]), "strided")
    check_file(res[1], np.ascontiguousarray(big[..., ::-1]), "swap_rb")
    check_file(res[2], np.ascontiguousarray(big[3:40, 10:30, 1]), "strided grey")


@pytest.mark.gpu
def test_determinism_alone_and_in_a_batch(engine, golden_dir):
    from msc_geom import ops
    corpus = _golden_corpus(golden_dir)
    imgs = [corpus["bev_mock"], _edge_images()["noise"], corpus["view_3"], _random_images()["grey_40x41"], corpus["mosaic"]]
    batch = ops.encode_png_batch(engine, imgs)
    assert ops.encode_png_batch(engine, imgs) == batch
    for img, f in zip(imgs, batch):
        assert ops.encode_png_batch(engine, [img]) == [f]
    assert ops.encode_png_batch(engine, imgs[::-1]) == batch[::-1]


@pytest.mark.gpu
def test_overflow_reports_the_exact_size(engine, golden_dir):
    import torch
    corpus = _golden_corpus(golden_dir)
    imgs = [torch.from_numpy(corpus[k]).to(engine.device) for k in ("bev_synth", "density_synth", "view_1")]
    want = engine.run_png_encode(imgs).to_host()
    total = sum(len(f) for f in want)
    small = engine.alloc_png(imgs, out_bytes=total - 1)
    small.arena.fill_(0xab)
    with pytest.raises(_capi.MscError) as e:
        engine.run_png_encode(imgs, out=small).to_host()
    assert e.value.status == 1 and small.needed == total
    assert bool((small.arena == 0xab).all())  # nothing written
    exact = engine.run_png_encode(imgs, out=engine.alloc_png(imgs, out_bytes=small.needed)).to_host()
    assert exact == want


def _agent_corpus(engine, golden_dir):
    """The agent's images: the golden BEVs, views and mosaic, and the test batch's BEVs and mosaics (RGB, as Pillow gets them)."""
    import torch
    from msc_geom.lidar_agent import LiDARAgent, set_order
    from tests.test_lidar_images import _batch, _golden_samples, _mixed_samples
    imgs = list(_golden_corpus(golden_dir).values())
    lr = _batch(engine, _golden_samples(golden_dir) + _mixed_samples(golden_dir)[5:7])
    bev = engine.run_lidar_bev(lr, 800, 50.0)
    imgs += [np.ascontiguousarray(s["semantic"][..., ::-1]) for s in bev.to_host(("semantic",))]
    per = lr.to_host()
    views = [(r["object_off"], r["object_off"] + len(r["object"]), l) for r in per for l in set_order(r["cluster_first"], r["noise_first"])
             if int(r["clusters"][l, 10]) >= 5]
    vr = engine.run_cluster_views(lr.object, lr.labels, views)
    groups = [(a, min(10, len(views) - a)) for a in range(0, len(views), 10)]
    mos = engine.run_cluster_mosaics(vr, groups)
    imgs += [np.ascontiguousarray(m.cpu().numpy()[..., ::-1]) for m in mos.images]
    return imgs


@pytest.mark.gpu
def test_size_bars_on_the_agent_images(engine, golden_dir):
    """The files against Pillow's on the agent's images: all together at most 1.15 times Pillow's bytes, none above 1.35 times."""
    from msc_geom import ops
    imgs = _agent_corpus(engine, golden_dir)
    assert len(imgs) > 20
    files = ops.encode_png_batch(engine, imgs)
    ref = [len(pillow_png(im)) for im in imgs]
    ratios = [len(f) / r for f, r in zip(files, ref)]
    print("size ratios: total %.4f, worst %.4f" % (sum(len(f) for f in files) / sum(ref), max(ratios)))
    assert sum(len(f) for f in files) <= 1.15 * sum(ref), sum(len(f) for f in files) / sum(ref)
    assert max(ratios) <= 1.35, max(ratios)
    for f, im in zip(files, imgs):
        check_file(f, im)


@pytest.mark.gpu
def test_mosaics_equal_cluster_mosaic(engine, golden_dir):
    import torch
    from msc_geom.engine import ClusterViewsResult
    g = np.load(os.path.join(golden_dir, "cluster_views.npz"))
    golden = np.stack([g[f"img_{k}"] for k in range(int(g["n"]))])
    rng = np.random.default_rng(3)
    rand = rng.integers(0, 256, (12, 512, 512, 3), np.uint8)
    views = np.concatenate([golden, rand])
    vr = ClusterViewsResult(len(views), torch.from_numpy(views).to(engine.device), torch.zeros(1, dtype=torch.int32, device=engine.device))
    groups = [(0, 5)] + [(len(golden) + 12 - c, c) for c in range(1, 11)] + [(2, 1), (0, 6)]
    mos = engine.run_cluster_mosaics(vr, groups)
    got = [m.cpu().numpy() for m in mos.images]
    assert np.array_equal(got[0], g["mosaic"])
    for (f, c), m in zip(groups, got):
        assert np.array_equal(m, cluster_mosaic(list(views[f:f + c]))), (f, c)


@pytest.mark.gpu
def test_process_batch_png_against_arrays(engine, golden_dir, monkeypatch):
    """process_batch(png=True) hands the callables what goes on the wire, with the same results, calls and metadata as png=False."""
    from msc_geom import lidar_agent
    from msc_geom.lidar_agent import LiDARAgent
    from tests.test_lidar_batch import _Recorder, _json_form
    from tests.test_lidar_images import _golden_samples, _mixed_samples
    monkeypatch.setattr(lidar_agent, "CLUSTER_IMAGES_PER_CALL", 7)

    class PngRecorder(_Recorder):
        def llm(self, messages, **kw):
            self.llm_calls.append((messages, kw.get("bev_png")))
            return "seen %d" % len(self.llm_calls)

    samples = _golden_samples(golden_dir) + _mixed_samples(golden_dir)[5:7]
    ra, rb = _Recorder(), PngRecorder()
    a = LiDARAgent(object(), "m", "LiDARAgent", engine=engine, llm=ra.llm, cluster_classifier=ra.classifier)
    b = LiDARAgent(object(), "m", "LiDARAgent", engine=engine, llm=rb.llm, cluster_classifier=rb.classifier)
    want = a.process_batch(samples)
    got = b.process_batch(samples, png=True)
    assert [_json_form(x) for x in got] == [_json_form(x) for x in want]
    assert len(ra.calls) == len(rb.calls) > 2
    for (ia, ma, meta_a), (ib, mb, meta_b) in zip(ra.calls, rb.calls):
        assert ib is None and isinstance(mb, str)
        assert json.dumps(meta_a, default=_plain) == json.dumps(meta_b, default=_plain)
        png = base64.b64decode(mb)
        check_file(png, np.ascontiguousarray(cluster_mosaic(ia)[..., ::-1]))
    assert len(ra.llm_calls) == len(rb.llm_calls) == len(samples)
    for (ma, sa), (mb, pb) in zip(ra.llm_calls, rb.llm_calls):
        assert ma == mb
        check_file(base64.b64decode(pb), np.ascontiguousarray(sa[..., ::-1]))


def _plain(v):
    return v.tolist() if isinstance(v, np.ndarray) else float(v)



@pytest.mark.gpu
def test_process_batch_png_with_an_llm_and_no_classifier(engine, golden_dir):
    """png=True on an agent with an llm but no cluster classifier: the clusters take the default classification, as with png=False."""
    from msc_geom.lidar_agent import LiDARAgent
    from tests.test_lidar_batch import _json_form
    from tests.test_lidar_images import _golden_samples
    seen_a, seen_b = [], []
    a = LiDARAgent(object(), "m", "LiDARAgent", engine=engine, llm=lambda m, **kw: seen_a.append(kw["bev_semantic"]) or "ok")
    b = LiDARAgent(object(), "m", "LiDARAgent", engine=engine, llm=lambda m, **kw: seen_b.append(kw["bev_png"]) or "ok")
    samples = _golden_samples(golden_dir)
    want = a.process_batch(samples)
    got = b.process_batch(samples, png=True)
    assert [_json_form(x) for x in got] == [_json_form(x) for x in want]
    assert len(seen_a) == len(seen_b) == len(samples)
    for arr, text in zip(seen_a, seen_b):
        check_file(base64.b64decode(text), np.ascontiguousarray(arr[..., ::-1]))
