"""Device JPEG encode (msc_jpeg_encode_batch): every file must equal, byte for byte, what Pillow's
`Image.fromarray(img).save(buf, "JPEG", quality=q)` writes -- the reference's CameraAgent._encode_image (camera_agent.py:128-137)."""
import base64
import ctypes as C
from io import BytesIO

import numpy as np
import pytest
from PIL import Image

from msc_geom import _capi

QUALITIES = (1, 20, 50, 85, 95, 100)
SIZES = ((1, 1), (2, 3), (3, 2), (8, 8), (9, 17), (16, 16), (17, 33), (31, 45), (240, 321), (900, 1600))  # (H, W)


def pil_jpeg(img, q=85):
    buf = BytesIO()
    Image.fromarray(img).save(buf, format="JPEG", quality=q)
    return buf.getvalue()


def scene(rng, h, w):
    """Smooth structure + texture + hard edges + noise (like test_gpu_parity's frames), so every coefficient band is exercised."""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([127 + 120 * np.sin(xx / 17.0 + yy / 29.0), 127 + 120 * np.cos(xx / 7.0), 255 * ((xx // 13 + yy // 11) % 2)], -1)
    return np.clip(base + rng.normal(0, 25, (h, w, 3)), 0, 255).astype(np.uint8)


def contents(rng, h, w):
    return {"scene": scene(rng, h, w), "noise": rng.integers(0, 256, (h, w, 3), dtype=np.uint8),
            "constant": np.full((h, w, 3), (90, 160, 30), np.uint8), "black": np.zeros((h, w, 3), np.uint8),
            "white": np.full((h, w, 3), 255, np.uint8)}


def _coefficients(lib, data):
    buf = np.frombuffer(data, np.uint8)
    d = _capi.MscJpegDesc()
    _capi.check(lib.msc_jpeg_info(buf.ctypes.data, buf.size, C.byref(d)), "msc_jpeg_info")
    coef = np.zeros(int(d.coef_elems), np.int16)
    _capi.check(lib.msc_jpeg_entropy_decode_host(buf.ctypes.data, buf.size, C.byref(d), coef.ctypes.data), "msc_jpeg_entropy_decode_host")
    return d, coef


def first_difference(mine, ref):
    """Where two files of the same image first differ: the header, or the first (MCU, component) whose decoded coefficients differ."""
    lib = _capi.load()
    i = ref.index(b"\xff\xda") + 14
    if mine[:i] != ref[:i]:
        k = next(k for k in range(i) if k >= len(mine) or mine[k] != ref[k])
        return "headers differ at byte %d" % k
    try:
        d, a = _coefficients(lib, mine)
    except _capi.MscError as e:
        return "our scan does not decode: %s" % e
    _, b = _coefficients(lib, ref)
    best = None
    for c in range(d.n_comp):
        k = d.comp[c]
        n = k.blocks_x * k.blocks_y
        x = a[k.coef_off:k.coef_off + 64 * n].reshape(n, 64)
        y = b[k.coef_off:k.coef_off + 64 * n].reshape(n, 64)
        bad = np.nonzero((x != y).any(1))[0]
        if bad.size:
            by, bx = divmod(int(bad[0]), k.blocks_x)
            mcu = (by // k.v) * d.mcus_x + bx // k.h
            if best is None or (mcu, c) < best[:2]:
                best = (mcu, c, x[bad[0]], y[bad[0]])
    if best is None:
        return "same coefficients, scans differ (len %d vs %d)" % (len(mine), len(ref))
    mcu, c, x, y = best
    return "MCU %d (row %d, col %d), component %d: ours %s, Pillow's %s" % (mcu, mcu // d.mcus_x, mcu % d.mcus_x, c, x.tolist(), y.tolist())


def assert_files_equal(got, frames, q, labels):
    bad = []
    for f, img, lab in zip(got, frames, labels):
        ref = pil_jpeg(img, q)
        if f != ref:
            bad.append("%s q=%d %s: %s" % (lab, q, img.shape, first_difference(f, ref)))
    assert not bad, "%d of %d files differ from Pillow's; first: %s" % (len(bad), len(got), bad[:3])


# ---------------------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("q", QUALITIES)
def test_bytes_equal_pillow(engine, q):
    """Partial MCUs in both directions, a bottom row of dummy blocks (900 rows), noise (longest codes, 0xFF bytes, ZRL runs), constant
    images (all-EOB blocks) and the DC extremes, at every quality."""
    from msc_geom import ops
    rng = np.random.default_rng(100 + q)
    frames, labels = [], []
    for h, w in SIZES:
        for name, img in contents(rng, h, w).items():
            frames.append(img)
            labels.append(name)
    got = ops.encode_jpeg_batch(engine, frames, quality=q)
    assert_files_equal(got, frames, q, labels)


@pytest.mark.gpu
def test_many_small_random_images(engine):
    """About 600 seeded small images of random size, content and quality; at least one scan ends in a stuffed 0xFF (its last byte, padded
    with 1-bits, became 0xFF)."""
    from msc_geom import ops
    rng = np.random.default_rng(7)
    frames, qs = [], []
    for _ in range(600):
        h, w = (int(v) for v in rng.integers(1, 41, 2))
        frames.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if rng.random() < 0.7 else scene(rng, h, w))
        qs.append(int(rng.choice(QUALITIES)))
    by_q = {}
    for k, q in enumerate(qs):
        by_q.setdefault(q, []).append(k)
    stuffed_tail = 0
    for q, idx in by_q.items():
        got = ops.encode_jpeg_batch(engine, [frames[k] for k in idx], quality=q)
        assert_files_equal(got, [frames[k] for k in idx], q, ["random %d" % k for k in idx])
        stuffed_tail += sum(f.endswith(b"\xff\x00\xff\xd9") for f in got)
    assert stuffed_tail >= 1


def camera_frames(n, seed=3, h=900, w=1600):
    """n distinct camera-like frames: one scene, shifted and re-noised per frame."""
    rng = np.random.default_rng(seed)
    base = scene(rng, h, w).astype(np.int16)
    return [np.clip(np.roll(base, 37 * k, axis=1) + rng.integers(-12, 13, (h, w, 3), dtype=np.int16), 0, 255).astype(np.uint8) for k in range(n)]


@pytest.mark.gpu
def test_batch_of_64_frames_independent_of_position_and_batch_size(engine):
    import torch
    frames = camera_frames(64)
    dev = torch.from_numpy(np.stack(frames)).to(engine.device)
    got = engine.run_jpeg_encode(dev, 85).to_host()
    assert_files_equal(got, frames, 85, ["frame %d" % k for k in range(64)])
    perm = np.random.default_rng(5).permutation(64)
    shuffled = engine.run_jpeg_encode(dev[torch.from_numpy(perm).to(engine.device)].contiguous(), 85).to_host()
    assert all(shuffled[i] == got[perm[i]] for i in range(64))
    for k in (0, 17, 63):
        assert engine.run_jpeg_encode(dev[k:k + 1].contiguous(), 85).to_host()[0] == got[k]
    three = engine.run_jpeg_encode(dev[5:8].contiguous(), 85).to_host()
    assert three == got[5:8]


@pytest.mark.gpu
def test_overflow_sets_status_writes_nothing_and_reports_the_exact_size(engine):
    import torch
    from msc_geom import ops
    frames = [f[:120, :200] for f in camera_frames(3, seed=11)] + [np.random.default_rng(1).integers(0, 256, (120, 200, 3), dtype=np.uint8)]
    refs = [pil_jpeg(f, 95) for f in frames]
    dev = torch.from_numpy(np.stack(frames)).to(engine.device)
    small = 1000
    res = engine.alloc_jpeg(4, 120, 200, out_bytes=small)
    guard = torch.full((small + 4096,), 0xA5, dtype=torch.uint8, device=engine.device)
    res.arena = guard[:small]
    engine.run_jpeg_encode(dev, 95, out=res)
    with pytest.raises(_capi.MscError, match="need %d bytes" % sum(map(len, refs))) as ei:
        res.to_host()
    assert ei.value.status == 1
    assert bool((guard == 0xA5).all()), "the call wrote into an arena that is too small"
    assert res.out_off.cpu().numpy().tolist() == np.concatenate([[0], np.cumsum([len(r) for r in refs])]).tolist()
    again = engine.run_jpeg_encode(dev, 95, out=engine.alloc_jpeg(4, 120, 200, out_bytes=res.needed))
    assert again.to_host() == refs
    # the default arena (half the raw bytes) is too small for noise at q=100; ops retries with the exact size on its own
    noise = [np.random.default_rng(2 + k).integers(0, 256, (64, 64, 3), dtype=np.uint8) for k in range(3)]
    assert ops.encode_jpeg_batch(engine, noise, quality=100) == [pil_jpeg(f, 100) for f in noise]


@pytest.mark.gpu
def test_large_lists_are_split_by_workspace(engine, monkeypatch):
    """ops.encode_jpeg_batch splits a shape group into calls of at most JPEG_WORKSPACE_PER_CALL bytes of workspace; the files stay
    Pillow's, in order, for host lists and for one [N, H, W, 3] tensor."""
    import torch
    from msc_geom import ops
    rng = np.random.default_rng(17)
    frames = [scene(rng, 40, 56) for _ in range(5)]
    per_frame = int(engine.lib.msc_jpeg_encode_workspace_bytes(1, 40, 56, 0))
    monkeypatch.setattr(ops, "JPEG_WORKSPACE_PER_CALL", 2 * per_frame)
    launches = engine.kernel_launches
    refs = [pil_jpeg(f) for f in frames]
    assert ops.encode_jpeg_batch(engine, frames) == refs
    assert engine.kernel_launches - launches == 3 * 6  # calls of 2, 2 and 1 frames
    assert ops.encode_jpeg_batch(engine, torch.from_numpy(np.stack(frames)).to(engine.device)) == refs


@pytest.mark.gpu
def test_cuda_graph_capture_and_replay(engine):
    """The call allocates nothing and never synchronises the host: it can be captured in a CUDA graph and replayed."""
    import torch
    frames = camera_frames(6, seed=21)
    dev = torch.from_numpy(np.stack(frames)).to(engine.device)
    out = engine.alloc_jpeg(6, 900, 1600)
    engine.run_jpeg_encode(dev, 85, out=out)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        engine.run_jpeg_encode(dev, 85, out=out)
    out.arena.zero_()
    out.small.zero_()
    g.replay()
    assert out.to_host() == [pil_jpeg(f, 85) for f in frames]
    dev.copy_(torch.from_numpy(np.stack(frames[::-1])).to(engine.device))
    g.replay()
    assert out.to_host() == [pil_jpeg(f, 85) for f in frames[::-1]]


@pytest.mark.gpu
def test_camera_agent_device_path_equals_pil_path(engine):
    from msc_geom import ops
    from msc_geom.camera_agent import CameraAgent
    names = ["CAM_FRONT", "CAM_FRONT_LEFT", "CAM_FRONT_RIGHT", "CAM_BACK", "CAM_BACK_LEFT", "CAM_BACK_RIGHT"]
    frames = camera_frames(6, seed=31)
    plain = CameraAgent(None, "m", "camera")
    fast = CameraAgent(None, "m", "camera", engine=engine)
    assert fast.user_content(frames, names, {"k": 1}) == plain.user_content(frames, names, {"k": 1})
    # device frames straight from the decoder: no raw frame crosses PCIe
    blobs = [pil_jpeg(f, 90) for f in frames]
    on_device = ops.decode_jpeg_batch(engine, blobs, to_host=False)
    on_host = ops.decode_jpeg_batch(engine, blobs)
    assert fast.user_content(on_device, names) == plain.user_content(on_host, names)
    # a grayscale frame in the list still takes Pillow's path
    gray = frames[2][..., 1].copy()
    mixed = [frames[0], gray, frames[1]]
    assert fast.user_content(mixed, names[:3]) == plain.user_content(mixed, names[:3])


@pytest.mark.gpu
def test_refusals_and_empty_batch(engine):
    import torch
    from msc_geom import ops
    assert ops.encode_jpeg_batch(engine, []) == []
    res = engine.run_jpeg_encode(torch.empty((0, 16, 16, 3), dtype=torch.uint8, device=engine.device))
    assert res.to_host() == []
    with pytest.raises(_capi.MscError, match="quality"):
        ops.encode_jpeg_batch(engine, [np.zeros((8, 8, 3), np.uint8)], quality=0)
    for bad in (np.zeros((8, 8), np.uint8), np.zeros((8, 8, 4), np.uint8), torch.zeros((8, 8, 3), dtype=torch.float32, device=engine.device)):
        with pytest.raises(_capi.MscError):
            ops.encode_jpeg_batch(engine, [bad])


# ---------------------------------------------------------------------------------------------------------------------------- CPU
def test_argument_refusals_without_a_device():
    """Bad arguments are refused with MSC_ERR_BAD_ARGUMENT before anything is launched (on a box without a device, a launch would fail
    with another status)."""
    lib = _capi.load()
    need = int(lib.msc_jpeg_encode_workspace_bytes(2, 16, 16, 0))
    assert need > 0
    assert lib.msc_jpeg_encode_workspace_bytes(2, 0, 16, 0) == 0 and lib.msc_jpeg_encode_workspace_bytes(2, 16, 65536, 0) == 0
    p = 1 << 20  # a 256-byte aligned address that is never dereferenced

    def call(n=2, h=16, w=16, q=85, rgb=p, out=p, out_off=p, status=p, ws=p, ws_bytes=need):
        return lib.msc_jpeg_encode_batch(n, h, w, q, rgb, out, 1 << 16, out_off, status, ws, ws_bytes, None)

    for kw in ({"q": 0}, {"q": 101}, {"h": 0}, {"h": 65536}, {"w": 0}, {"w": 65536}, {"n": -1}, {"rgb": None}, {"out": None},
               {"out_off": None}, {"status": None}, {"ws": None}, {"ws_bytes": need - 1}):
        assert call(**kw) == _capi.MSC_ERR_BAD_ARGUMENT, kw
    assert call(n=0, rgb=None, out=None, out_off=None, status=None, ws=None, ws_bytes=0) == 0


def test_user_content_routes_rgb_frames_to_the_device_encoder(monkeypatch):
    """With an engine, only (H, W, 3) frames -- after the reference's uint8 conversion -- reach the device encoder, in order, in one
    call; every other frame keeps Pillow's path and its result."""
    from msc_geom import ops, serialize
    from msc_geom.camera_agent import CameraAgent
    rng = np.random.default_rng(0)
    rgb = rng.integers(0, 256, (24, 40, 3), dtype=np.uint8)
    flt = rng.random((16, 16, 3))
    gray = rng.integers(0, 256, (24, 40), dtype=np.uint8)
    rgba = rng.integers(0, 256, (24, 40, 4), dtype=np.uint8)
    rgb2 = rng.integers(0, 256, (24, 40, 3), dtype=np.uint8)
    calls = []

    def fake(eng, images, quality=85):
        calls.append((eng, [np.array(i) for i in images], quality))
        return [b"frame-%d" % k for k in range(len(images))]
    monkeypatch.setattr(ops, "encode_jpeg_batch", fake)
    eng = object()
    frames = [rgb, gray, flt, rgb2]
    names = ["A", "B", "C", "D"]
    content = CameraAgent(None, "m", "camera", engine=eng).user_content(frames, names)
    assert len(calls) == 1 and calls[0][0] is eng and calls[0][2] == 85
    sent = calls[0][1]
    assert len(sent) == 3 and all(s.dtype == np.uint8 and s.ndim == 3 and s.shape[2] == 3 for s in sent)
    assert np.array_equal(sent[0], rgb) and np.array_equal(sent[1], (flt * 255).astype(np.uint8)) and np.array_equal(sent[2], rgb2)
    urls = [c["image_url"]["url"] for c in content if c["type"] == "image_url"]
    expect = [base64.b64encode(b"frame-0").decode(), serialize.jpeg_base64(gray), base64.b64encode(b"frame-1").decode(),
              base64.b64encode(b"frame-2").decode()]
    assert urls == ["data:image/jpeg;base64," + e for e in expect]
    # without an engine nothing changes: every frame goes through Pillow
    calls.clear()
    plain = CameraAgent(None, "m", "camera").user_content(frames, names)
    assert not calls
    assert [c["image_url"]["url"] for c in plain if c["type"] == "image_url"] == ["data:image/jpeg;base64," + serialize.jpeg_base64(f) for f in frames]
    # an RGBA frame is Pillow's as before, with or without an engine: JPEG cannot hold it, and the error is Pillow's
    for agent in (CameraAgent(None, "m", "camera", engine=eng), CameraAgent(None, "m", "camera")):
        with pytest.raises(OSError):
            agent.user_content([rgb, rgba], ["A", "B"])
