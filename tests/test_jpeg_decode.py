"""Batched device JPEG decode (msc_jpeg_decode_batch): coefficients equal to the host Huffman decoder (msc_jpeg_entropy_decode_host) and
frames equal to np.array(Image.open(...)) -- NuScenesLoader._load_camera -- for every file of a batch, decoded in one call."""
import ctypes as C
import importlib
import os
import sys
from io import BytesIO

import numpy as np
import pytest
from PIL import Image

from msc_geom import _capi
from msc_geom.synthetic import make_sample

SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "devkit_shim")


def jpeg(img, **kw):
    b = BytesIO()
    Image.fromarray(img).save(b, "JPEG", **kw)
    return b.getvalue()


def scene(rng, h, w):
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([127 + 120 * np.sin(xx / 17.0 + yy / 29.0), 127 + 120 * np.cos(xx / 7.0), 255 * ((xx // 13 + yy // 11) % 2)], -1)
    return np.clip(base + rng.normal(0, 25, (h, w, 3)), 0, 255).astype(np.uint8)


def plan(lib, data):
    p = _capi.MscJpegPlan()
    buf = np.frombuffer(data, np.uint8)
    return lib.msc_jpeg_decode_plan(buf.ctypes.data, buf.size, C.byref(p)), p


def host_coef(lib, data):
    """(status, coefficients) of the host Huffman decoder."""
    buf = np.frombuffer(data, np.uint8)
    d = _capi.MscJpegDesc()
    _capi.check(lib.msc_jpeg_info(buf.ctypes.data, buf.size, C.byref(d)), "msc_jpeg_info")
    coef = np.zeros(int(d.coef_elems), np.int16)
    rc = lib.msc_jpeg_entropy_decode_host(buf.ctypes.data, buf.size, C.byref(d), coef.ctypes.data)
    return rc, coef


def corpus():
    """The cases of test_jpeg_decode_equals_pil_bit_for_bit, plus the streams that are hard for a parallel Huffman decode."""
    rng = np.random.default_rng(11)
    cases = []
    for (h, w) in ((16, 16), (17, 33), (1, 1), (2, 3), (3, 2), (8, 5), (9, 4), (31, 64), (240, 321)):
        img = scene(rng, h, w)
        for sub in (0, 1, 2):
            for q in (35, 90, 100):
                cases.append(jpeg(img, quality=q, subsampling=sub))
        cases.append(jpeg(img, quality=75, subsampling=2, optimize=True))
        cases.append(jpeg(img[..., 0].copy(), quality=80))
    big = scene(rng, 900, 1600)
    cases.append(jpeg(big, quality=90, subsampling=2))
    cases.append(jpeg(rng.integers(0, 256, (64, 96, 3), dtype=np.uint8), quality=95, subsampling=2))
    cases.append(jpeg(big[:200, :301], quality=85, subsampling=2, restart_marker_blocks=7))
    cases.append(jpeg(big[:100, :200], quality=85, subsampling=1, restart_marker_rows=1))
    # flat colour: a periodic code stream that need never self-synchronise
    for sub in (0, 1, 2):
        cases.append(jpeg(np.full((900, 1600, 3), (90, 160, 30), np.uint8), quality=90, subsampling=sub))
    cases.append(jpeg(np.zeros((900, 1600), np.uint8), quality=90))
    cases.append(jpeg(rng.integers(0, 256, (300, 500, 3), dtype=np.uint8), quality=100, subsampling=0))  # stuffed FFs, long codes
    cases.append(jpeg(big[:120, :250], quality=90, subsampling=2, restart_marker_blocks=1))  # restart interval 1
    d = jpeg(big[:64, :80], quality=90)
    cases.append(d[:-2] + bytes(rng.integers(0, 255, 300, dtype=np.uint8)) + b"\xff\xd9")  # garbage between the last MCU and EOI
    return cases


def decode(engine, datas, pad=0, sentinel=None, chunk=None):
    """One msc_jpeg_decode_batch call per `chunk` files (default: all): (status, coefficient arrays, frames, coef arena, out arena).
    Regions are separated by `pad` elements, and arenas pre-filled with `sentinel`, to expose writes outside an image's region."""
    import torch
    lib = engine.lib
    n = len(datas)
    plans = (_capi.MscJpegPlan * n)()
    file_off = np.zeros(n, np.int64)
    blob = b""
    for k, d in enumerate(datas):
        rc, p = plan(lib, d)
        assert rc == 0
        plans[k] = p
        file_off[k] = len(blob)
        blob += d + b"\0" * ((-len(d)) % 16 + 16)
    shapes = [(p.desc.height, p.desc.width, 3) if p.desc.n_comp == 3 else (p.desc.height, p.desc.width) for p in plans]
    coef_off, out_off = np.zeros(n, np.int64), np.zeros(n, np.int64)
    c = o = pad
    for k, p in enumerate(plans):
        coef_off[k], out_off[k] = c, o
        c += int(p.desc.coef_elems) + pad
        o += int(np.prod(shapes[k])) + pad
    dev = engine.device
    files = torch.from_numpy(np.frombuffer(blob, np.uint8).copy()).to(dev)
    coef = torch.full((c,), sentinel if sentinel is not None else 0, dtype=torch.int16, device=dev)
    out = torch.full((o,), sentinel if sentinel is not None else 0, dtype=torch.uint8, device=dev)
    status = torch.full((n,), 77, dtype=torch.int32, device=dev)
    chunk = chunk or n
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for a in range(0, n, chunk):
        k = min(chunk, n - a)
        base = C.addressof(plans) + a * C.sizeof(_capi.MscJpegPlan)
        need = int(lib.msc_jpeg_decode_batch_workspace_bytes(k, base))
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        _capi.check(lib.msc_jpeg_decode_batch(k, base, files.data_ptr(), file_off[a:].ctypes.data, coef.data_ptr(), coef_off[a:].ctypes.data,
                                              out.data_ptr(), out_off[a:].ctypes.data, status[a].data_ptr(), ws.data_ptr(), need, stream),
                    "msc_jpeg_decode_batch")
    st, ch, oh = status.cpu().numpy(), coef.cpu().numpy(), out.cpu().numpy()
    coefs = [ch[coef_off[k]:coef_off[k] + int(plans[k].desc.coef_elems)] for k in range(n)]
    frames = [oh[out_off[k]:out_off[k] + int(np.prod(shapes[k]))].reshape(shapes[k]) for k in range(n)]
    return st, coefs, frames, (ch, coef_off, [int(p.desc.coef_elems) for p in plans]), (oh, out_off, [int(np.prod(s)) for s in shapes])


def nuscenes_tree(tmp_path, n_samples=2, h=90, w=160):
    from msc_geom import io as mio
    rng = np.random.default_rng(3)
    sc = []
    for k in range(n_samples):
        s = make_sample(700 + k, n_sweeps=1, n_boxes=3)
        s["images"] = [scene(rng, h, w) for _ in s["cameras"]]
        s["scene_name"], s["scene_description"] = "scene-0000", "jpeg"
        sc.append(s)
    mio.write_nuscenes_tree(str(tmp_path), [sc])


@pytest.fixture()
def loader_module():
    """The loader with tests/devkit_shim standing in for the devkit; the shim and its modules are removed afterwards."""
    import msc_geom.nuscenes_loader as nl
    sys.path.insert(0, SHIM)
    importlib.reload(nl)
    yield nl
    sys.path.remove(SHIM)
    for m in [m for m in sys.modules if m == "nuscenes" or m.startswith("nuscenes.")]:
        del sys.modules[m]
    importlib.reload(nl)


# ------------------------------------------------------------------------------------------------ CPU
def test_plan_agrees_with_jpeg_info_and_refuses_the_same_files():
    lib = _capi.load()
    rng = np.random.default_rng(5)
    img = scene(rng, 40, 56)
    datas = corpus()[:40] + [jpeg(img, quality=85, subsampling=2, restart_marker_blocks=3)]
    fields = ("width", "height", "n_comp", "hmax", "vmax", "mcus_x", "mcus_y", "coef_elems", "plane_bytes")
    for d in datas:
        rc, p = plan(lib, d)
        ref = _capi.MscJpegDesc()
        buf = np.frombuffer(d, np.uint8)
        assert rc == lib.msc_jpeg_info(buf.ctypes.data, buf.size, C.byref(ref)) == 0
        assert bytes(p.desc) == bytes(ref), [(f, getattr(p.desc, f), getattr(ref, f)) for f in fields]
        sos = d.rindex(b"\xff\xda", 0, p.scan_off)  # the scan starts right after the SOS segment and runs to the end of the file
        assert sos + 2 + (d[sos + 2] << 8 | d[sos + 3]) == p.scan_off and p.scan_off + p.scan_bytes == len(d)
        assert int(lib.msc_jpeg_decode_batch_workspace_bytes(1, C.addressof(p))) > 0
    _, p = plan(lib, datas[-1])
    assert p.restart_interval == 3
    for bad in (jpeg(img, progressive=True), b"not a jpeg at all", b"\xff\xd8\xff\xd9", jpeg(img)[:300]):
        rc, _ = plan(lib, bad)
        buf = np.frombuffer(bad, np.uint8)
        assert rc == lib.msc_jpeg_info(buf.ctypes.data, buf.size, C.byref(_capi.MscJpegDesc())) != 0
    assert plan(lib, jpeg(img, progressive=True))[0] == _capi.MSC_ERR_UNSUPPORTED


def test_batch_refuses_bad_arguments_without_a_device():
    lib = _capi.load()
    rc, p = plan(lib, jpeg(scene(np.random.default_rng(1), 24, 24)))
    plans = (_capi.MscJpegPlan * 1)(p)
    need = int(lib.msc_jpeg_decode_batch_workspace_bytes(1, C.addressof(plans)))
    off = np.zeros(1, np.int64)
    fake = 1 << 20  # never dereferenced: every refusal happens before anything is launched

    def call(n=1, plans_=C.addressof(plans), files=fake, coef=fake, out=fake, status=fake, ws=fake, ws_bytes=need, coef_off=off.ctypes.data):
        return lib.msc_jpeg_decode_batch(n, plans_, files, off.ctypes.data, coef, coef_off, out, off.ctypes.data, status, ws, ws_bytes, None)
    for kw in ({"n": -1}, {"plans_": None}, {"files": None}, {"coef": None}, {"out": None}, {"status": None}, {"ws": None},
               {"ws_bytes": need - 1}, {"ws": fake + 16}, {"coef_off": np.array([3], np.int64).ctypes.data}):
        assert call(**kw) == _capi.MSC_ERR_BAD_ARGUMENT, kw
    assert call(n=0, plans_=None, files=None, coef=None, out=None, status=None, ws=None, ws_bytes=0) == 0
    broken = (_capi.MscJpegPlan * 1)(p)
    broken[0].desc.mcus_x += 1  # a descriptor parse_headers would not write
    assert lib.msc_jpeg_decode_batch_workspace_bytes(1, C.addressof(broken)) == 0
    assert call(plans_=C.addressof(broken)) == _capi.MSC_ERR_BAD_ARGUMENT
    assert lib.msc_jpeg_decode_batch_workspace_bytes(-1, C.addressof(plans)) == 0


def test_run_jpeg_decode_refuses_buffers_of_other_files_without_a_device(tmp_path):
    """Buffers allocated for other files (more pixels, another subsampling, fewer files) are refused before anything is copied or
    launched: their regions would not hold the new files' coefficients and frames."""
    import torch
    from msc_geom import io as mio
    from msc_geom.engine import GeometryEngine, JpegDecodeResult, jpeg_decode_layout
    rng = np.random.default_rng(8)

    def staged(specs):
        cams = []
        for k, (h, w, sub) in enumerate(specs):
            path = str(tmp_path / ("f%d_%d_%d_%d.jpg" % (k, h, w, sub)))
            open(path, "wb").write(jpeg(scene(rng, h, w), quality=90, subsampling=sub))
            cams.append({"path": path})
        return mio.stage_camera_files([{"cameras": cams}], pinned=False)

    def buffers(st):  # what alloc_jpeg_decode allocates, on the host
        shapes, coef_off, out_off = jpeg_decode_layout(st)
        n_coef = sum(int(st.plans[k].desc.coef_elems) for k in range(len(st)))
        return JpegDecodeResult(shapes, torch.empty(n_coef, dtype=torch.int16), coef_off, torch.empty(int(out_off[-1]), dtype=torch.uint8), out_off,
                                torch.zeros(len(st), dtype=torch.int32), torch.empty(st.nbytes, dtype=torch.uint8), torch.empty(256, dtype=torch.uint8))
    small = staged([(32, 48, 2), (32, 48, 2)])
    eng = object.__new__(GeometryEngine)  # the refusal needs neither a device nor the library
    for other in (staged([(64, 96, 2), (32, 48, 2)]), staged([(32, 48, 0), (32, 48, 2)]), staged([(32, 48, 2), (32, 48, 2), (16, 16, 2)]),
                  staged([(32, 48, 2)])):
        with pytest.raises(_capi.MscError) as e:
            eng.run_jpeg_decode(other, buffers(small))
        assert e.value.status == _capi.MSC_ERR_BAD_ARGUMENT
    short = buffers(small)
    short.out = short.out[:-1]
    with pytest.raises(_capi.MscError):
        eng.run_jpeg_decode(small, short)


def test_stage_camera_files_reads_exact_bytes(tmp_path):
    from msc_geom import io as mio
    nuscenes_tree(tmp_path)
    rng = np.random.default_rng(2)
    prog = str(tmp_path / "progressive.jpg")
    Image.fromarray(scene(rng, 32, 48)).save(prog, "JPEG", progressive=True)
    paths = sorted(str(p) for p in (tmp_path / "samples").rglob("*.jpg"))
    samples = [{"cameras": [{"path": p} for p in paths[:6]]}, {"cameras": [{"path": prog}] + [{"path": p} for p in paths[6:]]}]
    st = mio.stage_camera_files(samples, threads=3, pinned=False)
    assert st.unsupported == [(1, 0, prog)]
    assert st.index == [(0, c) for c in range(6)] + [(1, c) for c in range(1, 7)]
    lib = _capi.load()
    for k, (i, c) in enumerate(st.index):
        want = open(samples[i]["cameras"][c]["path"], "rb").read()
        a = int(st.file_off[k])
        assert a % 256 == 0 and int(st.size[k]) == len(want) and st.data[a:a + len(want)].tobytes() == want
        assert bytes(st.plans[k]) == bytes(plan(lib, want)[1])
    bad = str(tmp_path / "junk.jpg")
    open(bad, "wb").write(b"not a jpeg at all")
    with pytest.raises(_capi.MscError):
        mio.stage_camera_files([{"cameras": [{"path": bad}]}], pinned=False)


def test_lazy_loader_cameras_carry_paths_and_eager_output_is_unchanged(tmp_path, loader_module):
    nuscenes_tree(tmp_path)
    nl = loader_module
    eager = nl.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=1)
    lazy = nl.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=1, lazy_sweeps=True)
    tok = eager.scene_sample_tokens(eager.get_scene_list()[0]["token"])[0]
    e, z = eager.load_sample(tok), lazy.load_sample(tok)
    assert z["images"] == [] and len(z["cameras"]) == 6
    assert all(os.path.isfile(c["path"]) and c["channel"] in c["path"] for c in z["cameras"])
    assert all(set(c) == {"channel", "ego_pose", "calib", "intrinsic"} for c in e["cameras"])
    assert len(e["images"]) == 6 and all(np.array_equal(a, np.array(Image.open(c["path"]))) for a, c in zip(e["images"], z["cameras"]))


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_corpus_equals_host_decoder_and_pil(engine):
    datas = corpus()
    st, coefs, frames, _, _ = decode(engine, datas)
    for k, d in enumerate(datas):
        rc, ref = host_coef(engine.lib, d)
        assert rc == 0 and st[k] == 0, (k, rc, st[k])
        assert np.array_equal(coefs[k], ref), (k, int((coefs[k] != ref).sum()))
        pil = np.array(Image.open(BytesIO(d)))
        assert frames[k].shape == pil.shape and np.array_equal(frames[k], pil), (k, pil.shape, int((frames[k] != pil).sum()))


@pytest.mark.gpu
def test_mutated_and_truncated_scans_follow_the_host_decoder(engine):
    rng = np.random.default_rng(21)
    lib = engine.lib
    src = scene(rng, 96, 128)
    bases = [jpeg(src, quality=q, subsampling=s, **kw) for q, s, kw in ((90, 2, {}), (50, 0, {}), (85, 2, {"restart_marker_blocks": 5}),
                                                                          (100, 1, {"restart_marker_rows": 1}))]
    datas = []
    for b in bases:
        scan_off = plan(lib, b)[1].scan_off
        for _ in range(12):  # byte mutations of the scan
            m = bytearray(b)
            for _ in range(int(rng.integers(1, 6))):
                m[int(rng.integers(scan_off, len(b) - 2))] = int(rng.choice([0x00, 0xFF, 0xD3, int(rng.integers(0, 256))]))
            datas.append(bytes(m))
        for f in (0.1, 0.5, 0.9, 0.999):  # truncated, EOI dropped
            datas.append(b[:scan_off + int((len(b) - 2 - scan_off) * f)])
        datas.append(b)
    st, coefs, _, _, _ = decode(engine, datas)
    n_bad = 0
    for k, d in enumerate(datas):
        rc, ref = host_coef(lib, d)
        assert st[k] == rc, (k, st[k], rc)
        if rc == 0:
            assert np.array_equal(coefs[k], ref), (k, int((coefs[k] != ref).sum()))
        n_bad += rc != 0
    assert 0 < n_bad < len(datas)
    good = [d for d in datas if host_coef(lib, d)[0] == 0]
    _, c2, f2, _, _ = decode(engine, good)  # the same files without their failing neighbours
    st3, c3, f3, _, _ = decode(engine, datas)
    j = 0
    for k, d in enumerate(datas):
        if st3[k] == 0:
            assert np.array_equal(c3[k], c2[j]) and np.array_equal(f3[k], f2[j])
            j += 1


@pytest.mark.gpu
def test_results_do_not_depend_on_the_batch_and_stay_in_their_regions(engine):
    datas = corpus()[::3]
    st, coefs, frames, _, _ = decode(engine, datas)
    assert not st.any()
    one = [decode(engine, [d]) for d in datas]
    perm = np.random.default_rng(4).permutation(len(datas))
    stp, cp, fp, _, _ = decode(engine, [datas[k] for k in perm])
    for k in range(len(datas)):
        assert np.array_equal(one[k][1][0], coefs[k]) and np.array_equal(one[k][2][0], frames[k])
    for j, k in enumerate(perm):
        assert np.array_equal(cp[j], coefs[k]) and np.array_equal(fp[j], frames[k])
    pad = 24
    st2, c2, f2, (ch, coff, clen), (oh, ooff, olen) = decode(engine, datas, pad=pad, sentinel=0x5A, chunk=5)
    assert not st2.any()
    for k in range(len(datas)):
        assert np.array_equal(c2[k], coefs[k]) and np.array_equal(f2[k], frames[k])
    inside_c, inside_o = np.zeros(ch.size, bool), np.zeros(oh.size, bool)
    for k in range(len(datas)):
        inside_c[coff[k]:coff[k] + clen[k]] = True
        inside_o[ooff[k]:ooff[k] + olen[k]] = True
    assert (ch[~inside_c] == 0x5A).all() and (oh[~inside_o] == 0x5A).all()


@pytest.mark.gpu
def test_camera_frames_match_the_eager_loader_and_chunking(engine, tmp_path, monkeypatch, loader_module):
    from msc_geom import engine as eng_mod
    from msc_geom import io as mio
    from msc_geom import ops
    from msc_geom.camera_agent import CameraAgent
    nuscenes_tree(tmp_path, n_samples=3)
    nl = loader_module
    eager = nl.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=1, engine=engine)
    lazy = nl.NuScenesLoader(str(tmp_path), "v1.0-mini", n_sweeps=1, lazy_sweeps=True)
    toks = eager.scene_sample_tokens(eager.get_scene_list()[0]["token"])
    ref = [eager.load_sample(t)["images"] for t in toks]
    samples = [lazy.load_sample(t) for t in toks]
    dev = ops.camera_frames(engine, samples)
    host = ops.camera_frames(engine, samples, to_host=True)
    assert all(f.is_cuda for fr in dev for f in fr)
    for r, d, h in zip(ref, dev, host):
        assert len(r) == len(d) == len(h) == 6
        assert all(np.array_equal(a, b.cpu().numpy()) and np.array_equal(a, c) for a, b, c in zip(r, d, h))
    # byte-budget chunking: one file per call gives the same frames
    staged = mio.stage_camera_files(samples)
    whole = engine.run_jpeg_decode(staged).to_host()
    monkeypatch.setattr(eng_mod, "JPEG_DECODE_WORKSPACE_PER_CALL", 1)
    assert len(engine._jpeg_decode_chunks(staged)) == len(staged)
    parts = engine.run_jpeg_decode(staged).to_host()
    assert all(np.array_equal(a, b) for a, b in zip(whole, parts))
    # device frames go straight into the camera agent and give the same strings as the PIL-decoded frames
    names = samples[0]["camera_names"]
    agent = CameraAgent(None, "m", "camera", engine=engine)
    pil = [np.array(Image.open(c["path"])) for c in samples[0]["cameras"]]
    assert agent.user_content(dev[0], names) == agent.user_content(pil, names)


@pytest.mark.gpu
def test_a_corrupt_file_raises_naming_it(engine, tmp_path):
    from msc_geom import io as mio
    rng = np.random.default_rng(9)
    good = jpeg(scene(rng, 64, 64), quality=90)
    scan_off = plan(engine.lib, good)[1].scan_off
    bad = good[:scan_off] + b"\xfe" * 200 + good[scan_off + 200:]  # a run of ones is no valid code
    assert host_coef(engine.lib, bad)[0] == _capi.MSC_ERR_BAD_ARGUMENT
    paths = []
    for k, d in enumerate((good, bad, good)):
        paths.append(str(tmp_path / f"f{k}.jpg"))
        open(paths[-1], "wb").write(d)
    res = engine.run_jpeg_decode(mio.stage_camera_files([{"cameras": [{"path": p} for p in paths]}]))
    with pytest.raises(_capi.MscError) as e:
        res.to_host()
    assert e.value.status == _capi.MSC_ERR_BAD_ARGUMENT and "file 1" in str(e.value)
    f = res.frames()
    assert np.array_equal(f[0].cpu().numpy(), np.array(Image.open(paths[0]))) and np.array_equal(f[2].cpu().numpy(), f[0].cpu().numpy())
