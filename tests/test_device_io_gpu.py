"""Row N9 on the device: Pipeline.upload_photos / upload_images / upload from torch CUDA tensors (HWC, CHW views, crops,
gray photos, strided planes, column slices) bit for bit against the host routes on the same pixels, fetch(device=True)
and horizons(device=True) against fetch() / horizons(), ordering behind work queued on a side stream, bad input, the
VPK_PACK_CHECKS build on the strided cases, and nvJPEG output of a progressive JPEG fed to upload_photos."""
import functools
import io
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import files_oracle as F  # noqa: E402
from oracle import png_oracle as G  # noqa: E402
from vanishing_points_2017_b200 import synth  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda", 0)


def _pipe():
    from vanishing_points_2017_b200 import pipeline
    from vanishing_points_2017_b200 import cnn as vcnn
    ws, bs = vcnn.random_weights(0, scale=3.0)
    return pipeline.Pipeline(0, ws, bs, sphere_mode="votes")


def _rows(pipe, counts):
    from vanishing_points_2017_b200 import _lib
    rows = np.empty((int(np.sum(counts)), 7), np.float64)
    _lib.check(pipe.ctx.lib.vpk_lsd_fetch(pipe.ctx.h, _lib.ptr(rows)), "vpk_lsd_fetch")
    off = np.concatenate([[0], np.cumsum(counts)])
    return [rows[off[k]:off[k + 1]] for k in range(len(counts))]


def _same_results(a, b):
    for x, y in zip(a, b):
        assert (x["vp"] is None) == (y["vp"] is None)
        if x["vp"] is not None:
            for k in ("vp", "vp_assoc", "counts", "sigma", "counts_weighted"):
                np.testing.assert_array_equal(x[k], y[k], err_msg=k)


def _same_horizons(a, b):
    for x, y in zip(a, b):
        for q in range(6):
            np.testing.assert_array_equal(np.asarray(x[q]), np.asarray(y[q]))


@functools.lru_cache(None)
def photo_cases():
    """(name, device tensor view, the same pixels as a contiguous host array).  The views are made from tensors that
    stay alive in the cache."""
    rs = np.random.RandomState(5)
    keep, cases = [], []

    def add(name, t, host):
        keep.append(t)
        cases.append((name, t, np.ascontiguousarray(host)))

    p = synth.render_photo(50, 220, 1200, 800)
    add("hwc", torch.from_numpy(p).to(DEV), p)
    p = synth.render_photo(51, 220, 801, 1101)                      # odd sides: rows of 2403 bytes
    add("hwc_odd", torch.from_numpy(p).to(DEV), p)
    p = synth.render_photo(52, 220, 1000, 750)
    chw = torch.from_numpy(p).permute(2, 0, 1).contiguous().to(DEV)
    add("chw_view", chw.permute(1, 2, 0), p)
    big = synth.render_photo(53, 220, 1337, 1001)
    add("crop", torch.from_numpy(big).to(DEV)[37:37 + 900, 101:101 + 1100], big[37:37 + 900, 101:101 + 1100])
    bigc = torch.from_numpy(big).permute(2, 0, 1).contiguous().to(DEV)
    add("chw_crop", bigc[:, 5:5 + 640, 3:3 + 961].permute(1, 2, 0), big[5:5 + 640, 3:3 + 961])
    g = F.gray_image(54, 1000, 700) // 2 + synth.render_photo(55, 220, 1000, 700)[:, :, 1] // 2
    add("gray", torch.from_numpy(g).to(DEV), g)
    g2 = synth.render_photo(56, 220, 1203, 905)[:, :, 0]
    add("gray_crop", torch.from_numpy(g2).to(DEV)[3:3 + 880, 1:1 + 1170], g2[3:3 + 880, 1:1 + 1170])
    bits = (synth.render_photo(57, 220, 960, 720)[:, :, 1] > 128).astype(np.uint8)   # LSD sees it times 255
    add("gray_bits", torch.from_numpy(bits).to(DEV), bits)
    one = rs.randint(0, 256, (1, 1, 3)).astype(np.uint8)
    add("1x1", torch.from_numpy(one).to(DEV), one)
    huge = synth.render_photo(58, 400, 6000, 4000)
    add("6000x4000", torch.from_numpy(huge).to(DEV), huge)
    return cases, keep


@functools.lru_cache(None)
def as_file(k):
    """photo case k as the file upload_files prepares the same way: lossless PNG for colour, PGM for gray"""
    host = photo_cases()[0][k][2]
    return G.encode_cv2(host, 0) if host.ndim == 3 else F.write_pgm(host)      # stored deflate blocks: quick both ways


def check_photos(target, names=None):
    cases, _ = photo_cases()
    idx = [k for k, c in enumerate(cases) if names is None or c[0] in names]
    pipe = _pipe()
    counts, shapes = pipe.upload_photos([cases[k][1] for k in idx], target)
    rows = _rows(pipe, counts)
    pipe.run()
    got, hz = pipe.fetch(), pipe.horizons()
    # colour photos: the host upload_photos on the same pixels; gray ones: upload_files on PGM files of them
    col = [j for j, k in enumerate(idx) if cases[k][2].ndim == 3]
    gray = [j for j, k in enumerate(idx) if cases[k][2].ndim == 2]
    if col:
        rc, rs = pipe.upload_photos([cases[idx[j]][2] for j in col], target)
        assert rs == [shapes[j] for j in col]
        for j, r in zip(col, _rows(pipe, rc)):
            np.testing.assert_array_equal(rows[j], r, err_msg=cases[idx[j]][0])
    if gray:
        rc, rs, _ = pipe.upload_files([as_file(idx[j]) for j in gray], target)
        assert rs == [shapes[j] for j in gray]
        for j, r in zip(gray, _rows(pipe, rc)):
            np.testing.assert_array_equal(rows[j], r, err_msg=cases[idx[j]][0])
    # the whole batch, in input order, through the run
    ref_counts, ref_shapes, _ = pipe.upload_files([as_file(k) for k in idx], target)
    np.testing.assert_array_equal(ref_counts, counts)
    assert ref_shapes == shapes
    pipe.run()
    _same_results(got, pipe.fetch())
    _same_horizons(hz, pipe.horizons())
    return counts


@pytest.mark.parametrize("target", [None, 640, 800])
def test_upload_photos_from_device_tensors_equals_the_host_routes(target):
    counts = check_photos(target)
    assert counts.sum() > 100


def test_upload_photos_in_one_batch_with_repeated_views():
    """the same device memory twice (a photo and its crop) and a photo written twice into the batch"""
    cases, _ = photo_cases()
    t, host = cases[0][1], cases[0][2]
    pipe = _pipe()
    c1, s1 = pipe.upload_photos([t, t[100:500, 200:900], t], 640)
    r1 = _rows(pipe, c1)
    c2, s2 = pipe.upload_photos([host, np.ascontiguousarray(host[100:500, 200:900]), host], 640)
    assert s1 == s2 and c1.tolist() == c2.tolist()
    for a, b in zip(r1, _rows(pipe, c2)):
        np.testing.assert_array_equal(a, b)


def plane_cases(dtype):
    g = synth.render_photo(60, 220, 1300, 900)[:, :, 1]
    h = synth.render_photo(61, 220, 700, 1000)[:, :, 0]
    if dtype == "f64":
        g, h = g.astype(np.float64) * 0.75, h.astype(np.float64) + 0.25
    tg, th = torch.from_numpy(g).to(DEV), torch.from_numpy(h).to(DEV)
    return [(tg, g), (th[::2, ::3], h[::2, ::3]), (tg.t(), g.T), (tg[10:810, 7:1207], g[10:810, 7:1207])], (tg, th)


@pytest.mark.parametrize("dtype", ["u8", "f64"])
def test_upload_images_from_device_planes_equals_upload_images(dtype):
    cases, _ = plane_cases(dtype)
    pipe = _pipe()
    counts = pipe.upload_images([t for t, _ in cases])
    rows = _rows(pipe, counts)
    pipe.run()
    got = pipe.fetch()
    ref = pipe.upload_images([np.ascontiguousarray(h) for _, h in cases])
    np.testing.assert_array_equal(ref, counts)
    for a, b in zip(rows, _rows(pipe, ref)):
        np.testing.assert_array_equal(a, b)
    pipe.run()
    _same_results(got, pipe.fetch())


def segment_batch():
    ns = [90, 150, 0, 220, 75]
    seg = np.concatenate([synth.make_scene(4300 + k, n)["segments"] if n else np.zeros((0, 4)) for k, n in enumerate(ns)])
    off = np.concatenate([[0], np.cumsum(ns)]).astype(np.int32)
    return seg, off


def test_upload_from_device_segments_equals_upload():
    seg, off = segment_batch()
    pipe = _pipe()
    pipe.upload(seg, off)
    pipe.run()
    ref, ref_sig, ref_sph = pipe.fetch(want_response=True, want_sphere=True)
    ref_hz = pipe.horizons()
    wide = torch.zeros((seg.shape[0], 7), dtype=torch.float64, device=DEV)
    wide[:, 2:6] = torch.from_numpy(seg).to(DEV)
    for name, t, o in [("contiguous", torch.from_numpy(seg).to(DEV), off),
                       ("column_slice", wide[:, 2:6], off),
                       ("device_offsets", wide[:, 2:6], torch.from_numpy(off.astype(np.int64)).to(DEV))]:
        pipe.upload(t, o)
        pipe.run()
        got, sig, sph = pipe.fetch(want_response=True, want_sphere=True)
        _same_results(got, ref)
        np.testing.assert_array_equal(sig, ref_sig, err_msg=name)
        np.testing.assert_array_equal(sph, ref_sph, err_msg=name)
        _same_horizons(pipe.horizons(), ref_hz)


def test_fetch_and_horizons_on_the_device_equal_the_host_copies():
    from vanishing_points_2017_b200 import pipeline as P
    seg, off = segment_batch()
    pipe = _pipe()
    pipe.upload(seg, off)
    pipe.run()
    raw, sig, sph = pipe.fetch(raw=True, want_response=True, want_sphere=True)
    d, dsig, dsph = pipe.fetch(device=True, want_response=True, want_sphere=True)
    only = pipe.fetch(device=True)
    for k in P.RAW_PER_IMAGE + ("vp_assoc",):
        assert d[k].is_cuda and d[k].device == DEV
        np.testing.assert_array_equal(d[k].cpu().numpy(), raw[k], err_msg=k)
        np.testing.assert_array_equal(only[k].cpu().numpy(), raw[k], err_msg=k)
    np.testing.assert_array_equal(dsig.cpu().numpy(), sig)
    np.testing.assert_array_equal(dsph.cpu().numpy(), sph)
    B = len(off) - 1
    th = np.stack([np.array([0.01 * k, 1.0, -0.1 + 0.03 * k]) for k in range(B)])
    sc, hh = np.linspace(1.0, 2.0, B), np.full(B, 480.0)
    hz, err = pipe.horizons(true_horizons=th, scales=sc, image_heights=hh)
    for truth in [(th, sc, hh), (torch.from_numpy(th).to(DEV), torch.from_numpy(sc).to(DEV), 480.0)]:
        pts, combo, derr = pipe.horizons(device=True, true_horizons=truth[0], scales=truth[1], image_heights=truth[2])
        np.testing.assert_array_equal(derr.cpu().numpy(), err)
        for b in range(B):
            for q in range(5):
                np.testing.assert_array_equal(pts[b, q].cpu().numpy(), hz[b][q])
            k = len(hz[b][5])
            np.testing.assert_array_equal(combo[b, :k].cpu().numpy(), hz[b][5])
    pts, combo, none = pipe.horizons(device=True)
    assert none is None and pts.shape == (B, 5, 3) and combo.dtype == torch.int32


def test_ordering_after_work_queued_on_a_side_stream():
    """Inputs are written on a side stream behind a long kernel and the calls get that stream without a host
    synchronisation; the device outputs are consumed on it right after the call."""
    cases, _ = photo_cases()
    sel = [c for c in cases if c[0] in ("hwc", "chw_view", "crop", "gray")]
    seg, off = segment_batch()
    pipe = _pipe()
    ref_counts, ref_shapes = pipe.upload_photos([np.ascontiguousarray(h) for _, _, h in sel[:3]], 640)
    ref_rows = _rows(pipe, ref_counts)
    pipe.upload(seg, off)
    pipe.run()
    ref = pipe.fetch(raw=True)
    side = torch.cuda.Stream(DEV)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        dst = [torch.empty_like(t) for _, t, _ in sel[:3]]          # filled behind the sleep
        for d, (_, t, _) in zip(dst, sel[:3]):
            d.copy_(t)
    counts, shapes = pipe.upload_photos([dst[0], dst[1], dst[2]], 640, stream=side)
    assert shapes == ref_shapes and counts.tolist() == ref_counts.tolist()
    for a, b in zip(_rows(pipe, counts), ref_rows):
        np.testing.assert_array_equal(a, b)
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        dseg = torch.from_numpy(seg).to(DEV, non_blocking=False) * 1.0
    pipe.upload(dseg, off, stream=side)
    pipe.run()
    with torch.cuda.stream(side):
        torch.cuda._sleep(100_000_000)
    out = pipe.fetch(device=True, stream=side)
    with torch.cuda.stream(side):
        vp = out["vp"] * 1.0                                          # consumed on the stream right after the call
        assoc = out["vp_assoc"] + 0
    side.synchronize()
    np.testing.assert_array_equal(vp.cpu().numpy(), ref["vp"])
    np.testing.assert_array_equal(assoc.cpu().numpy(), ref["vp_assoc"])


def test_bad_input_is_refused_before_any_device_work():
    import ctypes as C
    from vanishing_points_2017_b200 import _lib
    pipe = _pipe()
    good = torch.from_numpy(synth.render_photo(70, 100, 320, 240)).to(DEV)
    host = np.zeros((240, 320, 3), np.uint8)

    class HostCAI:                                    # claims CUDA memory but points at host memory
        __cuda_array_interface__ = dict(shape=(240, 320, 3), typestr="|u1", strides=None, data=(host.ctypes.data, False), version=2)

    with pytest.raises(_lib.VpkError, match=r"photo 1 is host memory.*vpk_pipeline_upload_photos"):
        pipe.upload_photos([good, HostCAI()], 640)
    pinned = torch.zeros((240, 320, 3), dtype=torch.uint8).pin_memory()

    class PinnedCAI:
        __cuda_array_interface__ = dict(shape=(240, 320, 3), typestr="|u1", strides=None, data=(pinned.data_ptr(), False), version=2)

    with pytest.raises(_lib.VpkError, match="photo 0 is host memory"):
        pipe.upload_photos([PinnedCAI()], 640)
    # the C entry points refuse negative strides, a bad dtype, zero sizes and 2 or 4 channels
    lib, h = pipe.ctx.lib, pipe.ctx.h
    ptrs = (C.c_void_p * 1)(good.data_ptr())
    w, hh = np.array([320], np.int32), np.array([240], np.int32)
    cfg = _lib.lsd_config()
    counts = np.empty(1, np.int32)
    for strides, ch, width, match in [((960, -3, 1), 3, w, "negative stride"), ((960, 3, 1), 2, w, "2 channels"),
                                      ((960, 3, 1), 4, w, "4 channels"), ((960, 3, 1), 3, np.array([0], np.int32), "size 0 x 240")]:
        s = np.array(strides, np.int64)
        c = np.array([ch], np.int32)
        with pytest.raises(_lib.VpkError, match=match):
            _lib.check(lib.vpk_pipeline_upload_photos_device(h, ptrs, _lib.ptr(s), _lib.ptr(width), _lib.ptr(hh), _lib.ptr(c), 1, 640,
                                                             C.byref(cfg), 0, _lib.ptr(counts), None, None), "upload_photos_device")
    s = np.array([320, 1], np.int64)
    plane = good[:, :, 0].contiguous()
    pp = (C.c_void_p * 1)(plane.data_ptr())
    with pytest.raises(_lib.VpkError, match="dtype"):
        _lib.check(lib.vpk_pipeline_upload_images_device(h, pp, _lib.ptr(s), _lib.ptr(w), _lib.ptr(hh), 1, 7, C.byref(cfg), 0,
                                                         _lib.ptr(counts)), "upload_images_device")
    hp = (C.c_void_p * 1)(host.ctypes.data)
    with pytest.raises(_lib.VpkError, match="image 0 is host memory.*vpk_pipeline_upload_images"):
        _lib.check(lib.vpk_pipeline_upload_images_device(h, hp, _lib.ptr(s), _lib.ptr(w), _lib.ptr(hh), 1, _lib.PIX_U8, C.byref(cfg), 0,
                                                         _lib.ptr(counts)), "upload_images_device")
    off = np.array([0, 10], np.int32)
    seg_host = np.zeros((10, 4))
    with pytest.raises(_lib.VpkError, match="segments is host memory.*vpk_pipeline_upload"):
        _lib.check(lib.vpk_pipeline_upload_device(h, seg_host.ctypes.data, 4, 1, _lib.ptr(off), 1, 0), "upload_device")
    seg_dev = torch.zeros((10, 4), dtype=torch.float64, device=DEV)
    with pytest.raises(_lib.VpkError, match="negative stride"):
        _lib.check(lib.vpk_pipeline_upload_device(h, seg_dev.data_ptr(), -4, 1, _lib.ptr(off), 1, 0), "upload_device")
    # and in Python: wrong dtypes, ranks and channel counts, mixed host and device lists
    with pytest.raises(ValueError, match="type"):
        pipe.upload_photos([good.float()], 640)
    with pytest.raises(ValueError, match="channels"):
        pipe.upload_photos([torch.zeros((20, 30, 4), dtype=torch.uint8, device=DEV)], 640)
    with pytest.raises(ValueError, match="all in CUDA memory"):
        pipe.upload_photos([good, host], 640)
    with pytest.raises(ValueError, match="all uint8 or all float64"):
        pipe.upload_images([plane, plane.double()])
    with pytest.raises(ValueError, match="type"):
        pipe.upload(seg_dev.float(), off)
    # results into host memory are refused too
    pipe.upload(seg_dev, off)
    pipe.run()
    bad = np.zeros(64, np.int32)
    res = _lib.EmResult(*([bad.ctypes.data] * 8 + [None]))
    with pytest.raises(_lib.VpkError, match="status is host memory.*vpk_pipeline_fetch"):
        _lib.check(lib.vpk_pipeline_fetch_device(h, C.byref(res), None, None, 0), "fetch_device")
    pts = np.zeros((1, 5, 3))
    with pytest.raises(_lib.VpkError, match="points is host memory"):
        _lib.check(lib.vpk_pipeline_horizon_device(h, 10, 0.3, 0.7, None, None, None, pts.ctypes.data, bad.ctypes.data, None, 0),
                   "horizon_device")
    # the context still works
    counts, shapes = pipe.upload_photos([good], 640)
    assert shapes == [(240, 320)]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs a second GPU")
def test_a_tensor_on_another_device_is_refused():
    from vanishing_points_2017_b200 import _lib
    pipe = _pipe()
    other = torch.zeros((240, 320, 3), dtype=torch.uint8, device="cuda:1")
    with pytest.raises(_lib.VpkError, match="photo 0 is memory of device 1"):
        pipe.upload_photos([other], 640)


def test_progressive_jpeg_decoded_by_nvjpeg():
    """A progressive JPEG (which the decoder here refuses) decoded on the GPU by torchvision, fed to upload_photos as
    a device tensor: the same as the host upload_photos on the decoded pixels copied to the host."""
    tv = pytest.importorskip("torchvision")
    from PIL import Image
    photo = synth.render_photo(80, 220, 1024, 683)
    buf = io.BytesIO()
    Image.fromarray(photo).save(buf, format="JPEG", quality=90, progressive=True)
    data = torch.frombuffer(bytearray(buf.getvalue()), dtype=torch.uint8)
    try:
        chw = tv.io.decode_jpeg(data, device="cuda")
    except Exception as e:   # a torchvision without the GPU decoder
        pytest.skip("torchvision.io.decode_jpeg(device='cuda') is not available: %s" % e)
    assert chw.is_cuda and chw.shape == (3, 683, 1024)
    pipe = _pipe()
    counts, shapes = pipe.upload_photos([chw.permute(1, 2, 0)], 640)
    rows = _rows(pipe, counts)
    pipe.run()
    got = pipe.fetch()
    ref_counts, ref_shapes = pipe.upload_photos([chw.permute(1, 2, 0).cpu().numpy()], 640)
    assert shapes == ref_shapes and counts.tolist() == ref_counts.tolist() and counts.sum() > 10
    np.testing.assert_array_equal(rows[0], _rows(pipe, ref_counts)[0])
    pipe.run()
    _same_results(got, pipe.fetch())


def test_checked_build_runs_the_strided_cases(tmp_path):
    """A VPK_DEFINES=VPK_PACK_CHECKS copy of the library (every source and destination index of device_pack asserted)
    runs the photo, plane and segment cases without an assert firing."""
    tree = str(tmp_path / "tree")
    pkg = os.path.join(tree, "vanishing_points_2017_b200")
    shutil.copytree(os.path.join(ROOT, "vanishing_points_2017_b200"), pkg,
                    ignore=shutil.ignore_patterns("_obj", "*.so", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    env = dict(os.environ, VPK_DEFINES="VPK_PACK_CHECKS", PYTHONPATH=os.pathsep.join([tree, ROOT]))
    subprocess.check_call([sys.executable, "-m", "vanishing_points_2017_b200.build"], env=env, cwd=tree)
    code = ("import vanishing_points_2017_b200 as v, sys; assert v.__file__.startswith(%r), v.__file__; "
            "sys.path.insert(0, %r); import test_device_io_gpu as t; "
            "t.check_photos(800, ('hwc', 'hwc_odd', 'chw_view', 'crop', 'chw_crop', 'gray_crop', '1x1')); "
            "t.test_upload_images_from_device_planes_equals_upload_images('u8'); "
            "t.test_upload_images_from_device_planes_equals_upload_images('f64'); "
            "t.test_upload_from_device_segments_equals_upload(); print('checked ok')"
            % (tree, os.path.join(ROOT, "tests")))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=tree, capture_output=True, text=True)
    assert out.returncode == 0 and "checked ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
