"""Row N8 on the device: vpk_decode_files (images.decode_files) bit for bit against the oracles on the JPEG, PNG and PGM
corpora mixed, damaged files in a mixed batch, vpk_prepare_files on gray photos bit for bit against
oracle/files_oracle.prepare_file, Pipeline.upload_files against upload_photos / upload_images on the oracle's planes,
bad input, and the VPK_PREP_CHECKS build on the gray cases."""
import os
import shutil
import subprocess
import sys

import cv2
import numpy as np
import pytest

from oracle import files_oracle as F
from oracle import jpeg_oracle as J
from oracle import png_oracle as G
from vanishing_points_2017_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gray_jpeg(img, quality=90):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, quality])
    assert ok
    return buf.tobytes()


def noise(seed, w, h):
    return np.random.RandomState(seed).randint(0, 256, (h, w)).astype(np.uint8)


def ties(w, h):
    """0 / 1 checkerboard: every 2 x 2 block sums to 2, a tie of the integer path"""
    return (np.indices((h, w)).sum(axis=0) % 2).astype(np.uint8)


def bits_with_two(w, h):
    b = ties(w, h)
    b[h // 2, w // 3] = 2
    return b


def mixed_corpus():
    files = ([(n, b) for n, b in J.corpus(large=False)] + [(n, b) for n, b in G.corpus(large=False)]
             + [(n, b) for n, b, _ in F.pgm_corpus()])
    order = np.random.RandomState(8).permutation(len(files))
    return [files[i] for i in order]


def test_decode_files_equals_the_oracles_on_the_mixed_corpora():
    from vanishing_points_2017_b200 import images
    corpus = mixed_corpus()
    blobs = [b for _, b in corpus]
    refs = [F.decode(b) for b in blobs]
    for (name, blob), ref in zip(corpus, refs):
        got, st = images.decode_files([blob])
        assert st.tolist() == [0], name
        assert got[0].shape == ref.shape, name
        np.testing.assert_array_equal(got[0], ref, err_msg=name)
    got, st = images.decode_files(blobs)
    assert st.tolist() == [0] * len(blobs)
    for (name, _), g, ref in zip(corpus, got, refs):
        np.testing.assert_array_equal(g, ref, err_msg="batch " + name)


def test_damaged_files_in_a_mixed_batch():
    from vanishing_points_2017_b200 import _lib, images
    good_j = J.encode_cv2(J.photo(3, 200, 150, texture=6.0))
    good = [good_j, G.encode_cv2(G.photo(4, 90, 70, texture=6)), F.write_pgm(F.gray_image(5, 77, 51)),
            gray_jpeg(F.gray_image(6, 64, 48)), G.encode_cv2(F.gray_image(7, 50, 40))]
    bad_j = [(n, b) for n, b in J.corrupted(good_j, 1) if n != "bitflip"]
    bad_p = G.corrupted()[:4]
    batch, expect = [], []
    for k, (name, blob) in enumerate(bad_j + bad_p):
        batch += [good[k % len(good)], blob]
        expect += [None, _lib.JPEG_CORRUPT if k < len(bad_j) else _lib.PNG_CORRUPT]
    batch.append(good[-1])
    expect.append(None)
    got, st = images.decode_files(batch)
    for i, e in enumerate(expect):
        if e is None:
            assert st[i] == 0, i
            np.testing.assert_array_equal(got[i], F.decode(batch[i]))
        else:
            assert st[i] == e, i
    again, st2 = images.decode_files(batch)
    assert st2.tolist() == st.tolist()
    for a, b in zip(got, again):
        np.testing.assert_array_equal(a, b)


# (id, gray image factory, target); sizes are w x h
GRAY_CASES = [("integer2_ties", lambda: ties(1280, 960), 640),
              ("integer2", lambda: noise(1, 1280, 960), 640),
              ("integer3", lambda: noise(2, 1920, 1440), 640),
              ("integer4", lambda: noise(3, 2560, 1920), 640),
              ("integer8", lambda: noise(4, 5120, 3840), 640),
              ("generic_640", lambda: F.gray_image(5, 2000, 1333), 640),
              ("generic_800", lambda: F.gray_image(6, 1333, 2000), 800),
              ("generic_noise", lambda: noise(7, 1700, 1100), 640),
              ("no_resize", lambda: F.gray_image(8, 700, 500), None),
              ("smaller_than_target", lambda: F.gray_image(9, 600, 400), 640),
              ("5000x3", lambda: noise(10, 5000, 3), 640),
              ("1x1", lambda: noise(11, 1, 1), 640),
              ("constant", lambda: np.full((900, 1300), 137, np.uint8), 640),
              ("zero", lambda: np.zeros((600, 900), np.uint8), 640),
              ("bits", lambda: ties(901, 601), 640),
              ("bits_with_two", lambda: bits_with_two(901, 601), 640),
              ("bits_no_resize", lambda: ties(64, 48), None)]


def gray_file(k, img):
    """a gray file of each kind in turn: PGM, 1-component JPEG, gray PNG; a 0 / 1 image always losslessly, so that
    the "* 255 if max <= 1" rule is what is tested"""
    if img.max() <= 2:
        return [F.write_pgm, G.encode_cv2][k % 2](img)
    return [F.write_pgm, gray_jpeg, G.encode_cv2][k % 3](img)


def check_gray(cases):
    from vanishing_points_2017_b200 import images
    for k, (name, make, target) in enumerate(cases):
        blob = gray_file(k, make())
        got = images.prepare_files([blob], target)[0]
        ref, _ = F.prepare_file(blob, target)
        assert got.dtype == np.uint8 and got.shape == ref.shape, name
        np.testing.assert_array_equal(got, ref, err_msg=name)


@pytest.mark.parametrize("name,make,target", GRAY_CASES, ids=[c[0] for c in GRAY_CASES])
def test_prepare_files_on_gray_photos_equals_the_oracle(name, make, target):
    check_gray([(name, make, target)])


@pytest.mark.parametrize("target", [None, 640, 800])
def test_prepare_files_on_a_mixed_batch(target):
    from vanishing_points_2017_b200 import images
    colour = [synth.render_photo(1, 150, 1200, 800), J.photo(2, 1000, 700, texture=6.0), synth.render_photo(3, 150, 640, 480)]
    blobs = [J.encode_cv2(colour[0], 95), gray_jpeg(F.gray_image(1, 1100, 900)), G.encode_cv2(colour[1]),
             F.write_pgm(F.gray_image(2, 1280, 960)), G.encode_cv2(F.gray_image(3, 900, 1300)), F.write_pgm(ties(800, 600)),
             G.encode_pil(colour[2])]
    got = images.prepare_files(blobs, target)
    for k, (blob, g) in enumerate(zip(blobs, got)):
        ref, _ = F.prepare_file(blob, target)
        assert g.dtype == ref.dtype and g.shape == ref.shape, k
        np.testing.assert_array_equal(g, ref, err_msg=str(k))
    dec = [F.decode(b) for b in blobs]
    col = [k for k, d in enumerate(dec) if d.ndim == 3]
    for k, g in zip(col, images.prepare_images([dec[k] for k in col], target)):
        np.testing.assert_array_equal(got[k], g)


def _pipe():
    from vanishing_points_2017_b200 import pipeline
    from vanishing_points_2017_b200 import cnn as vcnn
    ws, bs = vcnn.random_weights(0, scale=3.0)
    return pipeline.Pipeline(0, ws, bs, sphere_mode="votes")


def _rows(pipe, n):
    from vanishing_points_2017_b200 import _lib
    rows = np.empty((int(n), 7), np.float64)
    _lib.check(pipe.ctx.lib.vpk_lsd_fetch(pipe.ctx.h, _lib.ptr(rows)), "vpk_lsd_fetch")
    return rows


def _split_rows(rows, counts):
    off = np.concatenate([[0], np.cumsum(counts)])
    return [rows[off[k]:off[k + 1]] for k in range(len(counts))]


@pytest.mark.parametrize("target", [None, 640, 800])
def test_upload_files_equals_upload_photos_and_upload_images(target):
    pipe = _pipe()
    c = [synth.render_photo(20 + k, 220, w, h) for k, (w, h) in enumerate([(1200, 800), (800, 1100), (1000, 750)])]
    g = [(F.gray_image(30, 1000, 700) // 2 + synth.render_photo(31, 220, 1000, 700)[:, :, 1] // 2)]
    g.append(synth.render_photo(32, 220, 900, 1200)[:, :, 0])
    g.append(synth.render_photo(33, 220, 1100, 800)[:, :, 2])
    bits = (synth.render_photo(34, 220, 960, 720)[:, :, 1] > 128).astype(np.uint8)
    blobs = [J.encode_cv2(c[0], 95), F.write_pgm(g[0]), gray_jpeg(g[1], 95), G.encode_cv2(c[1]), G.encode_cv2(g[2]),
             F.write_pgm(bits), J.encode_cv2(c[2], 90, "444")]
    counts, shapes, status = pipe.upload_files(blobs, target)
    assert status.tolist() == [0] * len(blobs) and counts.sum() > 100
    rows = _split_rows(_rows(pipe, counts.sum()), counts)
    pipe.run()
    got = pipe.fetch()
    hz = pipe.horizons()
    dec = [F.decode(b) for b in blobs]
    prepared = [F.prepare_file(b, target) for b in blobs]
    assert shapes == [p.shape for p, _ in prepared]
    assert prepared[5][1].max() == 255.0                   # the 0 / 1 file: LSD sees it times 255
    col = [k for k, d in enumerate(dec) if d.ndim == 3]
    gray = [k for k, d in enumerate(dec) if d.ndim == 2]
    rc, rs = pipe.upload_photos([dec[k] for k in col], target)
    assert rs == [shapes[k] for k in col]
    for k, r in zip(col, _split_rows(_rows(pipe, rc.sum()), rc)):
        np.testing.assert_array_equal(rows[k], r, err_msg=str(k))
    rc = pipe.upload_images([prepared[k][1] for k in gray])
    for k, r in zip(gray, _split_rows(_rows(pipe, rc.sum()), rc)):
        np.testing.assert_array_equal(rows[k], r, err_msg=str(k))
    ref_counts = pipe.upload_images([p[1] for p in prepared])    # the whole batch, in input order
    np.testing.assert_array_equal(ref_counts, counts)
    pipe.run()
    ref = pipe.fetch()
    rhz = pipe.horizons()
    for a, b in zip(got, ref):
        assert (a["vp"] is None) == (b["vp"] is None)
        if a["vp"] is not None:
            np.testing.assert_array_equal(a["vp"], b["vp"])
            np.testing.assert_array_equal(a["vp_assoc"], b["vp_assoc"])
    for a, b in zip(hz, rhz):
        for q in range(6):
            np.testing.assert_array_equal(np.asarray(a[q]), np.asarray(b[q]))


def test_bad_input_raises_and_names_the_first_refused_file():
    from vanishing_points_2017_b200 import _lib, images
    pipe = _pipe()
    good = [F.write_pgm(F.gray_image(1, 120, 90)), J.encode_cv2(J.photo(2, 120, 90, texture=6.0))]
    refused = {n: b for n, b, _ in F.pgm_refused()}
    jref = {n: b for n, b, _ in J.refused()}
    pref = {n: b for n, b, _ in G.refused()}
    with pytest.raises(_lib.VpkError, match=r"file 2 \(PGM\) is not supported: reason 5 \(maxval"):
        images.decode_files(good + [refused["maxval_100"], refused["ascii_p2"]])
    with pytest.raises(_lib.VpkError, match=r"file 1 \(PGM\) .*reason 1 \(ASCII"):
        pipe.upload_files([good[0], refused["ascii_p2"]], 640)
    with pytest.raises(_lib.VpkError, match=r"file 0 \(JPEG\) .*reason 1 \(progressive"):
        images.prepare_files([jref["progressive_cv2"]] + good, 640)
    with pytest.raises(_lib.VpkError, match=r"file 1 \(PNG\) .*reason 2 \(16-bit"):
        pipe.upload_files([good[1], pref["depth16_rgb"]], 640)
    with pytest.raises(_lib.VpkError, match="file 2 is not supported: unknown format"):
        pipe.upload_files(good + [b"BM" + bytes(60)], 640)
    with pytest.raises(ValueError):
        pipe.upload_files([], 640)
    counts, shapes, st = pipe.upload_files(good, 640)      # the context still works
    assert st.tolist() == [0, 0] and shapes == [(90, 120), (90, 120)]
    np.testing.assert_array_equal(images.prepare_files(good[:1])[0], F.gray_image(1, 120, 90))


def test_gray_files_are_still_refused_by_the_single_format_uploads():
    from vanishing_points_2017_b200 import _lib
    pipe = _pipe()
    with pytest.raises(_lib.VpkError, match="gray"):
        pipe.upload_jpegs([gray_jpeg(F.gray_image(1, 120, 90))], 640)
    with pytest.raises(_lib.VpkError, match="gray"):
        pipe.upload_pngs([G.encode_cv2(F.gray_image(1, 120, 90))], 640)


def test_checked_build_runs_the_gray_cases(tmp_path):
    """A VPK_DEFINES=VPK_PREP_CHECKS copy of the library (every shared- and global-memory index of image_prep and
    prep_gray_scale asserted) runs the gray cases without an assert firing."""
    tree = str(tmp_path / "tree")
    pkg = os.path.join(tree, "vanishing_points_2017_b200")
    shutil.copytree(os.path.join(ROOT, "vanishing_points_2017_b200"), pkg,
                    ignore=shutil.ignore_patterns("_obj", "*.so", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    env = dict(os.environ, VPK_DEFINES="VPK_PREP_CHECKS", PYTHONPATH=os.pathsep.join([tree, ROOT]))
    subprocess.check_call([sys.executable, "-m", "vanishing_points_2017_b200.build"], env=env, cwd=tree)
    code = ("import vanishing_points_2017_b200 as v, sys; assert v.__file__.startswith(%r), v.__file__; "
            "sys.path.insert(0, %r); import test_files_gpu as t; t.check_gray(t.GRAY_CASES); "
            "t.test_upload_files_equals_upload_photos_and_upload_images(640); print('checked ok')"
            % (tree, os.path.join(ROOT, "tests")))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=tree, capture_output=True, text=True)
    assert out.returncode == 0 and "checked ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
