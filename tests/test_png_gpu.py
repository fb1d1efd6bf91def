"""Row N7 on the device: vpk_decode_pngs (images.decode_pngs) bit for bit against libpng on the corpus of
oracle/png_oracle.py, one file per call and as one batch; damaged files in a batch; data after the last row;
Pipeline.upload_pngs against Pipeline.upload_photos on the oracle's decode; bad input; the VPK_PNG_CHECKS build."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from oracle import png_oracle as P

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CORPUS = P.corpus(large=True)


def check_corpus(corpus, batch=True):
    from vanishing_points_2017_b200 import images
    blobs = [b for _, b in corpus]
    refs = [P.decode(b) for b in blobs]
    for (name, blob), ref in zip(corpus, refs):
        got, st = images.decode_pngs([blob])
        assert st.tolist() == [0], name
        assert got[0].shape == ref.shape, name
        np.testing.assert_array_equal(got[0], ref, err_msg=name)
    if batch:
        got, st = images.decode_pngs(blobs)
        assert st.tolist() == [0] * len(blobs)
        for (name, _), g, ref in zip(corpus, got, refs):
            np.testing.assert_array_equal(g, ref, err_msg="batch " + name)


def test_decode_equals_libpng_bit_for_bit():
    check_corpus(CORPUS)


def test_damaged_files_are_flagged_and_do_not_touch_the_others():
    from vanishing_points_2017_b200 import images
    good = [P.write(P.samples(60 + k, 90, 70, t, 8), t, 8, interlace=k % 2) for k, t in enumerate((2, 6, 2, 6))]
    refs = [P.decode(b) for b in good]
    bad = P.corrupted()
    batch, where = [], []
    for k, (name, blob) in enumerate(bad):
        batch.append(good[k % len(good)])
        where.append(None)
        batch.append(blob)
        where.append(name)
    batch.append(good[0])
    where.append(None)
    got, st = images.decode_pngs(batch)
    for i, name in enumerate(where):
        if name is None:
            assert st[i] == 0, i
            np.testing.assert_array_equal(got[i], P.decode(batch[i]))
        else:
            assert st[i] == P.CORRUPT, name
    again, st2 = images.decode_pngs(batch)              # deterministic, damaged files included
    assert st2.tolist() == st.tolist()
    for a, b in zip(got, again):
        np.testing.assert_array_equal(a, b)
    assert len(refs) == 4


def test_extra_data_after_the_last_row_decodes():
    from vanishing_points_2017_b200 import images
    files = P.extra_data()
    got, st = images.decode_pngs([b for _, b, _ in files])
    assert st.tolist() == [0] * len(files)
    for (name, blob, exp), g in zip(files, got):
        np.testing.assert_array_equal(g, P.decode(blob), err_msg=name)
        np.testing.assert_array_equal(g, exp, err_msg=name)


def _pipe():
    from vanishing_points_2017_b200 import pipeline
    from vanishing_points_2017_b200 import cnn as vcnn
    ws, bs = vcnn.random_weights(0, scale=3.0)
    return pipeline.Pipeline(0, ws, bs, sphere_mode="votes")


@pytest.mark.parametrize("target", [640, 800])
def test_upload_pngs_equals_upload_photos_on_the_oracle_decode(target):
    from vanishing_points_2017_b200 import _lib
    pipe = _pipe()
    img = [P.photo(70 + k, w, h, texture=6) for k, (w, h) in enumerate([(2000, 1333), (1333, 2000), (1200, 800), (640, 480)])]
    pal = P.encode_pil(P.Image.fromarray(img[3]).quantize(200), optimize=True)
    blobs = [P.encode_cv2(img[0]), P.encode_pil(np.dstack([img[1], img[1][:, :, :1]])), P.encode_cv2(img[2], 9), pal]
    counts, shapes, status = pipe.upload_pngs(blobs, target)
    assert status.tolist() == [0] * len(blobs) and counts.sum() > 100
    rows = np.empty((int(counts.sum()), 7), np.float64)
    _lib.check(pipe.ctx.lib.vpk_lsd_fetch(pipe.ctx.h, _lib.ptr(rows)), "vpk_lsd_fetch")
    pipe.run()
    got = pipe.fetch()
    hz = pipe.horizons()
    rc, rs = pipe.upload_photos([P.decode(b) for b in blobs], target)
    np.testing.assert_array_equal(counts, rc)
    assert shapes == rs
    ref_rows = np.empty_like(rows)
    _lib.check(pipe.ctx.lib.vpk_lsd_fetch(pipe.ctx.h, _lib.ptr(ref_rows)), "vpk_lsd_fetch")
    np.testing.assert_array_equal(rows, ref_rows)
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


def test_bad_input_raises():
    from vanishing_points_2017_b200 import _lib, images
    pipe = _pipe()
    good = P.encode_cv2(P.photo(1, 120, 90, texture=6))
    refused = dict((n, b) for n, b, _ in P.refused())
    gray = P.encode_cv2(P.photo(2, 120, 90, texture=6)[:, :, 0])
    with pytest.raises(_lib.VpkError, match="file 1 .*depth"):
        images.decode_pngs([good, refused["depth16_rgb"]])
    with pytest.raises(_lib.VpkError, match="file 1 .*not png"):
        images.decode_pngs([good, refused["jpeg"]])
    with pytest.raises(_lib.VpkError, match="photo 1 is not supported: reason 2"):
        pipe.upload_pngs([good, refused["depth16_rgb"]], 640)
    with pytest.raises(_lib.VpkError, match="photo 2 is gray"):
        pipe.upload_pngs([good, good, gray], 640)
    with pytest.raises(ValueError):
        pipe.upload_pngs([], 640)
    got, st = images.decode_pngs([gray, good])          # gray files decode; they just cannot be prepared
    np.testing.assert_array_equal(got[0], P.decode(gray))
    np.testing.assert_array_equal(got[1], P.decode(good))
    counts, _, st = pipe.upload_pngs([good], 640)       # the context still works
    assert st.tolist() == [0]


def test_checked_build_runs_the_bit_equality_corpus(tmp_path):
    """A VPK_DEFINES=VPK_PNG_CHECKS copy of the library (every index into the files, tables, scanline buffers and
    outputs asserted) decodes the corpus, one file per call, without an assert firing."""
    tree = str(tmp_path / "tree")
    pkg = os.path.join(tree, "vanishing_points_2017_b200")
    shutil.copytree(os.path.join(ROOT, "vanishing_points_2017_b200"), pkg,
                    ignore=shutil.ignore_patterns("_obj", "*.so", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    env = dict(os.environ, VPK_DEFINES="VPK_PNG_CHECKS", PYTHONPATH=os.pathsep.join([tree, ROOT]))
    subprocess.check_call([sys.executable, "-m", "vanishing_points_2017_b200.build"], env=env, cwd=tree)
    code = ("import vanishing_points_2017_b200 as v, sys; assert v.__file__.startswith(%r), v.__file__; "
            "sys.path.insert(0, %r); import test_png_gpu as t; t.check_corpus(t.CORPUS, batch=False); print('checked ok')"
            % (tree, os.path.join(ROOT, "tests")))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=tree, capture_output=True, text=True)
    assert out.returncode == 0 and "checked ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
