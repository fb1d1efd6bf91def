"""Row N6 on the device: vpk_decode_jpegs (images.decode_jpegs) bit for bit against libjpeg-turbo on the corpus of
oracle/jpeg_oracle.py, one file per call and as one batch, at several subsequence lengths; damaged files in a batch;
Pipeline.upload_jpegs against Pipeline.upload_photos on the oracle's decode; bad input; the VPK_JPEG_CHECKS build."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from oracle import jpeg_oracle as J

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CORPUS = J.corpus(large=True)


def check_corpus(corpus, batch=True):
    from vanishing_points_2017_b200 import images
    blobs = [b for _, b in corpus]
    refs = [J.decode(b) for b in blobs]
    for (name, blob), ref in zip(corpus, refs):
        got, st = images.decode_jpegs([blob])
        assert st.tolist() == [0], name
        assert got[0].shape == ref.shape, name
        np.testing.assert_array_equal(got[0], ref, err_msg=name)
    if batch:
        got, st = images.decode_jpegs(blobs)
        assert st.tolist() == [0] * len(blobs)
        for (name, _), g, ref in zip(corpus, got, refs):
            np.testing.assert_array_equal(g, ref, err_msg="batch " + name)


def test_decode_equals_libjpeg_turbo_bit_for_bit():
    check_corpus(CORPUS)


@pytest.mark.parametrize("bits", [32, 256])
def test_subsequence_length_does_not_change_the_output(bits):
    from vanishing_points_2017_b200 import images
    small = [b for n, b in CORPUS if "6000x4000" not in n]
    ref, st0 = images.decode_jpegs(small)
    os.environ["VPK_JPEG_SUBSEQ_BITS"] = str(bits)
    try:
        got, st = images.decode_jpegs(small)
        stats = images.jpeg_stats()
    finally:
        del os.environ["VPK_JPEG_SUBSEQ_BITS"]
    assert st.tolist() == st0.tolist() == [0] * len(small)
    for a, b in zip(got, ref):
        np.testing.assert_array_equal(a, b)
    assert stats["subsequences"] > len(small)


def test_sync_statistics_when_profiling():
    from vanishing_points_2017_b200 import _lib, images
    ctx = _lib.default_context()
    blob = J.encode_cv2(J.noise(3, 640, 480), 100, "420")
    os.environ["VPK_JPEG_SUBSEQ_BITS"] = "32"
    ctx.profile_enable(True)
    try:
        got, st = images.decode_jpegs([blob])
        stats = images.jpeg_stats()
    finally:
        ctx.profile_enable(False)
        del os.environ["VPK_JPEG_SUBSEQ_BITS"]
    np.testing.assert_array_equal(got[0], J.decode(blob))
    assert stats["subsequences"] > 10000 and stats["redecoded"] > 0 and stats["max_rounds"] >= 1


def test_corrupt_files_are_flagged_and_do_not_touch_the_others():
    from vanishing_points_2017_b200 import images
    good = [J.encode_cv2(J.photo(40 + k, 300, 200, texture=8), 90, "420", restart=k) for k in range(3)]
    refs = [J.decode(b) for b in good]
    bad = [b for _, b in J.corrupted(good[0], 1) if _ != "bitflip"]
    batch = [good[0], bad[0], good[1], bad[1], good[2]]
    got, st = images.decode_jpegs(batch)
    assert st.tolist() == [0, J.CORRUPT, 0, J.CORRUPT, 0]
    for i, ref in zip((0, 2, 4), refs):
        np.testing.assert_array_equal(got[i], ref)
    again, st2 = images.decode_jpegs(batch)             # deterministic, corrupt photos included
    assert st2.tolist() == st.tolist()
    for a, b in zip(got, again):
        np.testing.assert_array_equal(a, b)


def _pipe():
    from vanishing_points_2017_b200 import pipeline
    from vanishing_points_2017_b200 import cnn as vcnn
    ws, bs = vcnn.random_weights(0, scale=3.0)
    return pipeline.Pipeline(0, ws, bs, sphere_mode="votes")


@pytest.mark.parametrize("target", [640, 800])
def test_upload_jpegs_equals_upload_photos_on_the_oracle_decode(target):
    from vanishing_points_2017_b200 import _lib
    pipe = _pipe()
    blobs = [J.encode_cv2(J.photo(60 + k, w, h, texture=6), 90, s) for k, (w, h, s) in
             enumerate([(2000, 1333, "420"), (1333, 2000, "422"), (1200, 800, "444"), (640, 480, "420")])]
    counts, shapes, status = pipe.upload_jpegs(blobs, target)
    assert status.tolist() == [0] * len(blobs) and counts.sum() > 100
    rows = np.empty((int(counts.sum()), 7), np.float64)
    _lib.check(pipe.ctx.lib.vpk_lsd_fetch(pipe.ctx.h, _lib.ptr(rows)), "vpk_lsd_fetch")
    pipe.run()
    got = pipe.fetch()
    hz = pipe.horizons()
    rc, rs = pipe.upload_photos([J.decode(b) for b in blobs], target)
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
    good = J.encode_cv2(J.photo(1, 120, 90, texture=6), 90, "420")
    prog = dict((n, b) for n, b, _ in J.refused())["progressive_cv2"]
    gray = J.encode_cv2(J.photo(2, 120, 90, texture=6)[:, :, 0], 90)
    with pytest.raises(_lib.VpkError, match="file 1 .*progressive"):
        images.decode_jpegs([good, prog])
    with pytest.raises(_lib.VpkError, match="photo 1 is not supported: reason 1"):
        pipe.upload_jpegs([good, prog], 640)
    with pytest.raises(_lib.VpkError, match="photo 2 has 1 component"):
        pipe.upload_jpegs([good, good, gray], 640)
    with pytest.raises(ValueError):
        pipe.upload_jpegs([], 640)
    got, st = images.decode_jpegs([gray, good])         # gray files decode; they just cannot be prepared
    np.testing.assert_array_equal(got[0], J.decode(gray))
    np.testing.assert_array_equal(got[1], J.decode(good))


def test_checked_build_runs_the_bit_equality_corpus(tmp_path):
    """A VPK_DEFINES=VPK_JPEG_CHECKS copy of the library (every index into the bitstreams, block arrays and planes
    asserted) decodes the corpus, one file per call, without an assert firing."""
    tree = str(tmp_path / "tree")
    pkg = os.path.join(tree, "vanishing_points_2017_b200")
    shutil.copytree(os.path.join(ROOT, "vanishing_points_2017_b200"), pkg,
                    ignore=shutil.ignore_patterns("_obj", "*.so", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    env = dict(os.environ, VPK_DEFINES="VPK_JPEG_CHECKS", PYTHONPATH=os.pathsep.join([tree, ROOT]))
    subprocess.check_call([sys.executable, "-m", "vanishing_points_2017_b200.build"], env=env, cwd=tree)
    code = ("import vanishing_points_2017_b200 as v, sys; assert v.__file__.startswith(%r), v.__file__; "
            "sys.path.insert(0, %r); import test_jpeg_gpu as t; t.check_corpus(t.CORPUS, batch=False); print('checked ok')"
            % (tree, os.path.join(ROOT, "tests")))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=tree, capture_output=True, text=True)
    assert out.returncode == 0 and "checked ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
