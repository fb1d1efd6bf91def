"""Row N5 on the device: vpk_prepare_images (images.prepare_images) bit for bit against oracle/image_prep_oracle.py,
batch against single calls, the fused Pipeline.upload_photos against the host-scaled path, bad input, and the
VPK_PREP_CHECKS build."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from oracle import image_prep_oracle as P
from vanishing_points_2017_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def noise(seed, w, h):
    return np.random.RandomState(seed).randint(0, 256, (h, w, 3)).astype(np.uint8)


# (id, photo factory, target_size); sizes are w x h
CASES = [("2000x1333_640", lambda: synth.render_photo(1, 200, 2000, 1333), 640),
         ("1333x2000_640", lambda: synth.render_photo(2, 200, 1333, 2000), 640),
         ("2048x1363_640", lambda: synth.render_photo(3, 200, 2048, 1363), 640),
         ("1280x960_640_integer2", lambda: synth.render_photo(4, 200, 1280, 960), 640),
         ("1200x900_800", lambda: synth.render_photo(5, 200, 1200, 900), 800),
         ("6000x4000_640", lambda: noise(6, 6000, 4000), 640),
         ("no_resize", lambda: synth.render_photo(7, 100, 700, 500), None),
         ("640x480_640", lambda: synth.render_photo(8, 100, 640, 480), 640),
         ("5000x3_640", lambda: noise(9, 5000, 3), 640),
         ("1x1", lambda: noise(10, 1, 1), 640),
         ("constant", lambda: np.full((900, 1300, 3), (37, 180, 99), np.uint8), 640),
         ("white", lambda: np.full((1000, 1500, 3), 255, np.uint8), 640),
         ("noise_integer4", lambda: noise(11, 2560, 1920), 640),
         ("noise", lambda: noise(12, 1700, 1100), 640)]


def check_cases(cases):
    from vanishing_points_2017_b200 import images
    for name, make, target in cases:
        img = make()
        got = images.prepare_images([img], target)[0]
        ref = P.prepare(img, target)
        assert got.shape == ref.shape, name
        np.testing.assert_array_equal(got, ref, err_msg=name)


@pytest.mark.parametrize("name,make,target", CASES, ids=[c[0] for c in CASES])
def test_prepare_images_equals_the_oracle_bit_for_bit(name, make, target):
    check_cases([(name, make, target)])


def test_white_photo_gives_exactly_255_for_lsd():
    from vanishing_points_2017_b200 import images
    g = images.prepare_images([np.full((1000, 1500, 3), 255, np.uint8)], 640)[0]
    assert g.shape == (427, 640) and np.all(g == 1.0) and np.all(g * 255 == 255.0)


def test_mixed_batch_equals_one_call_per_photo():
    from vanishing_points_2017_b200 import images
    photos = [make() for _, make, t in CASES if t == 640]
    photos.insert(3, noise(20, 33, 17))                  # identity inside a resizing batch (smaller than the target)
    batch = images.prepare_images(photos, 640)
    assert len(batch) == len(photos)
    for p, g in zip(photos, batch):
        np.testing.assert_array_equal(g, images.prepare_images([p], 640)[0])
        assert g.shape == P.prepared_size(p.shape[1], p.shape[0], 640)[::-1]


def test_upload_photos_equals_lsd_on_the_host_scaled_planes():
    from vanishing_points_2017_b200 import _lib, images, lsd, pipeline
    from vanishing_points_2017_b200 import cnn as vcnn
    ws, bs = vcnn.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes")
    photos = [synth.render_photo(80 + k, 250, w, h) for k, (w, h) in enumerate([(2000, 1333), (1333, 2000), (1280, 960), (1200, 900)])]
    planes = [g * 255 for g in images.prepare_images(photos, 640)]
    rows = lsd.detect_line_segments_batch(planes)
    counts, shapes = pipe.upload_photos(photos, 640)
    assert shapes == [p.shape for p in planes]
    np.testing.assert_array_equal(counts, [r.shape[0] for r in rows])
    assert counts.sum() > 100
    got_rows = np.empty((int(counts.sum()), 7), np.float64)
    _lib.check(pipe.ctx.lib.vpk_lsd_fetch(pipe.ctx.h, _lib.ptr(got_rows)), "vpk_lsd_fetch")
    np.testing.assert_array_equal(got_rows, np.concatenate(rows))
    pipe.run()
    got, sig, sph = pipe.fetch(want_response=True, want_sphere=True)
    hz = pipe.horizons()
    ref_counts = pipe.upload_images(planes)
    np.testing.assert_array_equal(ref_counts, counts)
    pipe.run()
    ref, rsig, rsph = pipe.fetch(want_response=True, want_sphere=True)
    rhz = pipe.horizons()
    np.testing.assert_array_equal(sph, rsph)
    np.testing.assert_array_equal(sig, rsig)
    for a, b in zip(got, ref):
        assert (a["vp"] is None) == (b["vp"] is None)
        if a["vp"] is not None:
            np.testing.assert_array_equal(a["vp"], b["vp"])
            np.testing.assert_array_equal(a["vp_assoc"], b["vp_assoc"])
    for a, b in zip(hz, rhz):
        for q in range(6):
            np.testing.assert_array_equal(np.asarray(a[q]), np.asarray(b[q]))


def test_bad_input_is_rejected():
    from vanishing_points_2017_b200 import _lib, images, pipeline
    from vanishing_points_2017_b200 import cnn as vcnn
    ok = noise(1, 40, 30)
    for bad in ([np.zeros((30, 40), np.uint8)], [ok.astype(np.float64)], [np.zeros((30, 40, 4), np.uint8)],
                [np.zeros((0, 40, 3), np.uint8)], ok):
        with pytest.raises(ValueError):
            images.prepare_images(bad, 640)
    ctx = _lib.default_context()
    lib = ctx.lib
    w = np.array([40], np.int32)
    h = np.array([30], np.int32)
    out = np.empty(40 * 30, np.float64)
    ow, oh = np.empty(1, np.int32), np.empty(1, np.int32)
    flat = np.ascontiguousarray(ok.reshape(-1))
    for off, ww in ((np.array([0, 40 * 30], np.int64), w), (np.array([0, 3 * 40 * 30], np.int64), np.array([0], np.int32))):
        st = lib.vpk_prepare_images(ctx.h, _lib.ptr(flat), _lib.ptr(off), _lib.ptr(ww), _lib.ptr(h), 1, 0, _lib.ptr(ow), _lib.ptr(oh),
                                    _lib.ptr(out))
        assert st == 1 and b"byte_offsets" in lib.vpk_last_error()
    ws, bs = vcnn.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes")
    with pytest.raises(ValueError):
        pipe.upload_photos([])
    with pytest.raises(_lib.VpkError, match="65536"):
        pipe.upload_photos([noise(2, 90000, 1)])              # the LSD limit applies to the prepared size
    with pytest.raises(_lib.VpkError, match="too large"):
        images.prepare_images([noise(3, 2000, 2000)], 4)       # factor 500: one output's source exceeds shared memory
    np.testing.assert_array_equal(images.prepare_images([ok], None)[0], P.prepare(ok))   # the context still works


def test_checked_build_runs_the_bit_equality_cases(tmp_path):
    """A VPK_DEFINES=VPK_PREP_CHECKS copy of the library (every shared- and global-memory index of image_prep
    asserted) runs the bit-equality cases without an assert firing."""
    tree = str(tmp_path / "tree")
    pkg = os.path.join(tree, "vanishing_points_2017_b200")
    shutil.copytree(os.path.join(ROOT, "vanishing_points_2017_b200"), pkg,
                    ignore=shutil.ignore_patterns("_obj", "*.so", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    env = dict(os.environ, VPK_DEFINES="VPK_PREP_CHECKS", PYTHONPATH=os.pathsep.join([tree, ROOT]))
    subprocess.check_call([sys.executable, "-m", "vanishing_points_2017_b200.build"], env=env, cwd=tree)
    code = ("import vanishing_points_2017_b200 as v, sys; assert v.__file__.startswith(%r), v.__file__; "
            "sys.path.insert(0, %r); import test_image_prep_gpu as t; t.check_cases(t.CASES); print('checked ok')"
            % (tree, os.path.join(ROOT, "tests")))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=tree, capture_output=True, text=True)
    assert out.returncode == 0 and "checked ok" in out.stdout, out.stdout + out.stderr
