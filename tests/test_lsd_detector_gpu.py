"""Row N4 on the device: vpk_lsd (through lsd.detect_line_segments[_batch]) against the float64 oracle of LSD 1.6,
batch / dtype / size-fallback consistency, and the path from images to horizons through Pipeline.upload_images."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import lsd_detector_oracle as L
from oracle import lsd_oracle
from vanishing_points_2017_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-9

CASES = [("640x480", lambda: synth.render_scene(21, 200)),
         ("480x640", lambda: synth.render_scene(22, 200, 480, 640)),
         ("800x533", lambda: synth.render_scene(23, 200, 800, 533)),
         ("odd_37x23", lambda: synth.render_scene(24, 6, 37, 23)),
         ("1x1", lambda: np.full((1, 1), 9.0)),
         ("constant", lambda: np.full((90, 120), 77.0)),
         ("noise", lambda: np.random.RandomState(3).uniform(0.0, 255.0, (256, 256)))]


def compare_rows(got, ref):
    """(rows paired, rows equal in all seven columns to 1e-9, max(len)).  Rows pair when their endpoints agree to
    1e-6; paired rows must come in the same order."""
    pair = []
    for a in got:
        d = np.abs(ref[:, :4] - a[:4]).max(axis=1) if len(ref) else np.zeros(0)
        pair.append(int(np.argmin(d)) if d.size and d.min() <= 1e-6 else -1)
    pair = np.array(pair, dtype=np.int64)
    ok = pair >= 0
    assert np.all(np.diff(pair[ok]) > 0), "paired rows out of order"
    exact = int(np.all(np.abs(got[ok] - ref[pair[ok]]) <= TOL, axis=1).sum())
    return int(ok.sum()), exact, max(len(got), len(ref))


def same_rows(got, ref, stats=None):
    """The device rows against the oracle's.  Agreement is bit-level except where a pixel lies exactly on a
    rectangle side: region2rect builds the sides through the region's extreme pixel centres, and whether rect_nfa
    counts such a pixel is decided by the last bit of cos / sin / atan2, where CUDA's libm and the C library differ
    by an ulp.  That moves p / -log10(NFA) of a row by one aligned pixel and can decide a marginal row
    (DESIGN.md section 4.6).  Required: >= 98 % of the rows pair up by their endpoints, >= 95 % agree in all seven
    columns to 1e-9."""
    paired, exact, n = compare_rows(got, ref)
    if stats is not None:
        stats += [paired, exact, n]
        return
    assert paired >= 0.98 * n, "only %d of %d rows pair up" % (paired, n)
    assert exact >= 0.95 * n, "only %d of %d rows within %g" % (exact, n, TOL)


@pytest.mark.parametrize("name,make", CASES, ids=[c[0] for c in CASES])
def test_vpk_lsd_matches_the_oracle(name, make):
    from vanishing_points_2017_b200 import lsd
    img = make()
    same_rows(lsd.detect_line_segments(img), L.detect_line_segments(img))


def test_vpk_lsd_nondefault_parameters():
    from vanishing_points_2017_b200 import lsd
    img = synth.render_scene(25, 200)
    kw = dict(scale=1.0, quant=3.0, ang_th=30.0, n_bins=256)
    ref = L.detect_line_segments(img, **kw)
    assert ref.shape[0] > 20
    same_rows(lsd.detect_line_segments(img, **kw), ref)


def test_mixed_size_batch_equals_per_image_calls_and_uint8_equals_float64():
    from vanishing_points_2017_b200 import lsd
    imgs = [synth.render_scene(30 + k, 120, w, h) for k, (w, h) in enumerate([(640, 480), (37, 23), (800, 533), (1, 1),
                                                                              (480, 640), (64, 48)])]
    batch = lsd.detect_line_segments_batch(imgs)
    batch_u8 = lsd.detect_line_segments_batch([im.astype(np.uint8) for im in imgs])
    for im, rows, rows_u8 in zip(imgs, batch, batch_u8):
        single = lsd.detect_line_segments(im)
        np.testing.assert_array_equal(rows, single)
        np.testing.assert_array_equal(rows_u8, rows)


def test_batch_of_more_images_than_resident_warps():
    """1100 images: more than the region kernel's 1024 warp slots, so warps take several images each.  The batch
    must give exactly the rows of one call per image (one warp, one wave each), and its rows must pair up with the
    oracle's by their endpoints."""
    from vanishing_points_2017_b200 import lsd
    imgs = [synth.render_scene(5000 + k, 10, 60 + k % 7, 44 + k % 5).astype(np.uint8) for k in range(1100)]
    got = lsd.detect_line_segments_batch(imgs)
    assert sum(r.shape[0] for r in got) > 100
    tot = np.zeros(3, np.int64)
    for g, im in zip(got, imgs):
        np.testing.assert_array_equal(g, lsd.detect_line_segments(im))
        st = []
        same_rows(g, L.detect_line_segments(im), st)
        tot += st
    paired, exact, n = tot
    assert paired >= 0.98 * n, tot


def test_image_too_large_for_the_shared_memory_bitmap_takes_the_global_memory_path():
    """1000 x 800 at scale 1: 800000 pixels, more than the 786432 bits of the shared-memory bitmap."""
    from vanishing_points_2017_b200 import lsd
    img = synth.render_scene(41, 300, 1000, 800)
    same_rows(lsd.detect_line_segments(img, scale=1.0), L.detect_line_segments(img, scale=1.0))


def test_image_with_more_rows_than_the_slab_is_rerun(tmp_path):
    """With the per-image row slab forced down to 4 rows, every image is re-run with the exact count."""
    code = ("import numpy as np, json; from vanishing_points_2017_b200 import lsd, synth; "
            "imgs = [synth.render_scene(51 + k, 150) for k in range(3)]; "
            "r = lsd.detect_line_segments_batch(imgs); np.savez(OUT, *r)")
    out = os.path.join(str(tmp_path), "rows.npz")
    env = dict(os.environ, VPK_LSD_ROWS_CAP="4", PYTHONPATH=ROOT)
    subprocess.check_call([sys.executable, "-c", code.replace("OUT", json.dumps(out))], env=env, cwd=ROOT)
    got = np.load(out)
    for k in range(3):
        ref = L.detect_line_segments(synth.render_scene(51 + k, 150))
        assert ref.shape[0] > 4
        same_rows(got["arr_%d" % k], ref)


def test_detect_lsd_lines_matches_the_oracle_rows_normalised():
    from vanishing_points_2017_b200 import evaluation
    img = synth.render_scene(61, 200)
    ref = lsd_oracle.segments_from_lsd(L.detect_line_segments(img), img.shape)
    got = evaluation.detect_lsd_lines(img)
    same_rows(np.column_stack([got["segments"], got["nfa"]]), np.column_stack([ref["segments"], ref["nfa"]]))
    got01 = evaluation.detect_lsd_lines(img / 255.0)       # the reference's "* 255 if max <= 1"
    assert got01["segments"].shape[0] > 0


def test_pipeline_from_images_equals_pipeline_from_lsd_rows():
    from vanishing_points_2017_b200 import cnn as vcnn, lsd, pipeline
    ws, bs = vcnn.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes")
    imgs = [synth.render_scene(70 + k, 250, w, h).astype(np.uint8) for k, (w, h) in enumerate([(640, 480), (800, 533), (480, 640), (640, 480)])]
    rows = lsd.detect_line_segments_batch(imgs)
    counts = pipe.upload_images(imgs)
    np.testing.assert_array_equal(counts, [r.shape[0] for r in rows])
    pipe.run()
    got, sig, sph = pipe.fetch(want_response=True, want_sphere=True)
    hz = pipe.horizons()
    off = np.concatenate([[0], np.cumsum([r.shape[0] for r in rows])]).astype(np.int32)
    pipe.upload_lsd(np.concatenate(rows), off, [im.shape[1] for im in imgs], [im.shape[0] for im in imgs])
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
