"""Row N4 on the CPU: the LSD 1.6 oracle (oracle/lsd_detector_oracle.py) on known answers, cross-checked against
OpenCV's independent port of LSD 1.6, and the host build of the sequential core the CUDA kernels run
(csrc/lsd_core.cuh through tests/hostsim/lsd_hostsim.cpp) against the oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import lsd_detector_oracle as L
from vanishing_points_2017_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "lsd_hostsim.cpp")
CORE = os.path.join(HERE, "..", "vanishing_points_2017_b200", "csrc", "lsd_core.cuh")
SO = os.path.join(HERE, "hostsim", "_lsd_hostsim.so")
NONDEFAULT = dict(scale=1.0, quant=3.0, ang_th=30.0, n_bins=256)
# rendered scenes of the OpenCV cross-check: 100 bars 3 px wide, noise sigma 1
CV_SCENES = [synth.render_scene(100 + s, 100, line_width=3.0, noise_sigma=1.0).astype(np.uint8) for s in range(8)]


def test_degenerate_images_give_no_segments():
    for shape in ((1, 1), (2, 2)):
        assert L.detect_line_segments(np.zeros(shape)).shape == (0, 7)
    assert L.detect_line_segments(np.full((60, 80), 123.0)).shape == (0, 7)


def test_one_step_edge_gives_one_segment_along_it():
    img = np.zeros((150, 200))
    img[:, 100:] = 200.0
    for kw in ({}, dict(scale=1.0)):
        rows = L.detect_line_segments(img, **kw)
        assert rows.shape == (1, 7)
        x1, y1, x2, y2 = rows[0, :4]
        # the edge lies between pixel centres 99 and 100 and runs over the pixel rows 0 .. 149
        assert abs(x1 - 99.5) <= 1.0 and abs(x2 - 99.5) <= 1.0
        assert abs(min(y1, y2) - 0.0) <= 1.0 and abs(max(y1, y2) - 149.0) <= 1.0
        assert rows[0, 6] > 0.0


def test_nfa_above_log_eps_and_a_contrario_bound_on_noise():
    for s in (3, 4):
        rows = L.detect_line_segments(synth.render_scene(s, 120))
        assert rows.shape[0] > 50 and np.all(rows[:, 6] > 0.0)
    rows = L.detect_line_segments(synth.render_scene(3, 120), log_eps=2.0)
    assert np.all(rows[:, 6] > 2.0)
    for seed in range(3):
        noise = np.random.RandomState(seed).uniform(0.0, 255.0, (256, 256))
        assert L.detect_line_segments(noise).shape[0] <= 3


def _match(A, B, tol=1.0, minlen=10.0):
    """share of A's segments of length >= minlen with a segment of B whose two endpoints are within tol (either
    orientation)"""
    A = A[np.hypot(A[:, 2] - A[:, 0], A[:, 3] - A[:, 1]) >= minlen]
    ok = 0
    for a in A:
        d1 = np.maximum(np.hypot(B[:, 0] - a[0], B[:, 1] - a[1]), np.hypot(B[:, 2] - a[2], B[:, 3] - a[3]))
        d2 = np.maximum(np.hypot(B[:, 0] - a[2], B[:, 1] - a[3]), np.hypot(B[:, 2] - a[0], B[:, 3] - a[1]))
        ok += bool((np.minimum(d1, d2) <= tol).any())
    return ok / max(len(A), 1)


@pytest.mark.parametrize("k", range(len(CV_SCENES)))
def test_oracle_agrees_with_opencv_lsd(k):
    cv2 = pytest.importorskip("cv2")
    img = CV_SCENES[k]
    ours = L.detect_line_segments(img, scale=1.0)[:, :4]
    theirs = cv2.createLineSegmentDetector(cv2.LSD_REFINE_ADV, 1.0).detect(img)[0].reshape(-1, 4).astype(np.float64)
    assert _match(theirs, ours) >= 0.90
    assert _match(ours, theirs) >= 0.90


@pytest.fixture(scope="module")
def hostsim():
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(SRC), os.path.getmtime(CORE)):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO, SRC])
    lib = C.CDLL(SO)
    lib.hostsim_lsd.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_double] * 6 + [C.c_int, C.c_void_p, C.c_int]

    def run(img, scale=0.8, sigma_scale=0.6, quant=2.0, ang_th=22.5, log_eps=0.0, density_th=0.7, n_bins=1024):
        img = np.ascontiguousarray(img, np.float64)
        cap = 1 << 16
        rows = np.zeros((cap, 7))
        n = lib.hostsim_lsd(img.ctypes.data, img.shape[1], img.shape[0], scale, sigma_scale, quant, ang_th, log_eps,
                            density_th, n_bins, rows.ctypes.data, cap)
        return rows[:n]
    return run


HOST_CASES = [("scene_640x480", lambda: synth.render_scene(11, 150)),
              ("scene_480x640", lambda: synth.render_scene(12, 150, 480, 640)),
              ("scene_800x533", lambda: synth.render_scene(13, 150, 800, 533)),
              ("cv_scene", lambda: CV_SCENES[0].astype(np.float64)),
              ("odd_37x23", lambda: synth.render_scene(14, 6, 37, 23)),
              ("noise_256", lambda: np.random.RandomState(7).uniform(0.0, 255.0, (256, 256)))]


@pytest.mark.parametrize("name,make", HOST_CASES, ids=[c[0] for c in HOST_CASES])
@pytest.mark.parametrize("kw", [{}, NONDEFAULT], ids=["defaults", "nondefault"])
def test_host_build_of_the_core_matches_the_oracle(hostsim, name, make, kw):
    img = make()
    ref = L.detect_line_segments(img, **kw)
    got = hostsim(img, **kw)
    assert got.shape == ref.shape
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-9)
