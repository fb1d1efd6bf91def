"""The per-kernel EM reference (oracle/em_kernel_oracle.py) on the CPU: the Python layouts agree with the ones
csrc/em_core.cuh defines (compiled with g++), the float64 emulation of em_pair / em_estep / em_wmat passes every
check, and every planted bug fails the check of the kernel it is in by a wide margin.  The GPU file
(test_em_kernels_gpu.py) applies the same checks to the buffers the kernels leave in the workspace."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import em_kernel_oracle as ek
from vanishing_points_2017_b200 import vp_localisation as vl

HERE = os.path.dirname(os.path.abspath(__file__))
CORE = os.path.join(HERE, "..", "vanishing_points_2017_b200", "csrc", "em_core.cuh")
SHIM = r"""
#include "%s"
using namespace vpk::em;
extern "C" void layout_lsim(int N, long long* out) {
    for (int j = 0; j < N; ++j) for (int k = 0; k < N; ++k) out[(size_t)j * N + k] = (long long)lsim_index(N, j, k);
}
extern "C" void layout_wt(int N, int M, int rows, long long* out) {
    for (int m = 0; m < rows; ++m) for (int n = 0; n < N; ++n) out[(size_t)m * N + n] = (long long)wt_index(N, n, m, M);
}
extern "C" long long layout_lsim_doubles(int N) { return (long long)lsim_doubles(N); }
"""
MARGIN = 4.0          # a planted bug must exceed its kernel's bound by this factor


@pytest.fixture(scope="module")
def layout(tmp_path_factory):
    d = tmp_path_factory.mktemp("em_layout")
    src, so = d / "layout.cpp", d / "layout.so"
    src.write_text(SHIM % os.path.abspath(CORE))
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(so), str(src)])
    lib = C.CDLL(str(so))
    lib.layout_lsim.argtypes = [C.c_int, C.c_void_p]
    lib.layout_wt.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.layout_lsim_doubles.argtypes = [C.c_int]
    lib.layout_lsim_doubles.restype = C.c_longlong
    return lib


@pytest.mark.parametrize("N", [1, 31, 63, 64, 65, 1537])
def test_lsim_layout_matches_em_core(layout, N):
    want = np.empty(N * N, np.int64)
    layout.layout_lsim(N, want.ctypes.data)
    j, k = np.meshgrid(np.arange(N), np.arange(N), indexing="ij")
    np.testing.assert_array_equal(vl.lsim_index(N, j, k).ravel(), want)
    assert layout.layout_lsim_doubles(N) == ek.lsim_doubles(N)
    # every element has its own place and the unpacker inverts the packer
    assert np.unique(want).size == N * N and want.max() < ek.lsim_doubles(N)
    L = np.random.RandomState(N).rand(N, N)
    np.testing.assert_array_equal(vl.unpack_lsim(ek.pack_lsim(L), N), L)


@pytest.mark.parametrize("N", [1, 31, 63, 64, 65, 1537])
@pytest.mark.parametrize("M", [1, 8, 9, 32, 33, 64])
def test_wt_layout_matches_em_core(layout, N, M):
    rows = vl.wt_rows(M)
    want = np.empty(rows * N, np.int64)
    layout.layout_wt(N, M, rows, want.ctypes.data)
    m, n = np.meshgrid(np.arange(rows), np.arange(N), indexing="ij")
    np.testing.assert_array_equal(vl.wt_index(N, n, m, M).ravel(), want)
    assert np.unique(want).size == rows * N and want.max() < (M + 31) // 32 * N * 36
    wt = np.random.RandomState(M).rand(rows, N)
    np.testing.assert_array_equal(vl.unpack_wt(ek.pack_wt(wt, N, M), N, M), wt)


def _constants(seed, vps):
    rs = np.random.RandomState(seed)
    M = vps.shape[0]
    return ek.estep_constants(vps, rs.uniform(1e-8, 1e-3, M), rs.uniform(0.1, 2.0, M))


# (N, M, wbias, use_weights): partial last chunk and slab, M = 1 ... 64 across both W passes, a 2-CTA cluster
EMU_CASES = [(33, 9, 1.0, True), (65, 1, 1.0, True), (200, 40, 0.37, True), (300, 64, 1.0, True),
             (1600, 33, 1.0, True), (150, 17, 1.0, False)]


@pytest.mark.parametrize("N,M,wbias,use_weights", EMU_CASES)
def test_emulation_passes_every_check(N, M, wbias, use_weights):
    sc = ek.vp_scene(N + M, N, M)
    buf = ek.emulate(sc["segments"], _constants(N, sc["vps"]), wbias=wbias, use_weights=use_weights)
    worst, ties = ek.check_all(sc["segments"], buf, wbias=wbias, use_weights=use_weights)
    print("N=%d M=%d worst |dev - ref| / bound: %s, near-ties %d" % (N, M, {k: "%.3g" % v for k, v in worst.items()}, len(ties)))
    assert max(worst.values()) <= 1.0, worst
    assert len(ties) <= max(1, N // 100), ties


def test_emulation_ties_resolved_by_index_without_near_ties():
    sc = ek.tie_scene(0, 300)
    lsim, colsum, lweight = ek.emulate_pair(sc["segments"])
    worst, ties = ek.check_lweight(sc["segments"], lweight, np.arange(300))
    assert ties == [] and worst <= 1.0, (worst, ties)


def _bug_case(bug):
    if bug == "knn_ties_larger_index":
        return ek.tie_scene(1, 300), 0, 1.0
    if bug == "rank_range_off_by_one":
        return ek.vp_scene(7, 1600, 40), 40, 1.0
    if bug == "stale_rows":
        return ek.vp_scene(7, 203, 40), 40, 1.0           # N % 32 != 0: the last chunk is partial
    return ek.vp_scene(7, 200, 40), 40, (0.37 if bug == "wbias_twice" else 1.0)


@pytest.mark.parametrize("bug", sorted(ek.BUGS))
def test_planted_bug_fails_its_kernel(bug):
    sc, M, wbias = _bug_case(bug)
    N = sc["segments"].shape[0]
    vps = sc["vps"] if M else np.tile([[0.3, 0.2, 0.93]], (1, 1))
    est = _constants(3, vps)
    buf = ek.emulate(sc["segments"], est, wbias=wbias, bug=bug)
    worst, _ = ek.check_all(sc["segments"], buf, wbias=wbias, exact=False)
    kernel = ek.BUGS[bug]
    print("%s: %s %.3g" % (bug, kernel, worst[kernel]))
    assert worst[kernel] > MARGIN, worst
    # and the kernels upstream of the bug still pass: the failure names the kernel
    upstream = {"lsim": [], "colsum": ["lsim"], "lweight": ["lsim", "colsum"], "pvl": ["lsim", "colsum", "lweight", "lvsq"],
                "w": ["lsim", "colsum", "lweight", "lvsq", "pvl"]}[kernel]
    assert all(worst[k] <= 1.0 for k in upstream), worst


def test_clip_at_0_98_is_an_equivalent_mutant():
    """Moving the cos 9 theta clip from cos(pi/18) down to 0.98 changes nothing: on (0.98, cos(pi/18)] T9 is negative
    and the clamp to cos(fl(pi/2)) gives the clipped value anyway.  The planted clip bug moves it up (0.99) instead."""
    c = np.linspace(0.98, ek.CLIP_C, 10001)
    t = c * (4.0 * c * c - 3.0)
    r = t * (4.0 * t * t - 3.0)
    assert np.all(np.where(r < ek.AT_CLIP, ek.AT_CLIP, r) == ek.AT_CLIP)
