"""Row N6 on the CPU: the host build of the decoder's core (csrc/jpeg_core.cuh through tests/hostsim/jpeg_hostsim.cpp)
decodes the corpus of oracle/jpeg_oracle.py sequentially and through a host emulation of the device's subsequence /
synchronisation / scan algorithm; both must equal libjpeg-turbo bit for bit.  A second build with
-fsanitize=address,undefined decodes damaged files and must report them CORRUPT without a sanitizer finding."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import jpeg_oracle as J

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "jpeg_hostsim.cpp")
CORE = os.path.join(HERE, "..", "vanishing_points_2017_b200", "csrc", "jpeg_core.cuh")
DEFAULT_BITS = 1024          # csrc/jpeg.cu kSubseqBits


def _build(path, extra):
    if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(SRC), os.path.getmtime(CORE)):
        tmp = path + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC"] + extra + ["-o", tmp, SRC])
        os.replace(tmp, path)
    return path


def _load(path):
    lib = C.CDLL(path)
    lib.hostsim_jpeg.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.hostsim_jpeg.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def hostsim(tmp_path_factory):
    return _load(_build(str(tmp_path_factory.mktemp("jpeg") / "_jpeg_hostsim.so"), []))


def run(lib, blob, L):
    buf = np.frombuffer(bytes(blob), np.uint8)
    dims = np.zeros(3, np.int32)
    stats = np.zeros(4, np.int64)
    cap = 0
    st = lib.hostsim_jpeg(buf.ctypes.data, buf.size, L, None, 0, dims.ctypes.data, None)
    if st == J.OK or st == -1:
        cap = int(dims[0]) * int(dims[1]) * int(dims[2])
    out = np.zeros(max(cap, 1), np.uint8)
    st = lib.hostsim_jpeg(buf.ctypes.data, buf.size, L, out.ctypes.data, cap, dims.ctypes.data, stats.ctypes.data)
    w, h, nc = (int(x) for x in dims)
    img = out[:w * h * nc].reshape((h, w, nc) if nc == 3 else (h, w)) if cap else None
    return st, img, stats


CORPUS = J.corpus(large=True)


@pytest.mark.parametrize("name,blob", CORPUS, ids=[c[0] for c in CORPUS])
def test_sequential_and_parallel_decode_equal_libjpeg_turbo(hostsim, name, blob):
    ref = J.decode(blob)
    bits = (32, 256, DEFAULT_BITS) if len(blob) < 2_000_000 else (256, DEFAULT_BITS)
    for L in (0,) + bits:
        st, img, stats = run(hostsim, blob, L)
        assert st == J.OK, (name, L, st)
        assert img.shape == ref.shape, (name, L)
        np.testing.assert_array_equal(img, ref, err_msg="%s L=%d" % (name, L))


def test_synchronisation_needs_rounds_with_small_subsequences(hostsim):
    """32-bit subsequences of a noise photo start most threads mid-symbol: the emulation must re-decode and
    still land on the sequential result"""
    blob = J.encode_cv2(J.noise(1, 160, 120), 100, "420")
    st, img, stats = run(hostsim, blob, 32)
    assert st == J.OK and stats[0] > 1000 and stats[1] > 0
    np.testing.assert_array_equal(img, J.decode(blob))


@pytest.fixture(scope="module")
def hostsim_asan(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("jpeg_asan") / "_jpeg_hostsim_asan.so")
    _build(path, ["-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-fno-omit-frame-pointer"])
    return path


def test_damaged_files_are_corrupt_without_sanitizer_findings(hostsim_asan):
    """A subprocess with the sanitizer runtime preloaded decodes truncated, bit-flipped and garbage-appended files
    both ways; any sanitizer finding aborts it."""
    import sys
    rt = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    script = os.path.join(HERE, "hostsim", "jpeg_damaged.py")
    env = dict(os.environ, LD_PRELOAD=rt, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1", PYTHONPATH=os.path.join(HERE, ".."))
    out = subprocess.run([sys.executable, script, hostsim_asan], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "damaged ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
