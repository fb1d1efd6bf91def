"""Row N7 on the CPU: the host build of the decoder's core (csrc/png_core.cuh through tests/hostsim/png_hostsim.cpp)
inflates every stream of oracle/png_oracle.py's corpus equal to zlib.decompress, sequentially and through a host
emulation of the warp's copy rule, and unfilters and expands equal to libpng.  A second build with
-fsanitize=address,undefined decodes the damaged files and must report them CORRUPT without a sanitizer finding."""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

from oracle import png_oracle as P

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "png_hostsim.cpp")
CORE = os.path.join(HERE, "..", "vanishing_points_2017_b200", "csrc", "png_core.cuh")


def _build(path, extra):
    tmp = path + ".%d.tmp" % os.getpid()
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC"] + extra + ["-o", tmp, SRC])
    os.replace(tmp, path)
    return path


def _load(path):
    lib = C.CDLL(path)
    lib.hostsim_png.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    lib.hostsim_png.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def hostsim(tmp_path_factory):
    return _load(_build(str(tmp_path_factory.mktemp("png") / "_png_hostsim.so"), []))


def run(lib, blob, mode):
    buf = np.frombuffer(bytes(blob), np.uint8)
    dims = np.zeros(5, np.int64)
    st = lib.hostsim_png(buf.ctypes.data, buf.size, mode, None, 0, None, 0, dims.ctypes.data)
    if st not in (P.OK, -1):
        return st, None, None
    raw = np.zeros(max(int(dims[3]), 1), np.uint8)
    out = np.zeros(max(int(dims[0] * dims[1] * dims[4]), 1), np.uint8)
    st = lib.hostsim_png(buf.ctypes.data, buf.size, mode, raw.ctypes.data, raw.size, out.ctypes.data, out.size, dims.ctypes.data)
    w, h, nc = int(dims[0]), int(dims[1]), int(dims[4])
    return st, raw[:int(dims[3])], out[:w * h * nc].reshape((h, w, 3) if nc == 3 else (h, w))


CORPUS = P.corpus(large=False)


@pytest.mark.parametrize("name,blob", CORPUS, ids=[c[0] for c in CORPUS])
def test_inflate_unfilter_expand_equal_zlib_and_libpng(hostsim, name, blob):
    raw_ref = zlib.decompress(P._zstream(blob))
    ref = P.decode(blob)
    for mode in (0, 1):
        st, raw, img = run(hostsim, blob, mode)
        assert st == P.OK, (name, mode, st)
        assert raw.tobytes() == raw_ref, (name, mode)
        assert img.shape == ref.shape, (name, mode)
        np.testing.assert_array_equal(img, ref, err_msg="%s mode %d" % (name, mode))


@pytest.mark.parametrize("d", list(range(1, 32)))
def test_periodic_copy_at_short_distances(hostsim, d):
    """a row of period d: deflate codes it as one long match at distance d; the warp's copy rule must reproduce it"""
    row = np.tile(np.random.RandomState(d).randint(0, 256, d).astype(np.uint8), 600 // d + 1)[:600]
    src = np.repeat(row[None, :], 4, axis=0)
    blob = P.write(src, 0, 8, filters=0, level=9)
    st, raw, img = run(hostsim, blob, 1)
    assert st == P.OK
    np.testing.assert_array_equal(img, src)


def test_extra_data_after_the_last_row_decodes(hostsim):
    for name, blob, exp in P.extra_data():
        for mode in (0, 1):
            st, _, img = run(hostsim, blob, mode)
            assert st == P.OK, (name, mode)
            np.testing.assert_array_equal(img, exp, err_msg=name)
            np.testing.assert_array_equal(img, P.decode(blob), err_msg=name)


def test_damaged_files_are_corrupt(hostsim):
    for name, blob in P.corrupted():
        assert [run(hostsim, blob, m)[0] for m in (0, 1)] == [P.CORRUPT] * 2, name


@pytest.fixture(scope="module")
def hostsim_asan(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("png_asan") / "_png_hostsim_asan.so")
    return _build(path, ["-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-fno-omit-frame-pointer"])


def test_damaged_files_without_sanitizer_findings(hostsim_asan):
    rt = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    script = os.path.join(HERE, "hostsim", "png_damaged.py")
    env = dict(os.environ, LD_PRELOAD=rt, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1", PYTHONPATH=os.path.join(HERE, ".."))
    out = subprocess.run([sys.executable, script, hostsim_asan], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "damaged ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
