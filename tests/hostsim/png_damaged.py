"""TEST INFRASTRUCTURE ONLY (run by tests/test_png_hostsim.py under the address / undefined-behaviour sanitizers):
decodes the damaged files of oracle/png_oracle.py, of several base files, with the sanitized host build both ways.
Every one must be CORRUPT, and both ways must give the same bytes."""
import ctypes as C
import sys

import numpy as np

from oracle import png_oracle as P


def run(lib, blob, mode):
    buf = np.frombuffer(bytes(blob), np.uint8)
    dims = np.zeros(5, np.int64)
    lib.hostsim_png(buf.ctypes.data, buf.size, mode, None, 0, None, 0, dims.ctypes.data)
    raw = np.zeros(max(int(dims[3]), 1), np.uint8)
    out = np.zeros(max(int(dims[0] * dims[1] * dims[4]), 1), np.uint8)
    st = lib.hostsim_png(buf.ctypes.data, buf.size, mode, raw.ctypes.data, raw.size, out.ctypes.data, out.size, dims.ctypes.data)
    return st, out


lib = C.CDLL(sys.argv[1])
lib.hostsim_png.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
lib.hostsim_png.restype = C.c_int
bases = [None, P.write(P.samples(1, 41, 29, 3, 4), 3, 4, P.palette_of(1, 16), interlace=1),
         P.write(P.samples(2, 70, 50, 6, 8), 6, 8, idat_size=100), P.encode_cv2(P.photo(3, 90, 60, texture=8), 9)]
n = 0
for base in bases:
    for name, bad in P.corrupted(base):
        res = [run(lib, bad, m) for m in (0, 1)]
        assert [r[0] for r in res] == [P.CORRUPT] * 2, (name, [r[0] for r in res])
        assert np.array_equal(res[0][1], res[1][1]), name
        n += 1
print("damaged ok", n)
