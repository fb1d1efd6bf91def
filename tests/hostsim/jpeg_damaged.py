"""TEST INFRASTRUCTURE ONLY (run by tests/test_jpeg_hostsim.py under the address / undefined-behaviour sanitizers):
decodes damaged corpus files with the sanitized host build, sequentially and with 32- and 1024-bit subsequences.
Truncated and garbage-appended files must be CORRUPT; a bit-flipped file must be CORRUPT or decode identically
both ways (a flipped magnitude bit can leave the stream consistent)."""
import ctypes as C
import sys

import numpy as np

from oracle import jpeg_oracle as J


def run(lib, blob, L):
    buf = np.frombuffer(bytes(blob), np.uint8)
    dims = np.zeros(3, np.int32)
    st = lib.hostsim_jpeg(buf.ctypes.data, buf.size, L, None, 0, dims.ctypes.data, None)
    cap = int(dims[0]) * int(dims[1]) * int(dims[2]) if st in (J.OK, -1) else 0
    out = np.zeros(max(cap, 1), np.uint8)
    st = lib.hostsim_jpeg(buf.ctypes.data, buf.size, L, out.ctypes.data, cap, dims.ctypes.data, None)
    return st, out[:cap]


lib = C.CDLL(sys.argv[1])
lib.hostsim_jpeg.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
lib.hostsim_jpeg.restype = C.c_int
blobs = [J.encode_cv2(J.photo(1, 200, 150, texture=8), 90, "420"),
         J.encode_cv2(J.noise(2, 97, 61), 100, "444", restart=3),
         J.encode_cv2(J.photo(3, 120, 90, texture=8)[:, :, 0], 75, restart=1),
         J.encode_pil(J.photo(4, 160, 100, texture=8), 90, 1)]
n = 0
for i, blob in enumerate(blobs):
    for seed in range(3):
        for name, bad in J.corrupted(blob, 10 * i + seed):
            res = [run(lib, bad, L) for L in (0, 32, 1024)]
            sts = [r[0] for r in res]
            if name == "bitflip":
                assert sts[0] in (J.OK, J.CORRUPT) and len(set(sts)) == 1, (i, seed, name, sts)
                if sts[0] == J.OK:
                    assert all(np.array_equal(r[1], res[0][1]) for r in res), (i, seed, name)
            else:
                assert sts == [J.CORRUPT] * 3, (i, seed, name, sts)
            n += 1
print("damaged ok", n)
