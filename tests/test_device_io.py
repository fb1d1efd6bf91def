"""Row N9 without a GPU: _lib.cuda_array reads __cuda_array_interface__ v2 / v3 descriptions (contiguous, strided,
permuted, with a producer stream) and refuses what the device entry points cannot take, _lib.call_stream picks the
stream a call is ordered on, and libvpk.so exports the device entry points with the prototypes include/vpk.h gives."""
import sys

import pytest

from vanishing_points_2017_b200 import _lib


class Fake:
    """An object exposing a __cuda_array_interface__ dict, as a CUDA array library would."""

    def __init__(self, shape, typestr="|u1", strides=None, version=2, ptr=0x7f0000001000, **extra):
        self.__cuda_array_interface__ = dict(shape=shape, typestr=typestr, strides=strides, data=(ptr, False), version=version,
                                             **extra)


def test_contiguous_arrays_get_c_strides():
    a = _lib.cuda_array(Fake((480, 640, 3)))
    assert a == _lib.CudaArray(0x7f0000001000, (480, 640, 3), (1920, 3, 1), _lib.U8, None)
    a = _lib.cuda_array(Fake((100, 4), "<f8"), (_lib.F64,), (2,))
    assert a.strides == (32, 8) and a.typestr == _lib.F64
    assert _lib.cuda_array(Fake((7, 5))).strides == (5, 1)


def test_strided_and_permuted_views_keep_their_strides():
    # a crop of a (1000, 1500, 3) photo, a CHW tensor permuted to HWC, a column slice of (N, 7) float64 rows
    crop = _lib.cuda_array(Fake((480, 640, 3), strides=(4500, 3, 1), ptr=0x7f0000001000 + 4500 * 11 + 3 * 7))
    assert crop.strides == (4500, 3, 1) and crop.ptr == 0x7f0000001000 + 49521
    chw = _lib.cuda_array(Fake((480, 640, 3), strides=(640, 1, 480 * 640)))
    assert chw.shape == (480, 640, 3) and chw.strides == (640, 1, 307200)
    cols = _lib.cuda_array(Fake((300, 4), "<f8", strides=(56, 8)), (_lib.F64,), (2,))
    assert cols.strides == (56, 8)
    gray = _lib.cuda_array(Fake((480, 640), strides=(2048, 2)))
    assert gray.strides == (2048, 2)
    zero = _lib.cuda_array(Fake((480, 640), strides=(0, 1)))       # a broadcast row: stride 0 repeats it
    assert zero.strides == (0, 1)


def test_v2_and_v3_streams():
    assert _lib.cuda_array(Fake((4, 4), version=2, stream=12345)).stream is None     # v2 has no stream
    assert _lib.cuda_array(Fake((4, 4), version=3, stream=12345)).stream == 12345
    assert _lib.cuda_array(Fake((4, 4), version=3, stream=None)).stream is None
    assert _lib.cuda_array(Fake((4, 4), version=3, stream=1)).stream == 1
    assert _lib.cuda_array(Fake((4, 4), "<u1")).typestr == _lib.U8                    # byte order of a byte is moot
    assert _lib.cuda_array(Fake((4, 4), "=f8"), (_lib.F64,)).typestr == _lib.F64


@pytest.mark.parametrize("fake,kw,match", [
    (Fake((4, 4), "<f4"), {}, "type"),
    (Fake((4, 4), "<f8"), {"typestrs": (_lib.U8,)}, "type"),
    (Fake((4, 4), "<i2"), {}, "type"),
    (Fake((4, 4, 3, 1)), {}, "dimensions"),
    (Fake((16,)), {}, "dimensions"),
    (Fake((4, 4, 3)), {"ndims": (2,)}, "dimensions"),
    (Fake((4, 4, 4)), {}, "channels"),
    (Fake((4, 4, 2)), {}, "channels"),
    (Fake((4, 4), strides=(-4, 1)), {}, "negative"),
    (Fake((4, 4, 3), strides=(12, 3, -1)), {}, "negative"),
    (Fake((4, 4), "<f8", strides=(32, 4)), {"typestrs": (_lib.F64,)}, "whole elements"),
    (Fake((4, 4), strides=(4,)), {}, "strides"),
    (Fake((4, 4), version=1), {}, "version"),
    (Fake((4, 4), mask=object()), {}, "mask"),
], ids=["float32", "f8_where_u8", "int16", "rank4", "rank1", "rank3_for_planes", "rgba", "two_channels", "negative_rows",
        "negative_channels", "half_element_stride", "stride_count", "version1", "mask"])
def test_refusals(fake, kw, match):
    with pytest.raises(ValueError, match=match):
        _lib.cuda_array(fake, **kw)


def test_cuda_array_imports_nothing():
    before = set(sys.modules)
    _lib.cuda_array(Fake((480, 640, 3), strides=(640, 1, 307200)))
    assert set(sys.modules) == before


class Handle:
    def __init__(self, h):
        self.cuda_stream = h


def test_call_stream_takes_handles_and_stream_objects():
    assert _lib.call_stream(0, 0) == 0
    assert _lib.call_stream(0xabc000, 0) == 0xabc000
    assert _lib.call_stream(Handle(0xdef000), 0) == 0xdef000
    # an input that exports the legacy default stream (1) is already ordered on stream 0, and the reverse
    a = _lib.cuda_array(Fake((4, 4), version=3, stream=1))
    assert _lib.call_stream(0, 0, [a]) == 0
    assert _lib.call_stream(1, 0, [_lib.cuda_array(Fake((4, 4), version=3, stream=None))]) == 1


def test_library_exports_the_device_entry_points():
    lib = _lib.load()
    names = ["vpk_pipeline_upload_device", "vpk_pipeline_upload_images_device", "vpk_pipeline_upload_photos_device",
             "vpk_pipeline_fetch_device", "vpk_pipeline_horizon_device"]
    for n in names:
        assert n in _lib.SYMBOLS and hasattr(lib, n), n
