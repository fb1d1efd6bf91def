"""Row N7 on the CPU: the PNG oracle's two decoders (cv2 and PIL) agree bit for bit on the corpus, the hand-written
files decode to the arrays they were written from, and vpk_png_info (host only) reads every corpus file's size and
colour type and the reason for every refused file."""
import numpy as np
import pytest

from oracle import png_oracle as P
from vanishing_points_2017_b200 import images

CORPUS = P.corpus(large=True)
REFUSED = P.refused()


@pytest.mark.parametrize("name,blob", CORPUS, ids=[c[0] for c in CORPUS])
def test_cv2_and_pil_decode_identically(name, blob):
    a, b = P.decode(blob), P.decode_pil(blob)
    assert a.shape == b.shape and a.dtype == np.uint8
    np.testing.assert_array_equal(a, b)


def test_written_files_equal_their_source_arrays():
    for name, blob, exp in P.written() + P.extra_data():
        np.testing.assert_array_equal(P.decode(blob), exp, err_msg=name)


def test_damaged_files_fail_in_libpng():
    for name, blob in P.corrupted():
        assert P.decode(blob) is None, name


def test_info_reads_size_colour_type_and_support_of_the_corpus():
    info = images.png_info([b for _, b in CORPUS])
    for (name, blob), (w, h, t, s) in zip(CORPUS, info):
        ref = P.decode(blob)
        assert s == P.OK, name
        assert (h, w) == ref.shape[:2], name
        assert t == P.color_type(blob), name


def test_info_gives_the_reason_of_every_refused_file():
    info = images.png_info([b for _, b, _ in REFUSED])
    for (name, _, why), (w, h, t, s) in zip(REFUSED, info):
        assert s == why, (name, s, why)


def test_info_accepts_arrays_and_rejects_other_input():
    blob = CORPUS[0][1]
    assert images.png_info([np.frombuffer(blob, np.uint8)]) == images.png_info([blob])
    assert images.png_info([]) == []
    for bad in (blob, [np.zeros((2, 2), np.uint8)], [np.zeros(4, np.int32)]):
        with pytest.raises(ValueError):
            images.png_info(bad)
