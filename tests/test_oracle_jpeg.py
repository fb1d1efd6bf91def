"""Row N6 on the CPU: the JPEG oracle's two decoders (cv2 and PIL, each with its own libjpeg-turbo) agree bit for bit
on the corpus, and vpk_jpeg_info (host only) reads every corpus file's size and components and the reason for every
refused file."""
import numpy as np
import pytest

from oracle import jpeg_oracle as J
from vanishing_points_2017_b200 import images

CORPUS = J.corpus(large=True)
REFUSED = J.refused()


@pytest.mark.parametrize("name,blob", CORPUS, ids=[c[0] for c in CORPUS])
def test_cv2_and_pil_decode_identically(name, blob):
    a, b = J.decode(blob), J.decode_pil(blob)
    assert a.shape == b.shape and a.dtype == np.uint8
    np.testing.assert_array_equal(a, b)


def test_exif_orientation_is_ignored_by_the_reference():
    blob = dict(CORPUS)["pil_exif_orientation6_257x191"]
    assert J.decode(blob).shape == (191, 257, 3)


def test_info_reads_size_components_and_support_of_the_corpus():
    info = images.jpeg_info([b for _, b in CORPUS])
    for (name, blob), (w, h, c, s) in zip(CORPUS, info):
        ref = J.decode(blob)
        assert s == J.OK, name
        assert (h, w) == ref.shape[:2], name
        assert c == (1 if ref.ndim == 2 else 3), name


def test_info_gives_the_reason_of_every_refused_file():
    info = images.jpeg_info([b for _, b, _ in REFUSED])
    for (name, _, why), (w, h, c, s) in zip(REFUSED, info):
        assert s == why, (name, s, why)


def test_info_accepts_arrays_and_rejects_other_input():
    blob = CORPUS[0][1]
    assert images.jpeg_info([np.frombuffer(blob, np.uint8)]) == images.jpeg_info([blob])
    assert images.jpeg_info([]) == []
    for bad in (blob, [np.zeros((2, 2), np.uint8)], [np.zeros(4, np.int32)]):
        with pytest.raises(ValueError):
            images.jpeg_info(bad)
