"""Row N8 on the CPU: vpk_file_info (host only) on the JPEG, PNG and PGM corpora interleaved and on every refused
file, the PGM oracle's two decoders (cv2 and PIL) on the PGM corpus, the gray INTER_AREA oracle against cv2.resize,
and the gray rules of oracle/files_oracle.prepare_file."""
import numpy as np
import pytest

from oracle import files_oracle as F
from oracle import image_prep_oracle as P
from oracle import jpeg_oracle as J
from oracle import png_oracle as G
from vanishing_points_2017_b200 import _lib, images

PGM_CORPUS = F.pgm_corpus()


def interleaved():
    """(name, file, format) of the three corpora, dealt round-robin"""
    parts = [[(n, b, F.JPEG) for n, b in J.corpus(large=False)], [(n, b, F.PNG) for n, b in G.corpus(large=False)],
             [(n, b, F.PGM) for n, b, _ in PGM_CORPUS]]
    out = []
    for k in range(max(len(p) for p in parts)):
        out += [p[k] for p in parts if k < len(p)]
    return out


@pytest.mark.parametrize("name,blob,img", PGM_CORPUS, ids=[c[0] for c in PGM_CORPUS])
def test_cv2_and_pil_decode_the_pgm_corpus_identically(name, blob, img):
    a, b = F.decode_pgm(blob), F.decode_pgm_pil(blob)
    assert a.dtype == np.uint8 and a.shape == img.shape
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(a, img)


def test_file_info_reads_format_size_channels_and_support_of_the_corpora():
    files = interleaved()
    assert {f for _, _, f in files} == {F.JPEG, F.PNG, F.PGM}
    info = images.file_info([b for _, b, _ in files])
    for (name, blob, fmt), (f, w, h, c, s) in zip(files, info):
        ref = F.decode(blob)
        assert (f, s) == (fmt, 0), name
        assert (h, w) == ref.shape[:2], name
        assert c == (1 if ref.ndim == 2 else 3), name


def test_file_info_gives_the_reason_of_every_refused_file():
    refused = [(n, b, fmt, why) for fmt, files in ((F.PGM, F.pgm_refused()), (F.JPEG, J.refused()), (F.PNG, G.refused()))
               for n, b, why in files]
    # a file too damaged to show its format's leading bytes is of unknown format; one of another format is not refused
    refused = [(n, b, fmt, why) if F.sniff(b) == fmt else (n, b, F.UNKNOWN, 1) for n, b, fmt, why in refused
               if F.sniff(b) in (fmt, F.UNKNOWN)]
    unknown = [("empty", b"", F.UNKNOWN, 1), ("text", b"hello", F.UNKNOWN, 1), ("bmp", b"BM" + bytes(60), F.UNKNOWN, 1),
               ("jpeg_without_marker", b"\xff\xd8\x00\x00", F.UNKNOWN, 1), ("p8", b"P8\n1 1\n255\n\x00", F.UNKNOWN, 1)]
    files = refused + unknown
    info = images.file_info([b for _, b, _, _ in files])
    for (name, _, fmt, why), (f, w, h, c, s) in zip(files, info):
        assert (f, s) == (fmt, why), (name, f, s)
    names = {n: i for (n, _, _, _), i in zip(files, info)}
    assert names["maxval_100"][1:4] == (20, 10, 1) and names["truncated"][1:4] == (20, 10, 1)
    assert len(_lib.PGM_REASONS) == F.PGM_MALFORMED + 1 and _lib.FILE_PGM == F.PGM


def test_file_info_accepts_arrays_and_rejects_other_input():
    blob = PGM_CORPUS[4][1]
    assert images.file_info([np.frombuffer(blob, np.uint8)]) == images.file_info([blob])
    assert images.file_info([]) == []
    for bad in (blob, [np.zeros((2, 2), np.uint8)], [np.zeros(4, np.int32)]):
        with pytest.raises(ValueError):
            images.file_info(bad)


def photo(rs, w, h):
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    base = 128 + 60 * np.sin(xx / 37.0) * np.cos(yy / 23.0)
    return np.clip(np.round(base + rs.normal(0, 20, (h, w))), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("k", [2, 3, 4, 5, 8])
def test_gray_integer_factors_equal_cv2_exactly(k):
    cv2 = pytest.importorskip("cv2")
    rs = np.random.RandomState(k)
    ties = np.tile(np.array([[0, 1], [1, 0]], np.uint8), (24 * k, 30 * k))          # 2 x 2 blocks of sum 2: ties
    for img in (photo(rs, 96 * k, 64 * k), rs.randint(0, 256, (40 * k, 56 * k)).astype(np.uint8), ties):
        h, w = img.shape
        ref = cv2.resize(img, (w // k, h // k), interpolation=cv2.INTER_AREA)
        np.testing.assert_array_equal(F.resize_area(img, w // k, h // k), ref)


@pytest.mark.parametrize("w,h,target", [(2000, 1333, 640), (1500, 2000, 640), (2048, 1363, 640), (1000, 700, 800)])
def test_gray_generic_factors_match_cv2_to_one_level(w, h, target):
    """cv2 accumulates in float32, the oracle in float64: rare differences of one level."""
    cv2 = pytest.importorskip("cv2")
    img = photo(np.random.RandomState(w + h), w, h)
    W, H = P.prepared_size(w, h, target)
    ref = cv2.resize(img, (W, H), interpolation=cv2.INTER_AREA)
    d = np.abs(F.resize_area(img, W, H).astype(np.int64) - ref.astype(np.int64))
    assert d.max() <= 1
    assert np.mean(d == 0) >= 0.999


def test_gray_resize_is_the_rgb_rule_on_one_channel():
    img = photo(np.random.RandomState(3), 301, 211)
    for W, H in ((301, 211), (150, 105), (100, 70), (97, 68)):
        rgb = P.resize_area(np.dstack([img] * 3), W, H)
        np.testing.assert_array_equal(F.resize_area(img, W, H), rgb[:, :, 0])


def test_prepare_file_follows_the_reference_gray_rules():
    img = photo(np.random.RandomState(5), 900, 600)
    g, lsd = F.prepare_file(F.write_pgm(img), 640)
    assert g.dtype == np.uint8 and g.shape == (427, 640)
    np.testing.assert_array_equal(lsd, g.astype(np.float64))            # max > 1: the values themselves
    bits = (img > 128).astype(np.uint8)
    g, lsd = F.prepare_file(F.write_pgm(bits), None)
    np.testing.assert_array_equal(g, bits)
    np.testing.assert_array_equal(lsd, bits * 255.0)                      # max <= 1: times 255
    bits[7, 9] = 2
    g, lsd = F.prepare_file(F.write_pgm(bits), None)
    np.testing.assert_array_equal(lsd, bits.astype(np.float64))
    rgb = np.dstack([img, img[::-1], img[:, ::-1]])
    g, lsd = F.prepare_file(G.encode_cv2(rgb), 640)
    np.testing.assert_array_equal(g, P.prepare(rgb, 640))
    np.testing.assert_array_equal(lsd, g * 255)
