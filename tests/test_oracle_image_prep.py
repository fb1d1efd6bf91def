"""Row N5 on the CPU: oracle/image_prep_oracle.py (INTER_AREA resize + rgb2gray in float64) against OpenCV 4.13's
cv2.resize, and the library's vpk_prepared_size against the oracle's size rule (no GPU needed)."""
import numpy as np
import pytest

from oracle import image_prep_oracle as P


def photo(rs, w, h):
    """Smooth content with texture and noise, like a photo."""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    base = 128 + 60 * np.sin(xx / 37.0)[:, :, None] * np.cos(yy / 23.0)[:, :, None] * np.array([1.0, 0.7, -0.5])
    return np.clip(np.round(base + rs.normal(0, 20, (h, w, 3))), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("k", [2, 3, 4, 5, 8])
def test_integer_factors_equal_cv2_exactly(k):
    cv2 = pytest.importorskip("cv2")
    rs = np.random.RandomState(k)
    for img in (photo(rs, 96 * k, 64 * k), rs.randint(0, 256, (40 * k, 56 * k, 3)).astype(np.uint8)):
        h, w = img.shape[:2]
        ref = cv2.resize(img, (w // k, h // k), interpolation=cv2.INTER_AREA)
        np.testing.assert_array_equal(P.resize_area(img, w // k, h // k), ref)


@pytest.mark.parametrize("w,h,target", [(2000, 1333, 640), (1500, 2000, 640), (2048, 1363, 640), (1000, 700, 800)])
def test_generic_factors_match_cv2_to_one_level(w, h, target):
    """cv2 accumulates in float32, the oracle in float64: rare differences of one level."""
    cv2 = pytest.importorskip("cv2")
    img = photo(np.random.RandomState(w + h), w, h)
    W, H = P.prepared_size(w, h, target)
    ref = cv2.resize(img, (W, H), interpolation=cv2.INTER_AREA)
    d = np.abs(P.resize_area(img, W, H).astype(np.int64) - ref.astype(np.int64))
    assert d.max() <= 1
    assert np.mean(d == 0) >= 0.999


def test_prepared_size_of_the_library_equals_the_oracle():
    from vanishing_points_2017_b200 import images
    sizes = [(w, h) for w in (1, 3, 639, 640, 641, 800, 1200, 1333, 2000, 2048, 5000) for h in (1, 2, 3, 480, 640, 901, 1363, 4000)]
    for target in (None, 0, -5, 1, 2, 640, 800, 1000):
        for w, h in sizes:
            assert images.prepared_size(w, h, target) == P.prepared_size(w, h, target), (w, h, target)
    assert images.prepared_size(640, 480, 640) == (640, 480)        # max side == target: no resize
    assert images.prepared_size(300, 200, 640) == (300, 200)        # smaller than the target: never enlarged
    assert images.prepared_size(5000, 3, 640) == (640, 1)
    assert images.prepared_size(2000, 1333, 640) == (640, 427)
    assert images.prepared_size(1200, 900, 800) == (800, 600)


def test_prepared_size_rejects_empty_sides():
    from vanishing_points_2017_b200 import _lib, images
    with pytest.raises(_lib.VpkError):
        images.prepared_size(0, 10, 640)


def test_white_is_one_and_255_after_scaling():
    g = P.prepare(np.full((30, 40, 3), 255, np.uint8), 16)
    assert g.shape == (12, 16)
    assert np.all(g == 1.0) and np.all(g * 255 == 255.0)


def test_gray_is_monotone_and_at_most_one():
    """detect_lsd_lines multiplies by 255 when max <= 1 (evaluation.py:229-231): rgb2gray of uint8 never exceeds 1."""
    v = np.arange(256, dtype=np.uint8)
    for c in range(3):
        img = np.full((1, 256, 3), 255, np.uint8)
        img[0, :, c] = v
        g = P.rgb2gray(img)[0]
        assert np.all(np.diff(g) > 0) and g.max() == 1.0


def test_photos_are_not_enlarged_and_identity_is_exact():
    img = photo(np.random.RandomState(1), 64, 48)
    g = P.prepare(img, None)
    np.testing.assert_array_equal(g, P.rgb2gray(img))
    np.testing.assert_array_equal(P.prepare(img, 640), g)
