"""The tissue-segmentation oracle (oracle/tissue.py) against the installed OpenCV, and the filter rule on small cases."""
import numpy as np
import pytest

from oracle import tissue as tis

cv2 = pytest.importorskip("cv2")


def test_saturation_equals_opencv_for_every_max_min_pair():
    a = np.array([[[v, m, m]] for v in range(256) for m in range(v + 1)], np.uint8)   # 32 896 (max, min) pairs
    assert np.array_equal(tis.saturation(a), cv2.cvtColor(a, cv2.COLOR_RGB2HSV)[..., 1])
    rng = np.random.default_rng(0)
    for _ in range(10):
        h, w = rng.integers(1, 200, 2)
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(tis.saturation(img), cv2.cvtColor(img, cv2.COLOR_RGB2HSV)[..., 1])
        assert np.array_equal(tis.saturation(img), cv2.cvtColor(img, cv2.COLOR_BGR2HSV)[..., 1])


@pytest.mark.parametrize("k", [1, 3, 5, 7])
def test_median_blur_equals_opencv(k):
    rng = np.random.default_rng(k)
    shapes = [(1, 1), (1, 17), (17, 1), (2, 3), (k - 1 or 1, k + 1), (k + 2, k - 1 or 1), (64, 65)]
    shapes += [tuple(rng.integers(1, 150, 2)) for _ in range(8)]
    for h, w in shapes:
        x = rng.integers(0, 256, (h, w), dtype=np.uint8)
        assert np.array_equal(tis.median_blur(x, k), cv2.medianBlur(x, k)), (h, w)


def _otsu_cases(rng):
    yield np.zeros((5, 7), np.uint8)
    yield np.full((1, 1), 93, np.uint8)
    for v in range(0, 256, 15):
        yield np.full((3, 4), v, np.uint8)                                                 # constant
    for i in range(60):
        a, b = rng.integers(0, 256, 2)
        yield np.where(rng.random(tuple(rng.integers(1, 40, 2))) < rng.random(), a, b).astype(np.uint8)   # two-valued
    for i in range(60):
        yield rng.integers(0, 256, (1, 1), dtype=np.uint8)                                 # single pixel
    for i in range(400):
        h, w = rng.integers(1, 120, 2)
        yield np.clip(rng.normal(rng.uniform(-50, 300), rng.uniform(1, 80), (h, w)), 0, 255).astype(np.uint8)   # clipped normal


def test_otsu_threshold_equals_opencv():
    rng = np.random.default_rng(3)
    n = 0
    for x in _otsu_cases(rng):
        t, _ = cv2.threshold(x, 0, 255, cv2.THRESH_BINARY + cv2.THRESH_OTSU)
        assert tis.otsu_threshold(x) == int(t), x
        n += 1
    assert n >= 500


def test_segment_equals_opencv_chain():
    from ss25_hierarchical_multiscale_image_classification_b200 import synthetic
    img = synthetic.make_level(1234, 2, 700, 600)
    blur = cv2.medianBlur(cv2.cvtColor(img, cv2.COLOR_RGB2HSV)[..., 1], 7)
    t, want = cv2.threshold(blur, 0, 255, cv2.THRESH_BINARY + cv2.THRESH_OTSU)
    mask, t_o, blur_o = tis.segment(img, 7)
    assert t_o == int(t) and np.array_equal(blur_o, blur) and np.array_equal(mask, want)
    _, want8 = cv2.threshold(blur, 8, 255, cv2.THRESH_BINARY)
    assert np.array_equal(tis.segment(img, 7, 8)[0], want8)


def test_min_tissue_pixels_is_exact_ceil():
    assert tis.min_tissue_pixels(0.5, 224, 8) == 392
    assert tis.min_tissue_pixels(0, 1792, 8) == 0
    assert tis.min_tissue_pixels(1, 448, 2) == 224 * 224
    assert tis.min_tissue_pixels(0.1, 224, 1) == 5018        # 0.1 is a binary fraction a hair above 1/10: ceil(5017.6...)


def test_filter_rule_on_small_levels():
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (700, 900, 3), dtype=np.uint8)
    m = 4
    tissue = (rng.random((100, 150)) < 0.3).astype(np.uint8) * 255      # smaller than the footprint of the grid (225 x 175)
    p = 448
    for min_tissue in (0, 0.3, 1):
        out = tis.extract_patches_tissue_oracle(img, None, 2, tissue, m, min_tissue=min_tissue, want_images=False)
        need = tis.min_tissue_pixels(min_tissue, p, m)
        want = [(x, y) for x in range(0, 900, 224) for y in range(0, 700, 224)
                if np.count_nonzero(tissue[y // m:(y + p) // m, x // m:(x + p) // m]) >= need]
        assert [tuple(c) for c in out["coords"]] == want
        assert out["candidates"] == 5 * 4
    assert len(tis.extract_patches_tissue_oracle(img, None, 2, tissue, m, min_tissue=0, want_images=False)["coords"]) == 20
    # a candidate whose whole footprint lies beyond the mask counts zero tissue pixels
    assert tis.tissue_count(tissue, 896, 672, p, m) == 0
