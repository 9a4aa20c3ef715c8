"""CPU: the rectangle table of the rolling ball's banded pass (csrc/morph.cu build_bands, dumped through
dc_debug_rolling_ball_bands) against cv2's own ellipse, and a numpy model of the banded kernel
(tests/rb_banded_model.py) against OpenCV's erode / dilate with the reference's structuring element
(utils/data_loader.py:17-19).  No GPU needed; tests/test_gpu_rolling_ball_banded.py pins the kernel itself."""
import numpy as np
import pytest

from rb_banded_model import band_pass, load_bands


def cv2_rects(k: int) -> list[tuple[int, int, int, int]]:
    """(ya, yb, xa, xb) of cv2's k x k ellipse relative to the anchor, widest chord first."""
    import cv2
    an = k // 2
    se = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))
    lo = np.array([np.flatnonzero(r)[0] for r in se]) - an
    hi = np.array([np.flatnonzero(r)[-1] for r in se]) - an
    rects = []
    for a, b in sorted(set(zip(lo.tolist(), hi.tolist())), key=lambda t: t[0] - t[1]):
        ys = np.flatnonzero((lo <= a) & (hi >= b)) - an
        assert np.array_equal(ys, np.arange(ys[0], ys[-1] + 1)), f"k={k}: band of [{a},{b}] is not contiguous"
        rects.append((int(ys[0]), int(ys[-1]), int(a), int(b)))
    return rects


@pytest.mark.parametrize("k", list(range(1, 401)) + [511, 777, 1023, 1500, 2046, 2047])
def test_bands_match_cv2_ellipse(k):
    import cv2
    bands = load_bands(k)
    assert bands["k"] == k
    assert bands["rects"] == cv2_rects(k)
    an = k // 2
    se = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))
    union = np.zeros((k, k), np.uint8)
    for ya, yb, xa, xb in bands["rects"]:
        assert ya <= 0 <= yb and xa <= 0 <= xb, "every rectangle contains the anchor"
        union[ya + an:yb + an + 1, xa + an:xb + an + 1] = 1
    np.testing.assert_array_equal(union, se)


@pytest.mark.parametrize("k,K", [(50, 16), (174, 52), (300, 89), (511, 150), (1023, 300), (2047, 600)])
def test_band_counts(k, K):
    assert load_bands(k)["K"] == K


def test_bands_refuse_out_of_range():
    from unet_dc_segmentation_b200 import _lib
    import ctypes as C
    lib = _lib.load()
    buf = (C.c_int * 8192)()
    for k in (0, 2048):
        assert lib.dc_debug_rolling_ball_bands(k, buf, 8192) == _lib.DC_EINVAL
    assert lib.dc_debug_rolling_ball_bands(300, buf, 10) == _lib.DC_EINVAL       # buffer too small


def _frame(rs, H, W):
    img = rs.randint(0, 256, (H, W)).astype(np.uint8)
    img[H // 3:H // 2 + 1, W // 4:W // 2 + 1] //= 4
    return img


CASES = [(1, (37, 41), 1), (2, (37, 41), 4), (3, (20, 33), 3), (4, (19, 22), 16),
         (50, (70, 93), 4), (50, (70, 93), 16), (174, (90, 181), 8), (175, (61, 203), 16), (176, (40, 177), 2),
         (300, (50, 311), 16), (300, (1, 517), 1), (300, (517, 1), 4), (511, (33, 47), 16), (511, (45, 530), 4),
         (175, (9, 7), 1), (176, (1, 1), 16), (50, (1, 61), 2), (50, (61, 1), 16)]


@pytest.mark.parametrize("radius,shape,T", CASES)
def test_kernel_model_matches_cv2(radius, shape, T):
    import cv2
    rs = np.random.RandomState(radius * 1000 + shape[0] * 7 + shape[1])
    img = _frame(rs, *shape)
    bands = load_bands(radius)
    se = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (radius, radius))
    np.testing.assert_array_equal(band_pass(img, bands, False, T), cv2.erode(img, se))
    np.testing.assert_array_equal(band_pass(img, bands, True, T), cv2.dilate(img, se))


def test_limits():
    from unet_dc_segmentation_b200.morphology import max_radius, tiled_max_radius
    assert max_radius() == 2047
    assert tiled_max_radius() == 170
