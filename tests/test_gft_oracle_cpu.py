"""CPU: oracle/gft.py against OpenCV.  The oracle is what the GPU tests hold sos_corner_min_eigenval / sos_gft_detect to,
bit for bit; these tests pin the oracle itself to cv2.cornerMinEigenVal, cv2.Sobel and cv2.goodFeaturesToTrack.

cv2 is not bit-reproducible everywhere: its SIMD loops leave the last few columns of a row (up to 16) to a scalar tail
that rounds differently, so the corner measure and the Sobel derivatives are compared outside the last TAIL columns.
On sharp images a few interior pixels also differ: cv2's box filter keeps sliding-window sums in double down each column
(add the entering row, subtract the leaving one), which can round a double sum differently from the kernel's direct
three-term sums, and more often the taller the image.  The float32 a, b or c then moves by one unit; through the
cancellation in (a + c) - sqrt((a - c)^2 + b^2) that is many units of a small result (64 measured), but never more than
half a unit of the image's largest measure.  Measured on 849-row images (the panorama height), 3 seeds per width from 64
to 2400: at most 3.4e-5 of the interior pixels of raw noise and 1.4e-6 of median-filtered raw noise differ; blurred
images and median-filtered panoramas (the front-end's input) never differ."""
import cv2
import numpy as np
import pytest

from oracle import gft as ogft

TAIL = 17


def interior_mismatches(got, ref):
    """Pixels outside the tail columns that differ; each may differ by at most one unit in the last place of the image's
    largest measure."""
    w = got.shape[1]
    a, b = got[:, :w - TAIL], ref[:, :w - TAIL]
    assert np.abs(a.astype(np.float64) - b).max() <= np.spacing(np.abs(b).max())
    assert np.abs(got - ref).max() <= 1e-6 * np.abs(ref).max()
    return int((a != b).sum()), a.size


def image(kind, h, w, seed):
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "blur":
        return cv2.GaussianBlur(g, (0, 0), 1.5)
    if kind == "median":
        return cv2.medianBlur(g, 11)
    if kind == "median_pano":            # what the front-end feeds it: 11 x 11 median of a BGR panorama, then gray
        bgr = cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), 1.0)
        return cv2.cvtColor(cv2.medianBlur(bgr, 11), cv2.COLOR_BGR2GRAY)
    if kind == "checker":
        return ((np.indices((h, w)).sum(0) // 8) % 2 * 255).astype(np.uint8)
    if kind == "tiles":                  # 8 x 8 binary tiles: thousands of exactly tied corner strengths
        t = np.kron(rng.integers(0, 2, (h // 8 + 1, w // 8 + 1)), np.ones((8, 8), np.int64))
        return (t[:h, :w] * 200).astype(np.uint8)
    assert kind == "noise"
    return g


WIDTHS = (64, 131, 257, 300, 1000, 2400)


@pytest.mark.parametrize("w", WIDTHS)
@pytest.mark.parametrize("kind,max_rate", [("blur", 0.0), ("median_pano", 0.0), ("median", 5e-6), ("noise", 5e-5)])
def test_corner_measure_vs_cv2(kind, max_rate, w):
    bad = total = 0
    for seed in range(3):
        g = image(kind, 849, w, seed)
        b, t = interior_mismatches(ogft.corner_min_eigenval(g), cv2.cornerMinEigenVal(g, 3, ksize=3))
        bad, total = bad + b, total + t
    assert bad <= max_rate * total, (bad, total)


@pytest.mark.parametrize("h,w", [(1, 1), (1, 7), (2, 2), (2, 9), (7, 1), (9, 2), (1, 300), (300, 2)])
@pytest.mark.parametrize("kind", ["noise", "blur"])
def test_corner_measure_tiny_images(kind, h, w):
    """H or W of 1 or 2: the reflection lands on the pixel itself or its neighbour.  (From W = 3 on, rows shorter than
    cv2's vectors are all tail columns, so only the shapes here are compared with cv2; the GPU tests cover the rest.)"""
    g = image("noise", h, w, h * 100 + w)
    if kind == "blur":
        g = cv2.GaussianBlur(g, (3, 3), 0)
    got, ref = ogft.corner_min_eigenval(g), cv2.cornerMinEigenVal(g, 3, ksize=3)
    assert got.shape == ref.shape and np.array_equal(got, ref)


@pytest.mark.parametrize("h,w", [(97, 131), (300, 257), (849, 2400), (16, 1000)])
def test_sobel_equals_cv2(h, w):
    """dx and the tap-ordered dy of the oracle are cv2.Sobel(scale = s) on every pixel outside the tail columns, on raw noise
    (where rounding differences show up most)."""
    for seed in range(2):
        g = image("noise", h, w, seed)
        dx, dy = ogft.sobel(g)
        s = float(ogft.SCALE)
        DX = cv2.Sobel(g, cv2.CV_32F, 1, 0, ksize=3, scale=s, borderType=cv2.BORDER_REFLECT_101)
        DY = cv2.Sobel(g, cv2.CV_32F, 0, 1, ksize=3, scale=s, borderType=cv2.BORDER_REFLECT_101)
        assert np.array_equal(dx, DX)
        assert np.array_equal(dy[:, :w - TAIL], DY[:, :w - TAIL]), int((dy != DY)[:, :w - TAIL].sum())


def test_fma32_checks_exactness():
    a = np.float32(1.0 + 2.0 ** -23)
    assert ogft.fma32(ogft.SCALE, np.float32(1020), np.float32(0.25)) == np.float32(float(ogft.SCALE) * 1020 + 0.25)
    with pytest.raises(AssertionError):
        ogft.fma32(a, a, np.float32(2.0 ** -60))      # the sum needs more than 53 bits


def cv_gft(g, n, q, d, mask=None):
    pts = cv2.goodFeaturesToTrack(image=g, maxCorners=n, qualityLevel=q, minDistance=d, mask=mask, useHarrisDetector=False)
    return np.zeros((0, 2), np.float32) if pts is None else pts.reshape(-1, 2)


SEL_IMAGES = {
    "blur": lambda: image("blur", 180, 640, 0),
    "noise": lambda: image("noise", 97, 131, 0),
    "checker": lambda: image("checker", 180, 640, 0),
    "tiles": lambda: image("tiles", 180, 640, 0),
}


@pytest.mark.parametrize("name", list(SEL_IMAGES))
@pytest.mark.parametrize("d", [0.0, 0.5, 1.0, 1.5, 2.5, 5.0, 9.0, 25.0])
def test_good_features_equals_cv2(name, d):
    g = SEL_IMAGES[name]()
    eig = cv2.cornerMinEigenVal(g, 3, ksize=3)
    third = np.zeros(g.shape, np.uint8)
    third[:, :g.shape[1] // 3] = 255
    for n in (0, 1, 50, 300, 100_000):
        for q in (0.01, 0.5, 0.9999):
            for mask in (None, third):
                want = cv_gft(g, n, q, d, mask)
                got, nc = ogft.good_features(eig, mask, n, q, d)
                assert got.shape == want.shape and np.array_equal(got, want), (n, q, mask is None, got.shape, want.shape)
                assert nc >= len(got)


def masks_for(shape):
    h, w = shape
    yy, xx = np.indices(shape)
    flat = np.zeros(shape, np.uint8)
    flat[30:70, 120:180] = 255
    border = np.zeros(shape, np.uint8)
    border[:2], border[-2:], border[:, :2], border[:, -2:] = 255, 255, 255, 255
    return {"empty": np.zeros(shape, np.uint8), "flat": flat, "border": border,
            "row_band": ((yy // 13) % 3 == 1).astype(np.uint8) * 255,
            "diagonal": (np.abs(xx - yy * w / h) < 40).astype(np.uint8) * 255}


@pytest.mark.parametrize("mask_name", ["empty", "flat", "border", "row_band", "diagonal"])
def test_good_features_masks_equal_cv2(mask_name):
    g = image("blur", 180, 640, 5)
    g[20:80, 100:200] = 128                       # a flat region: corner measure exactly 0 under the "flat" mask
    m = masks_for(g.shape)[mask_name]
    eig = cv2.cornerMinEigenVal(g, 3, ksize=3)
    for n, q, d in ((300, 0.01, 5.0), (0, 0.01, 2.5), (50, 0.5, 0.0), (100_000, 0.9999, 9.0)):
        want = cv_gft(g, n, q, d, m)
        got, nc = ogft.good_features(eig, m, n, q, d)
        assert np.array_equal(got, want), (n, q, d, got.shape, want.shape)
    if mask_name in ("empty", "flat"):
        assert nc == 0
