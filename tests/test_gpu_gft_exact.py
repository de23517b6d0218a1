"""GPU: Shi-Tomasi detection (csrc/gft.cu) equals oracle/gft.py with no tolerance anywhere.

The corner measure of both entry points (sos_corner_min_eigenval and sos_gft_detect's eig_out) equals
oracle.gft.corner_min_eigenval on every pixel, at shapes that put strips on the generic and the fast path, partial warps
and blocks, and H or W of 1 or 2.  Every corner list equals oracle.gft.good_features run on the GPU's own corner measure:
minimum distances from 0 to 63.5, quality levels that move the per-mask maximum, disjoint and overlapping masks, masks
that change down a column, plateaus of tied strengths, chunk and prefix boundaries of the selection, and the
16 384-candidate limit on both sides."""
import cv2
import numpy as np
import pytest
import torch

from oracle import gft as ogft

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def images(h, w, seed):
    """The corner-measure images: raw noise, 0/255 checkerboards (1- and 3-pixel cells), a single bright pixel, step
    edges (vertical, horizontal, diagonal), a constant image and an 11 x 11 median of a BGR panorama."""
    rng = np.random.default_rng(seed)
    yy, xx = np.indices((h, w))
    dot = np.zeros((h, w), np.uint8)
    dot[h // 2, w // 2] = 255
    bgr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    out = {
        "noise": rng.integers(0, 256, (h, w), dtype=np.uint8),
        "checker1": ((yy + xx) % 2 * 255).astype(np.uint8),
        "checker3": (((yy // 3 + xx // 3) % 2) * 255).astype(np.uint8),
        "dot": dot,
        "steps": np.where(xx >= w // 2, 200, 0).astype(np.uint8) + np.where(yy >= h // 3, 40, 0).astype(np.uint8)
        + np.where(xx + 2 * yy > w // 3, 15, 0).astype(np.uint8),
        "constant": np.full((h, w), 77, np.uint8),
        "median_pano": cv2.cvtColor(cv2.medianBlur(cv2.GaussianBlur(bgr, (0, 0), 1.0), 11), cv2.COLOR_BGR2GRAY),
        "median_noise": cv2.medianBlur(rng.integers(0, 256, (h, w), dtype=np.uint8), 11),
    }
    return list(out), np.stack(list(out.values()))


@pytest.mark.parametrize("h", [3, 4, 5, 15, 16, 17, 18, 33, 849])
@pytest.mark.parametrize("w", [3, 5, 31, 33, 255, 256, 257, 2400])
def test_corner_measure_equals_oracle(ctx, h, w):
    names, g = images(h, w, h * 10_000 + w)
    want = ogft.corner_min_eigenval(g)
    got = ctx.corner_min_eigenval(dev(g)).cpu().numpy()
    # a one-pixel mask keeps every list below the candidate limit (checkerboards tie everywhere); only eig_out is read here
    one = np.zeros((1, h, w), np.uint8)
    one[0, h // 2, w // 2] = 255
    _, _, eig = ctx.gft_detect(dev(g), dev(one), 1, 0.01, 5.0, want_eig=True)
    eig = eig.cpu().numpy()
    for i, name in enumerate(names):
        assert np.array_equal(got[i], want[i]), (name, int((got[i] != want[i]).sum()), np.argwhere(got[i] != want[i])[:4])
        assert np.array_equal(eig[i], want[i]), (name, int((eig[i] != want[i]).sum()))


@pytest.mark.parametrize("h,w", [(1, 1), (1, 5), (2, 2), (2, 300), (5, 1), (300, 2), (1, 2400), (2400, 1), (2, 257)])
def test_corner_measure_tiny_equals_oracle(ctx, h, w):
    names, g = images(h, w, h * 10_000 + w)
    got = ctx.corner_min_eigenval(dev(g)).cpu().numpy()
    want = ogft.corner_min_eigenval(g)
    for i, name in enumerate(names):
        assert np.array_equal(got[i], want[i]), name


# ---- selection ------------------------------------------------------------------------------------------------------
H, W = 180, 640


def sel_images():
    """Three images of one shape, each with a flat patch (corner measure exactly 0) in the last quarter: Gaussian-blurred
    noise (~6 700 candidates at quality 0.01), 8 x 8 binary tiles (thousands of exactly tied strengths) and a median-11
    panorama."""
    rng = np.random.default_rng(7)
    blur = cv2.GaussianBlur(rng.integers(0, 256, (H, W), dtype=np.uint8), (0, 0), 1.2)
    tiles = (np.kron(rng.integers(0, 2, (H // 8 + 1, W // 8 + 1)), np.ones((8, 8), np.int64))[:H, :W] * 200).astype(np.uint8)
    pano = cv2.cvtColor(cv2.medianBlur(cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), (0, 0), 1.0), 11),
                        cv2.COLOR_BGR2GRAY)
    g = np.stack([blur, tiles, pano])
    g[:, 30:90, 3 * W // 4 + 10:3 * W // 4 + 110] = 128
    return g


def disjoint_masks():
    """Pixel-disjoint (one selection launch): a plain column range inside an elevation band, row bands (the mask set
    changes down a column), a diagonal band, a mask over the flat patch only, and an empty mask."""
    yy, xx = np.indices((H, W))
    q = xx // (W // 4)
    m = np.zeros((5, H, W), bool)
    m[0] = (q == 0) & (yy >= 12) & (yy < H - 9)
    m[1] = (q == 1) & ((yy // 13) % 3 == 1)
    m[2] = (q == 2) & (np.abs((xx - W // 2) - yy * (W // 4) / H) < 25)
    m[3] = (yy >= 40) & (yy < 80) & (xx >= 3 * W // 4 + 20) & (xx < 3 * W // 4 + 100)
    assert m.sum(0).max() == 1
    return m.astype(np.uint8) * 255


def overlapping_masks():
    """Overlapping (one selection launch per mask): column ranges that share 40 columns, a row band across all of them and
    the whole image."""
    yy, xx = np.indices((H, W))
    m = np.zeros((5, H, W), bool)
    for k in range(3):
        m[k] = (xx >= k * W // 3 - 40) & (xx < (k + 1) * W // 3)
    m[3] = (yy >= 50) & (yy < 120)
    m[4] = True
    return m.astype(np.uint8) * 255


def check_lists(ctx, g, masks, N, q, d):
    xy, cnt, eig = ctx.gft_detect(dev(g), None if masks is None else dev(masks), N, q, d, want_eig=True)
    xy, cnt, eig = xy.cpu().numpy(), cnt.cpu().numpy(), eig.cpu().numpy()
    ms = [None] if masks is None else list(masks)
    stats = []
    for b in range(len(g)):
        assert np.array_equal(eig[b], ogft.corner_min_eigenval(g[b]))
        for m, mask in enumerate(ms):
            want, n_cand = ogft.good_features(eig[b], mask, N, q, d)
            got = xy[b, m, :cnt[b, m]]
            assert cnt[b, m] == len(want) and np.array_equal(got, want), (b, m, N, q, d, int(cnt[b, m]), len(want))
            stats.append((n_cand, len(want)))
    return xy, cnt, stats


D_VALUES = [0.0, 0.5, 1.0, 1.5, 2.5, 5.0, 9.0, 25.0, 63.5]


@pytest.mark.parametrize("d", D_VALUES)
@pytest.mark.parametrize("overlap", [False, True])
def test_lists_equal_oracle(ctx, d, overlap):
    g = sel_images()
    masks = overlapping_masks() if overlap else disjoint_masks()
    for q in (0.01, 0.5, 0.9999):
        xy, cnt, _ = check_lists(ctx, g, masks, 300, q, d)
        if overlap and q == 0.01:
            # one launch per mask gives the lists of single-mask calls
            for m in range(len(masks)):
                xs, cs = ctx.gft_detect(dev(g), dev(masks[m:m + 1]), 300, q, d)
                assert np.array_equal(cs.cpu().numpy()[:, 0], cnt[:, m])
                for b in range(len(g)):
                    assert np.array_equal(xs.cpu().numpy()[b, 0, :cnt[b, m]], xy[b, m, :cnt[b, m]])


def test_32_masks(ctx):
    g = sel_images()
    xx = np.indices((H, W))[1]
    masks = np.stack([(xx // (W // 32) == k) for k in range(32)]).astype(np.uint8) * 255
    for d in (0.0, 5.0):
        check_lists(ctx, g, masks, 40, 0.01, d)


@pytest.mark.parametrize("N,d", [(5000, 1.0), (5000, 1.5), (100_000, 0.0), (300, 5.0), (300, 25.0), (1200, 9.0)])
def test_long_lists_equal_oracle(ctx, N, d):
    """One list of ~6 700 candidates: more than 2 048 decided candidates (chunk boundary, N = 5000), the histogram prefix
    holding enough (N = 300, d = 5) and running dry (N = 300, d = 25), minDistance < 1 with more corners asked for than
    there are candidates."""
    g = sel_images()
    _, _, stats = check_lists(ctx, g, None, N, 0.01, d)
    n_cand, n_out = stats[0]
    assert n_cand > 6000
    if N == 5000:
        assert n_out > 2048
    if (N, d) == (300, 25.0):
        assert n_out < 300            # the prefix ran dry: the whole list was decided


def test_plateau_rescan(ctx):
    """8 x 8 tiles: thousands of tied strengths ordered by pixel index, and at d = 9 / 25 candidates with more stronger
    neighbours than the selection remembers (the rank-image rescan)."""
    g = sel_images()[1:2]
    for d in (2.5, 9.0, 25.0):
        _, _, stats = check_lists(ctx, g, None, 2000, 0.01, d)
        assert stats[0][0] > 1500


def prefix_mask(eig, q, target):
    """A mask whose list has exactly `target` candidates: a raster-order prefix of the image plus the pixel of the image's
    largest measure (so the mask's maximum, and the threshold, are those of the whole image)."""
    cand = np.sort(ogft.candidates(eig, None, q))
    amax = int(np.argmax(eig))
    for t in range(target - 1, target + 2):
        mask = np.zeros(eig.size, np.uint8)
        mask[:cand[t - 1] + 1] = 255
        mask[amax] = 255
        mask = mask.reshape(eig.shape)
        if len(ogft.candidates(eig, mask, q)) == target:
            return mask
    raise AssertionError("no prefix mask with %d candidates" % target)


def test_candidate_limit(ctx):
    """16 384 candidates in one list are selected; 16 385 are refused with SosError (with one mask and with several)."""
    from vo_single_camera_sos_b200._lib import SosError
    g = np.random.default_rng(9).integers(0, 256, (400, 1000), dtype=np.uint8)
    eig = ctx.corner_min_eigenval(dev(g)).cpu().numpy()
    assert len(ogft.candidates(eig, None, 0.01)) > 20_000
    ok, over = prefix_mask(eig, 0.01, 16384), prefix_mask(eig, 0.01, 16385)
    xy, cnt = ctx.gft_detect(dev(g), dev(ok[None]), 500, 0.01, 5.0)
    want, n_cand = ogft.good_features(eig, ok, 500, 0.01, 5.0)
    assert n_cand == 16384 and int(cnt[0, 0]) == len(want) and np.array_equal(xy.cpu().numpy()[0, 0, :len(want)], want)
    for masks in (over[None], np.stack([ok, over]), np.stack([over, 255 - over])):
        with pytest.raises(SosError):
            ctx.gft_detect(dev(g), dev(masks), 500, 0.01, 5.0)
    with pytest.raises(SosError):
        ctx.gft_detect(dev(g), None, 500, 0.01, 5.0)        # no mask: 26 k candidates


def test_max_corners_must_be_positive(ctx):
    """cv2 reads maxCorners <= 0 as "no limit"; sos_gft_detect sizes out_xy by it and refuses it."""
    from vo_single_camera_sos_b200._lib import SosError, check
    g = dev(sel_images())
    xy = torch.zeros((3, 1, 1, 2), dtype=torch.float32, device=g.device)
    cnt = torch.zeros((3, 1), dtype=torch.int32, device=g.device)
    for n in (0, -1):                  # straight to the C entry point (the wrapper cannot allocate a negative size)
        with pytest.raises(SosError):
            check(ctx.lib.sos_gft_detect(ctx._h, g.data_ptr(), None, 3, H, W, 1, n, 0.01, 5.0, xy.data_ptr(),
                                         cnt.data_ptr(), None))
    with pytest.raises(SosError):
        ctx.gft_detect(g, None, 0, 0.01, 5.0)


def test_one_bucket_feature_front_refuses_overflow(ctx):
    """A one-bucket FeatureFront on a textured 849 x 2400 panorama (>100 k candidates) raises instead of returning fewer
    corners."""
    from vo_single_camera_sos_b200._lib import SosError
    from vo_single_camera_sos_b200.features import FeatureFront
    rng = np.random.default_rng(4)
    rows, cols = 849, 2400
    pano = cv2.GaussianBlur(rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8), (0, 0), 1.0)
    gray = cv2.cvtColor(cv2.medianBlur(pano, 11), cv2.COLOR_BGR2GRAY)
    assert len(ogft.candidates(ogft.corner_min_eigenval(gray), None, 0.01)) > 16384
    full = np.full((1, rows, cols), 255, np.uint8)
    front = FeatureFront(ctx, full, full, corners_per_bucket=100, max_feat_per_view=100)
    with pytest.raises(SosError):
        front.detect(dev(np.stack([pano, pano])[None]))
