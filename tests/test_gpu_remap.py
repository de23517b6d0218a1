"""GPU parity: LUT pack + remap kernels vs cv2.remap (the reference's call) — bit-exact, bar is 1 LSB."""
import numpy as np
import pytest
import torch

from conftest import load_golden, sub
from oracle import geometry, remap

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(params=["aligned", "offset"])
def place(request):
    """Every test of this file runs its remap sources at two placements, which select the kernel csrc/remap.cu launches: an
    allocation's own (aligned) address takes the batch-looped kernel with TMA-staged LUT tiles for 3 channels whose rows are
    a multiple of 4 bytes; one byte into a fresh buffer (offset) takes the generic kernel, as do 1 and 4 channels and every
    other row size.  Returns (to_device, expected kernel name for a source of width w and ch channels)."""
    offset = request.param == "offset"

    def to_device(a):
        a = np.ascontiguousarray(a)
        if not offset:
            return dev(a)
        t = torch.empty(a.size + 1, dtype=torch.uint8, device="cuda")[1:].view(a.shape)
        t.copy_(torch.from_numpy(a))
        return t

    def kernel(w, ch):
        return "remap3b_kernel" if ch == 3 and w % 4 == 0 and not offset else "remap_kernel"
    return to_device, kernel


def remap_on(ctx, kernel, src, lut, **kw):
    """ctx.remap, asserting that it launched `kernel` exactly once."""
    ctx.profile_begin()
    out = ctx.remap(src, lut, **kw)
    assert [name for name, _ in ctx.profile_end()] == [kernel]
    return out


def test_golden_panoramas(ctx, place):
    to_device, kernel = place
    g = load_golden("remap.npz")
    img = to_device(g["img"][None])
    k3 = kernel(g["img"].shape[1], 3)
    luts = []
    for name in ("top", "bot"):
        lut = ctx.lut_pack(dev(g[f"map_x32_{name}"]), dev(g[f"map_y32_{name}"]), g["img"].shape[:2], mask=dev(g[f"mask_{name}"]))
        spec = remap.lut_pack_spec(g[f"map_x32_{name}"], g[f"map_y32_{name}"], g["img"].shape[:2], g[f"mask_{name}"])
        assert np.array_equal(lut.cpu().numpy().view(np.uint64), spec)
        luts.append(lut)
    out = remap_on(ctx, k3, img, torch.stack(luts)).cpu().numpy()
    assert np.array_equal(out[0, 0], g["pano_top"]) and np.array_equal(out[0, 1], g["pano_bot"])
    out = remap_on(ctx, k3, img, torch.stack(luts), border=(250, 60, 30), background=(90, 200, 10)).cpu().numpy()
    assert np.array_equal(out[0, 0], g["pano_colour_top"]) and np.array_equal(out[0, 1], g["pano_colour_bot"])
    # single channel, no mask: the mirror mask remapped (panorama.py:534)
    for i, name in enumerate(("top", "bot")):
        lut = ctx.lut_pack(dev(g[f"map_x32_{name}"]), dev(g[f"map_y32_{name}"]), g["img"].shape[:2])
        out = remap_on(ctx, kernel(g["img"].shape[1], 1), to_device(g[f"mask_{name}"][None]), lut).cpu().numpy()
        assert np.array_equal(out[0, 0], g[f"pano_of_mask_{name}"])


@pytest.mark.parametrize("ch", [1, 3, 4])
@pytest.mark.parametrize("shape", [((97, 131), (120, 203)), ((64, 64), (33, 128)), ((240, 320), (61, 1200))])
def test_adversarial_maps_vs_cv2(ctx, place, ch, shape):
    to_device, kernel = place
    (H, W), (R, C) = shape
    rng = np.random.default_rng(H * 3 + C + ch)
    src = rng.integers(0, 256, (2, H, W, ch), dtype=np.uint8)
    mx = rng.uniform(-3, W + 3, (R, C))
    my = rng.uniform(-3, H + 3, (R, C))
    mx[rng.random((R, C)) < 0.05] = np.nan
    my[rng.random((R, C)) < 0.05] = np.nan
    mx[0, :10] = [0, 0.5 / 32, 1.5 / 32, 2.5 / 32, W - 1, W - 1 + 0.5 / 32, W - 0.5, -1, -0.999, 1e20]
    my[0, :10] = [0, 0.5 / 32, 1.5 / 32, 2.5 / 32, H - 1, H - 1, H - 0.5, -1, -0.5, 3]
    mask = (rng.random((H, W)) < 0.7).astype(np.uint8) * 255
    border = (7, 9, 11, 13)[:ch]
    bg = (200, 100, 50, 25)[:ch]
    # float64 maps: the kernel performs the reference's float64 -> float32 cast (panorama.py:291-292)
    lut = ctx.lut_pack(dev(mx), dev(my), (H, W), mask=dev(mask))
    out = remap_on(ctx, kernel(W, ch), to_device(src), lut, border=border, background=bg).cpu().numpy()
    for b in range(2):
        s = src[b] if ch > 1 else src[b, :, :, 0]
        ref = remap.remap_reference(remap.masked_image(s, mask, bg), mx, my, border=border)
        got = out[b, 0] if ch > 1 else out[b, 0, :, :, 0]
        assert np.array_equal(got, ref)


def test_full_size_c2_against_cv2(ctx, place):
    """2048 x 2048 source, 2400-wide panorama LUT built on the device from random-ish GUM parameters."""
    g = load_golden("remap.npz")
    W = H = 2048
    p = sub(g, "gum_top_")
    s = W / 320.0
    p.update(gamma1=p["gamma1"] * s, gamma2=p["gamma2"] * s, u_center=W / 2 + 3.1, v_center=H / 2 - 2.2)
    pano = geometry.pano_geometry(2400, np.deg2rad(20.0), np.deg2rad(-35.0))
    lo, hi = np.deg2rad(-30.0), np.deg2rad(14.0)
    mx, my = ctx.lut_build(geometry.gum_vector(p), pano["rows"], pano["cols"], pano["cyl_height_max"], pano["cyl_height_min"], lo, hi)
    ru, rv = geometry.lut_build(p, pano["rows"], pano["cols"], pano["cyl_height_max"], pano["cyl_height_min"], lo, hi)
    mxh, myh = mx.cpu().numpy(), my.cpu().numpy()
    assert np.array_equal(np.isnan(mxh), np.isnan(ru))
    ok = ~np.isnan(ru)
    assert 0.3 < ok.mean() < 1.0
    assert np.max(np.abs(mxh[ok] - ru[ok])) < 1e-6 and np.max(np.abs(myh[ok] - rv[ok])) < 1e-6
    rng = np.random.default_rng(9)
    img = rng.integers(0, 256, (H // 16, W // 16, 3), dtype=np.uint8).repeat(16, 0).repeat(16, 1)
    img = (img.astype(np.int16) + rng.integers(-30, 31, img.shape)).clip(0, 255).astype(np.uint8)
    yy, xx = np.mgrid[:H, :W]
    r = np.hypot(xx - p["u_center"], yy - p["v_center"])
    mask = ((r < 0.48 * H) & (r > 0.2 * H)).astype(np.uint8) * 255
    lut = ctx.lut_pack(mx, my, (H, W), mask=dev(mask))
    to_device, kernel = place
    out = remap_on(ctx, kernel(W, 3), to_device(np.stack([img, img[::-1].copy()])), lut).cpu().numpy()
    ref = remap.remap_reference(remap.masked_image(img, mask), mxh, myh)
    assert np.array_equal(out[0, 0], ref)
    assert np.array_equal(out[1, 0], remap.remap_reference(remap.masked_image(img[::-1].copy(), mask), mxh, myh))
    assert (out[0, 0] > 0).mean() > 0.2
