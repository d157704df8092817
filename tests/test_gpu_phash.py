"""GPU parity of the perceptual hash against Pillow + scipy (the libraries imagehash.phash calls)."""
import numpy as np
import pytest

from facet_b200.synth import synth_image_bgr

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape", [(683, 1024), (1024, 683), (97, 131), (400, 600), (33, 35), (2000, 3000)])
def test_phash_matches_pillow_scipy(shape):
    from facet_b200 import ops
    from oracle import phash as op
    h, w = shape
    imgs = np.stack([synth_image_bgr(i, h, w) for i in range(6)])
    hashes, small, dct = ops.phash(imgs, debug=True)
    hexes = ops.phash_hex(imgs)
    for i in range(len(imgs)):
        ref_small, ref_low, ref_val = op.phash_parts(imgs[i])
        assert np.array_equal(small[i], ref_small), "32x32 luma thumbnail must be bit-exact with Pillow"
        np.testing.assert_allclose(dct[i], ref_low, rtol=1e-9, atol=1e-6)
        # bits can only differ where a coefficient sits within float64 noise of the median
        med = np.median(ref_low)
        safe = np.abs(ref_low - med).flatten() > 1e-6
        got_bits = np.array([(int(hashes[i]) >> (63 - k)) & 1 for k in range(64)])
        want_bits = np.array([(ref_val >> (63 - k)) & 1 for k in range(64)])
        assert np.array_equal(got_bits[safe], want_bits[safe])
        if safe.all():
            assert hexes[i] == op.phash_hex(imgs[i])
    # RGB-order input gives the same hash
    assert np.array_equal(ops.phash(np.ascontiguousarray(imgs[..., ::-1]), rgb_order=True), hashes)


def test_phash_tensor_core_route_is_exact():
    from facet_b200 import ops
    # width 16 000: the 204 KB coefficient matrix leaves shared memory for one image stage, so the streaming schedule runs
    for (h, w) in [(683, 1024), (400, 608), (2000, 3008), (48, 16000)]:
        imgs = np.stack([synth_image_bgr(40 + i, h, w) for i in range(3)])
        a = ops.phash(imgs, debug=True, tensor_cores=True)
        b = ops.phash(imgs, debug=True, tensor_cores=False)
        assert np.array_equal(a[1], b[1]) and np.array_equal(a[0], b[0])


def test_luma_plane_from_technical_pass():
    """fb_tech_stats_luma: same statistics, plus Pillow's luma plane that phash() can consume."""
    import torch
    from PIL import Image
    from facet_b200 import ops
    for (h, w, rgb) in [(200, 640, False), (683, 1024, True), (97, 131, False)]:
        imgs = np.stack([synth_image_bgr(50 + i, h, w) for i in range(3)])
        if rgb:
            imgs = np.ascontiguousarray(imgs[..., ::-1])
        t = ops.to_device_u8(imgs)
        luma = torch.zeros((3, h, w), dtype=torch.uint8, device="cuda")
        a = ops.tech_stats_raw(t, rgb_order=rgb, luma_out=luma)
        b = ops.tech_stats_raw(t, rgb_order=rgb)
        for x, y in zip(a, b):
            assert torch.equal(x, y)
        for i in range(3):
            rgb_img = imgs[i] if rgb else np.ascontiguousarray(imgs[i][..., ::-1])
            want = np.asarray(Image.fromarray(rgb_img).convert("L"))
            assert np.array_equal(luma[i].cpu().numpy(), want)
        if ops.phash_uses_luma_plane(h, w):
            assert np.array_equal(ops.phash(t, rgb_order=rgb, luma=luma), ops.phash(t, rgb_order=rgb))


def test_phash_24mp():
    from facet_b200 import ops
    from oracle import phash as op
    img = synth_image_bgr(4, 4000, 6000)
    assert ops.phash_hex(img[None])[0] == op.phash_hex(img)
