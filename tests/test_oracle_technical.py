"""Pin the NumPy oracle: (1) against golden outputs of the reference's own
analyzers (tests/golden/technical_golden.json), (2) against the installed cv2
for the integer stages, exhaustively over all 2^24 colours for gray/HSV."""
import math

import numpy as np
import pytest

from conftest import approx_rel
from facet_b200.synth import synth_image_bgr
from oracle import technical_np as onp

INT_KEYS = ("shadow_clipped", "highlight_clipped", "is_silhouette", "is_monochrome")


def _cmp_dict(got, want, rel, abs_=2e-4):
    for k, w in want.items():
        g = got[k]
        if k == "histogram_bytes":
            gb = g.hex() if isinstance(g, (bytes, bytearray)) else g
            wb = w.hex() if isinstance(w, (bytes, bytearray)) else w
            assert gb == wb, "histogram_bytes differ"
        elif k in INT_KEYS:
            assert int(g) == int(w), k
        else:
            assert approx_rel(float(g), float(w), rel=rel, abs_=abs_), (k, g, w)


def test_oracle_matches_reference_golden(technical_golden):
    for rec in technical_golden["cases"]:
        img = synth_image_bgr(rec["index"], rec["height"], rec["width"])
        m = onp.all_metrics(img, mono_threshold=0.10)
        st = m["stats"]
        assert st["hist256"].tolist() == rec["hist256"]
        nzb = np.flatnonzero(st["hs_hist"].ravel())
        assert nzb.tolist() == rec["hs_nonzero_bins"]
        assert st["hs_hist"].ravel()[nzb].tolist() == rec["hs_nonzero_counts"]
        assert st["sum_lap"] == rec["sum_lap"]
        assert st["sum_lap_sq"] == rec["sum_lap_sq"]
        assert st["sum_abs_noise"] == rec["sum_abs_noise"]
        assert approx_rel(onp.laplacian_variance(st), rec["laplacian_variance"], rel=1e-9, abs_=1e-9)
        for name in ("sharpness", "color", "histogram", "monochrome", "dynamic_range", "noise", "contrast"):
            _cmp_dict(m[name], rec[name], rel=1e-5)


def test_gray_hsv_exhaustive_vs_cv2():
    cv2 = pytest.importorskip("cv2")
    # all 2^24 BGR triples as a 4096x4096 image
    v = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([(v & 255), (v >> 8) & 255, (v >> 16) & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)
    assert np.array_equal(onp.gray_u8(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))
    h, s, vv = onp.hsv_u8(img)
    ref = cv2.cvtColor(img, cv2.COLOR_BGR2HSV)
    assert np.array_equal(h.astype(np.uint8), ref[..., 0])
    assert np.array_equal(s.astype(np.uint8), ref[..., 1])
    assert np.array_equal(vv.astype(np.uint8), ref[..., 2])
    assert int(h.max()) <= 179


def test_stencils_vs_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    for (h, w) in [(2, 2), (2, 9), (7, 3), (64, 50), (201, 333)]:
        g = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
        lap = cv2.Laplacian(g, cv2.CV_64F)
        assert np.array_equal(onp.laplacian_i32(g).astype(np.float64), lap)
        M = np.array([[1, -2, 1], [-2, 4, -2], [1, -2, 1]])
        nz = cv2.filter2D(g.astype(np.float64), -1, M)
        assert np.array_equal(onp.immerkaer_i32(g).astype(np.float64), nz)


def test_percentile_matches_numpy():
    rng = np.random.default_rng(9)
    for n in (4, 5, 100, 1001, 65536):
        for trial in range(4):
            if trial == 0:
                g = rng.integers(0, 256, size=n, dtype=np.uint8)
            elif trial == 1:
                g = rng.integers(100, 104, size=n, dtype=np.uint8)
            elif trial == 2:
                g = np.full(n, 7, np.uint8)
            else:
                g = (rng.random(n) ** 3 * 255).astype(np.uint8)
            hist = np.bincount(g, minlength=256)
            for q in (2, 5, 95, 98):
                assert onp.percentile_from_hist(hist, q) == pytest.approx(float(np.percentile(g, q)), rel=0, abs=1e-12)
            assert math.isclose(onp.contrast_data({"hist256": hist})["rms_contrast"],
                                round(float(np.std(g.astype(np.float64)) / 255.0), 4), abs_tol=1e-4)


def test_validator_invariants():
    """validation/database_validator.py:282-350,584-607 range invariants."""
    for idx in range(8):
        img = synth_image_bgr(idx, 96, 144)
        m = onp.all_metrics(img)
        assert len(m["histogram"]["histogram_bytes"]) == 1024
        assert 0.0 <= m["histogram"]["mean_luminance"] <= 1.0
        assert 0.0 <= m["histogram"]["exposure_score"] <= 10.0
        if m["monochrome"]["is_monochrome"]:
            assert m["monochrome"]["mean_saturation"] < 0.1


def test_oracle_vs_reference_golden_tight(technical_golden):
    """The reference's analyzer dicts as tests/golden/make_golden.py recorded them, held to the tolerances of a side-by-side
    run with the reference's modules: 1e-5 for the colour and histogram dicts, 1e-9 for the others."""
    rel = {"sharpness": 1e-9, "color": 1e-5, "histogram": 1e-5, "monochrome": 1e-9, "dynamic_range": 1e-9, "noise": 1e-9,
           "contrast": 1e-9}
    for rec in technical_golden["cases"]:
        m = onp.all_metrics(synth_image_bgr(rec["index"], rec["height"], rec["width"]), 0.10)
        for name, r in rel.items():
            _cmp_dict(m[name], rec[name], rel=r)


def test_roi_laplacian_thin_crops_match_cv2():
    """`_get_crop_sharpness` on crops with an extent of one pixel: reflect-101 maps onto the pixel itself."""
    import cv2
    from facet_b200.synth import synth_image_bgr
    from oracle import technical_np as onp
    img = synth_image_bgr(5, 120, 160)
    for box in [(100, 100, 101, 103), (10, 10, 12, 12), (30, 40, 37, 41), (5, 5, 6, 6), (0, 0, 160, 120), (20, 30, 140, 100)]:
        crop = img[box[1]:box[3], box[0]:box[2]]
        want = cv2.Laplacian(cv2.cvtColor(crop, cv2.COLOR_BGR2GRAY), cv2.CV_64F).var()
        n, s1, s2 = onp.roi_laplacian_sums(img, box)
        assert n == crop.shape[0] * crop.shape[1]
        assert abs((s2 / n - (s1 / n) ** 2) - want) <= 1e-9 * max(1.0, want), box
    assert onp.roi_laplacian_sums(img, (50, 50, 50, 90)) == (0, 0, 0)
