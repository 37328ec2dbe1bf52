"""CPU tests: the oracle restatement (oracle/*_oracle.c) against the golden vectors frozen from the
unmodified reference on (a) its own fixtures, (b) synthetic frames.  No GPU, no product code."""
import ast

import numpy as np
import pytest

HARRIS_CASES = ["default", "cpp_default", "sobel_shi_sorted", "harmonic_quartic_top50", "grid100_quadratic",
                "two_scales", "no_gaussian"]


@pytest.mark.parametrize("fixture", ["chairs", "building"])
@pytest.mark.parametrize("case", HARRIS_CASES)
def test_harris_oracle_matches_golden(oracle, golden, fixture, case):
    g = golden("harris_" + fixture)
    kw = ast.literal_eval(str(g[case + "_args"]))
    x, y, s = oracle.harris_detect(g["image"], impl="oracle", **kw)
    assert len(x) == len(g[case + "_x"])
    # bit-exact: same corners, same order, same float strengths
    assert np.array_equal(x, g[case + "_x"]) and np.array_equal(y, g[case + "_y"])
    assert np.array_equal(s, g[case + "_s"])


def test_harris_oracle_response_matches_golden(oracle, golden):
    g = golden("harris_chairs")
    R, _ = oracle.harris_response(g["image"], impl="oracle")
    assert oracle.digest(R) == str(g["R_default_digest"])


def test_harris_window_predicate_equals_scan_on_tie_free_maps(oracle):
    """SURVEY §8a-H6: on tie-free data the order-free window predicate (what the CUDA kernel
    implements) reproduces the reference scan exactly."""
    rng = np.random.default_rng(7)
    for trial in range(30):
        ny, nx = rng.integers(24, 90), rng.integers(24, 90)
        R = rng.standard_normal((ny, nx)).astype(np.float32) * 100
        r = int(rng.integers(1, 7))
        a = oracle.harris_nms(R, 10.0, r)
        b = oracle.harris_nms(R, 10.0, r, window=True)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
        assert b[3].sum() == 0


def test_harris_nms_small_image_returns_nothing(oracle):
    R = np.ones((11, 40), np.float32) * 1000
    assert len(oracle.harris_nms(R, 1.0, 5)[0]) == 0        # ny <= 2r+1  (harris.cpp:151)


@pytest.mark.parametrize("case", ["default", "cpp_default", "fractional_thr"])
def test_canny_oracle_matches_golden(oracle, golden, case):
    g = golden("canny_chairs")
    kw = ast.literal_eval(str(g[case + "_args"]))
    e, nz = oracle.canny(g["image"], impl="oracle", **kw)
    ref = np.unpackbits(g[case + "_edges"])[: e.size].reshape(e.shape).astype(bool)
    assert nz == int(g[case + "_nonzero"])
    assert np.array_equal(e == 255, ref)          # integer edge map: bit-exact
    assert set(np.unique(e)) <= {0, 255}


def test_canny_taps_are_symmetric_and_normalised(oracle):
    c, w = oracle.canny_taps(1920, 2.0)
    assert c[0] == -c[-1] and np.allclose(w, w[::-1], rtol=0, atol=0)
    assert abs(w.sum() - 1) < 1e-15
    assert len(c) == 27                            # |c| <= 13 for s = 2  (exp(-c^2/4) >= 2^-64)


# ------------------------------------------------------------------ against the reference
# The reference's outputs on these inputs are frozen in tests/golden (make_golden_parity.py runs it).

def harris_frame_cases():
    """(key, image, arguments) of the synthetic-frame comparison with the reference."""
    from image_b200 import synth
    for seed, (ny, nx) in enumerate([(120, 200), (97, 131), (256, 64), (70, 70)]):
        img = synth.frame_shapes(100 + seed, ny, nx)
        for j, kw in enumerate([dict(), dict(gaussian=1), dict(gradient=1, measure=2, precision=1), dict(Nscales=2, strategy=1)]):
            yield "harris_frame_%d_%d" % (seed, j), img, dict(threshold=10, **kw)


def harris_tiny_cases():
    rng = np.random.default_rng(3)
    for ny, nx in [(2, 50), (50, 2), (9, 9), (12, 30), (30, 12), (13, 13)]:
        yield "harris_tiny_%dx%d" % (ny, nx), rng.integers(0, 255, (ny, nx)), dict(threshold=0.001)


def canny_frame_cases():
    """(key, image, accGrad); the reference's blurred plane of each image is stored under the key without its suffix."""
    from image_b200 import synth
    for seed, (ny, nx) in enumerate([(108, 192), (75, 101), (64, 64), (9, 7)]):
        img = synth.frame_shapes(200 + seed, ny, nx)
        for acc in (True, False):
            yield "canny_frame_%d_acc%d" % (seed, acc), img, acc


def test_harris_oracle_equals_reference_on_random_frames(oracle, reference_digests):
    for key, img, kw in harris_frame_cases():
        x, y, s = oracle.harris_detect(img, impl="oracle", **kw)
        assert oracle.digests(x=x, y=y, s=s) == reference_digests[key], key


def test_harris_tiny_images_match_reference(oracle, reference_digests):
    for key, img, kw in harris_tiny_cases():
        x, y, s = oracle.harris_detect(img, impl="oracle", **kw)
        assert oracle.digests(x=x, y=y, s=s) == reference_digests[key], key


def test_canny_oracle_equals_reference_shim(oracle, golden, reference_digests):
    """The restatement (direct circular convolution) against the reference's own tools.c driven by
    the DFT shim: blurred planes may differ in float rounding for ~1e-7 of the pixels; edge maps
    must agree (a flip would need a blur flip AND a gradient tie)."""
    blur_ref = golden("canny_blur_reference")
    for key, img, acc in canny_frame_cases():
        eo, no, blur, _ = oracle.canny(img, impl="oracle", accGrad=acc, stages=True)
        flips = int((blur_ref[key.rsplit("_", 1)[0]] != blur).sum())
        assert flips <= max(1, img.size // 100000)
        assert oracle.digests(edges=eo, nonzero=no) == reference_digests[key], key
