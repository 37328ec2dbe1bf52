"""CPU tests: FHOG / SURF restatements against dlib's own golden vectors and the frozen outputs of the
unmodified reference on its fixture and on synthetic frames."""
import ast

import numpy as np
import pytest


def test_fhog_oracle_reproduces_dlib_regression_vectors(oracle, golden):
    """dlib/test/fhog.cpp:34-81 asserts max|hog - ref| < 1e-6 on these vectors; same bar here."""
    g = golden("fhog_dlib_face")
    for k in (1, 2):
        hog = oracle.fhog(g["image"], int(g["cell%d" % k]), 1, 1)
        ref = g["hog%d" % k]
        assert hog.shape == ref.shape
        assert np.abs(hog - ref).max() < 1e-6


@pytest.mark.parametrize("case", ["default", "cell4_pad3"])
def test_fhog_oracle_matches_reference_on_fixture(oracle, golden, case):
    g = golden("fhog_boat")
    kw = ast.literal_eval(str(g[case + "_args"]))
    hog = oracle.fhog(g["image"], **kw)
    assert oracle.digest(hog.astype(np.float32)) == str(g[case + "_digest"])          # bit-exact (outputs are floats)


@pytest.mark.parametrize("case", ["default", "all"])
def test_surf_oracle_matches_reference_on_fixture(oracle, golden, case):
    g = golden("surf_boat")
    kw = ast.literal_eval(str(g[case + "_args"]))
    r = oracle.surf(g["image"], **kw)
    assert len(r["x"]) == len(g[case + "_x"]) > 50
    for k in ("x", "y", "pyramid_scale", "score", "laplacian", "angle", "surf"):
        assert np.array_equal(r[k], g[case + "_" + k]), k              # bit-exact, including order


def test_integral_image_property(oracle):
    """dlib/test/image.cpp:718-763: box sums from the SAT equal direct sums over random rectangles."""
    import ctypes as C
    rng = np.random.default_rng(2)
    img = rng.integers(0, 255, (37, 53, 3)).astype(np.int32)
    sat = np.zeros((37, 53), np.int32)
    oracle.lib("oracle").orc_surf_sat(img.ctypes.data_as(C.c_void_p), 37, 53, sat.ctypes.data_as(C.c_void_p))
    grey = (img.sum(axis=2) // 3).astype(np.int64)
    assert np.array_equal(sat, grey.cumsum(0).cumsum(1))


# The reference's outputs on the synthetic inputs below are frozen in tests/golden/reference_digests.json
# (make_golden_parity.py runs it).

def fhog_frame_cases():
    """(key, image, cell, frp, fcp)."""
    from image_b200 import synth
    rng = np.random.default_rng(1)
    for rows, cols, cell, frp, fcp in [(100, 131, 8, 1, 1), (97, 203, 4, 1, 1), (120, 160, 8, 2, 5), (75, 90, 5, 1, 1), (23, 300, 8, 1, 1)]:
        for j, im in enumerate((synth.frame_rgb(rows, rows, cols), (synth.frame_rgb(cols, rows, cols) // 16 * 16).astype(np.uint8),
                                rng.integers(0, 255, (rows, cols, 3)).astype(np.uint8))):
            yield "fhog_frame_%dx%d_cell%d_pad%d_%d_%d" % (rows, cols, cell, frp, fcp, j), im, cell, frp, fcp


def surf_frame_cases():
    """(key, image, max_points, threshold)."""
    from image_b200 import synth
    for rows, cols, mp, thr in [(300, 417, 10000, 10.0), (480, 640, 50, 30.0), (540, 960, 10000, 30.0)]:
        yield "surf_frame_%dx%d_%d_%g" % (rows, cols, mp, thr), synth.frame_blobs(rows + cols, rows, cols), mp, thr


def otsu_cases():
    """(key, pixels, width, height, threshold)."""
    rng = np.random.default_rng(5)
    for k in range(12):
        hh, ww = int(rng.integers(1, 60)), int(rng.integers(1, 80))
        x = rng.integers(0, 256, hh * ww).astype(np.float64) if k % 2 else rng.random(hh * ww) * 255.9
        for thr in (0, 33):
            yield "otsu_%d_thr%d" % (k, thr), x, ww, hh, thr


def test_fhog_oracle_equals_reference_incl_colour_ties(oracle, reference_digests):
    for key, im, cell, frp, fcp in fhog_frame_cases():
        assert oracle.digests(fhog=oracle.fhog(im, cell, frp, fcp)) == reference_digests[key], key


def test_surf_oracle_equals_reference(oracle, reference_digests):
    for key, img, mp, thr in surf_frame_cases():
        b = oracle.surf(img, mp, thr)
        assert oracle.digests(points=len(b["x"]), **b) == reference_digests[key], key


def test_fhog_cell_size_1_oracle_matches_reference_fixture(oracle, golden):
    """cell_size == 1 takes dlib's separate routine (fhog.h:495-694); fixture = oracle/_ref output."""
    g = golden("fhog_cell1")
    out = oracle.fhog(g["image"], cell=1)
    assert out.shape == g["fhog"].shape and np.array_equal(out.astype(np.float32), g["fhog"])
    assert int((out != 0).sum()) <= 6 * out.shape[0] * out.shape[1]


def test_otsu_oracle_matches_reference_build_and_fixture(oracle, golden, reference_digests):
    """image.Otsu (8f rank 4): the restatement equals the unmodified source compiled in place on random
    inputs, and the frozen output of that build on the package's own coins.jpeg."""
    g = golden("otsu_coins")
    img = g["image"].astype(np.float64)
    h, w = img.shape
    o, t = oracle.otsu(img.ravel(order="F"), w, h, 0)
    assert t == int(g["threshold"])
    assert np.array_equal(o.reshape(img.shape, order="F") > 0, np.unpackbits(g["mask"])[: img.size].reshape(img.shape).astype(bool))
    for key, x, ww, hh, thr in otsu_cases():
        a, ta = oracle.otsu(x, ww, hh, thr)
        assert oracle.digests(out=a, threshold=ta) == reference_digests[key], key
