"""Drop-in check at the reference's own boundary: the replacement bodies of the four Rcpp exports
(image_b200/rshim/*.cpp) are compiled against an Rcpp-shaped header, linked with libb200feat.so and
called like .Call would; results must equal the oracle's run of the reference glue."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("shim") / "libshim.so")
    rs = os.path.join(ROOT, "image_b200", "rshim")
    srcs = [os.path.join(rs, f) for f in ("rcpp_harris.cpp", "rcpp_canny.cpp", "rcpp_fhog.cpp", "rcpp_surf.cpp", "rcpp_otsu.cpp")]
    objs = []
    for f in ("contour_front.c", "lsd_front.c"):                      # the two plain-C front-end shims
        o = str(tmp_path_factory.mktemp("obj") / (f + ".o"))
        subprocess.check_call(["gcc", "-O1", "-fPIC", "-c", "-I" + os.path.join(ROOT, "include"), os.path.join(rs, f), "-o", o])
        objs.append(o)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "oracle", "stubs"),
                           "-I" + os.path.join(ROOT, "include"), "-I" + rs, os.path.join(ROOT, "tests", "rshim_harness.cpp")] + srcs + objs +
                          ["-L" + os.path.join(ROOT, "image_b200"), "-lb200feat", "-Wl,-rpath," + os.path.join(ROOT, "image_b200"), "-o", out])
    return C.CDLL(out)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_detect_corners_shim(shim, oracle):
    from image_b200 import synth
    img = synth.frame_shapes(21, 180, 250)
    cap = 50000
    x = np.zeros(cap, np.float32); y = np.zeros(cap, np.float32); s = np.zeros(cap, np.float32)
    d = img.astype(np.float64).ravel()
    n = shim.shim_harris(_p(d), 250, 180, C.c_float(60.0), 0, 0, _p(x), _p(y), _p(s), cap)
    ox, oy, os_ = oracle.harris_detect(img, threshold=60.0, gaussian=0, precision=0)
    assert n == len(ox) and np.array_equal(x[:n], ox) and np.array_equal(y[:n], oy)
    assert np.array_equal(s[:n], os_)                 # default path of the shim: the reference's strengths bit for bit


def test_canny_shim(shim, oracle):
    from image_b200 import synth
    img = synth.frame_shapes(22, 120, 200)
    e = np.zeros(120 * 200, np.uint8)
    nz = shim.shim_canny(_p(img.astype(np.int32).ravel()), 200, 120, _p(e))
    oe, onz = oracle.canny(img)
    assert nz == onz and np.array_equal(e.reshape(120, 200), oe)


def test_fhog_shim(shim, oracle):
    from image_b200 import synth
    img = synth.frame_rgb(23, 96, 160)
    nr, nc = C.c_int(0), C.c_int(0)
    a = np.ascontiguousarray(img.astype(np.int32))
    assert shim.shim_fhog(_p(a), 96, 160, None, C.byref(nr), C.byref(nc)) == 0
    out = np.zeros(nr.value * nc.value * 31)
    assert shim.shim_fhog(_p(a), 96, 160, _p(out), C.byref(nr), C.byref(nc)) == 0
    ref = oracle.fhog(img)
    assert np.array_equal(out.reshape(31, nc.value, nr.value).transpose(2, 1, 0), ref)


def test_surf_shim(shim, oracle):
    from image_b200 import synth
    img = synth.frame_blobs(24, 300, 400)
    a = np.ascontiguousarray(img.astype(np.int32))
    cap = 2000
    x = np.zeros(cap); sc = np.zeros(cap); des = np.zeros(cap * 64)
    shim.shim_surf.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_long, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    n = shim.shim_surf(_p(a), 300, 400, 1000, 5.0, cap, _p(x), _p(sc), _p(des))
    ref = oracle.surf(img, 1000, 5.0)
    assert n == len(ref["x"]) and np.array_equal(x[:n], ref["x"]) and np.array_equal(sc[:n], ref["score"])
    if n:
        np.testing.assert_allclose(des[: n * 64].reshape(n, 64), ref["surf"], rtol=1e-4, atol=1e-9)


def test_otsu_shim(shim, oracle):
    from image_b200 import synth
    img = synth.frame_shapes(25, 90, 140).astype(np.float64)
    out = np.zeros(90 * 140, np.float64)
    t = shim.shim_otsu(_p(img.ravel()), 140, 90, 0, _p(out))
    o, ot = oracle.otsu(img.ravel(), 140, 90, 0)
    assert t == ot and np.array_equal(out, o)


CONTOUR_SHIM_FRAME = (24, 150, 230)                                  # (seed, Y, X)


def test_contour_front_shim_feeds_the_reference_chainer(shim, oracle, reference_digests):
    """b2f_contour_front (rshim/contour_front.c) rebuilds the planes the reference's sequential chainer reads: Ex / Ey equal
    the reference's planes everywhere, Gx / Gy at every edge point (the only pixels where its chain() reads them), so the
    reference's own chain_edge_points -> simplify_chains -> list_chained_edge_points gives the same curves on them as on
    the reference's planes; where the reference is built, that is checked by running it."""
    from image_b200 import synth
    seed, Y, X = CONTOUR_SHIM_FRAME
    img = synth.frame_shapes(seed, Y, X).astype(np.float64)
    gauss = np.zeros((Y, X)); Gx = np.zeros((Y, X)); Gy = np.zeros((Y, X)); Ex = np.zeros((Y, X)); Ey = np.zeros((Y, X))
    shim.b2f_contour_front.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double] + [C.c_void_p] * 5
    assert shim.b2f_contour_front(_p(img), X, Y, 0.0, _p(gauss), _p(Gx), _p(Gy), _p(Ex), _p(Ey)) == 0
    g = oracle.contour_gaussian(img)
    assert np.array_equal(gauss, g)
    r = oracle.contour_edge_points(g)
    assert oracle.digests(**r) == reference_digests["contour_shim_frame"]    # the reference's edge points and gradients
    ex = np.full(X * Y, -1.0); ey = np.full(X * Y, -1.0)
    ex[r["idx"]] = r["Ex"]; ey[r["idx"]] = r["Ey"]
    assert np.array_equal(Ex.ravel(), ex) and np.array_equal(Ey.ravel(), ey)
    assert np.array_equal(Gx.ravel()[r["idx"]], r["Gx"]) and np.array_equal(Gy.ravel()[r["idx"]], r["Gy"])
    if oracle.have_ref("contour"):
        rEx, rEy, rGx, rGy = oracle.contour_planes_ref(g)
        a = oracle.contour_chain_ref(Ex, Ey, Gx, Gy)
        b = oracle.contour_chain_ref(rEx, rEy, rGx, rGy)
        assert len(b[0]) > 100
        for u, v in zip(a, b):
            assert np.array_equal(u, v)


def test_lsd_front_shim_builds_the_ordered_chain(shim, oracle):
    from image_b200 import synth

    class Cell(C.Structure):
        pass
    Cell._fields_ = [("x", C.c_int), ("y", C.c_int), ("next", C.POINTER(Cell))]
    Y, X = 120, 170
    img = synth.frame_shapes(25, Y, X).astype(np.float64)
    N, M = int(np.ceil(X * 0.8)), int(np.ceil(Y * 0.8))
    ang = np.zeros((M, N)); mod = np.zeros((M, N))
    head = C.POINTER(Cell)(); mem = C.c_void_p()
    shim.b2f_lsd_front.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_void_p,
                                   C.POINTER(C.POINTER(Cell)), C.POINTER(C.c_void_p)]
    assert shim.b2f_lsd_front(_p(img), X, Y, 0.8, 0.6, 2.0, 22.5, 1024, _p(ang), _p(mod), C.byref(head), C.byref(mem)) == 0
    a, m, lst = oracle.lsd_ll_angle(oracle.lsd_sampler(img))
    assert np.array_equal(mod, m) and np.array_equal(ang == -1024.0, a == -1024.0)
    got, p = [], head
    while p:
        got.append(p.contents.x + p.contents.y * N)
        p = p.contents.next
    assert np.array_equal(np.array(got, np.int32), lst)
    C.CDLL(None).free(mem)
