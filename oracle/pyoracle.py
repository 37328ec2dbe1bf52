"""TEST INFRASTRUCTURE — ctypes front-end to the CPU checkers.

`orc`  : oracle/liboracle.so      the C restatement in oracle/*_oracle.c (always buildable)
`ref`  : oracle/_ref/libref_*.so  the UNMODIFIED reference compiled in place from /root/reference
                                   (present where it was built; travels to the GPU box as a .so)
Tests compare with the reference through outputs frozen under tests/golden/ (whole arrays or their
`digest`s), so they need no `ref` library at run time; the tests/golden/make_golden*.py scripts use it.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product package image_b200 never does.
"""
import ctypes as C
import hashlib
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def digest(a):
    """'<dtype>[shape]:sha256' of an array's values.  Two arrays of one dtype have equal digests exactly when
    np.array_equal holds (-0.0 and +0.0 hash alike; a NaN fails, as it fails array_equal), so a stored digest
    of a reference output keeps a bit-exact comparison without storing the output."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        assert not np.isnan(a).any(), "NaN in an array to be compared"
        a = a + a.dtype.type(0)                       # -0.0 -> +0.0
    return "%s%s:%s" % (a.dtype.str, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest())


def digests(**values):
    """{name: digest(array) or int(scalar)}: one entry of tests/golden/reference_digests.json."""
    return {k: digest(v) if isinstance(v, np.ndarray) else int(v) for k, v in values.items()}


def build(ref=True):
    """(Re)build liboracle.so and, when /root/reference exists, oracle/_ref/*.so."""
    subprocess.check_call(["make", "-s", "-C", HERE, "oracle"] + (["ref"] if ref else []))


def _load(path):
    if not os.path.exists(path):
        return None
    return C.CDLL(path)


_cache = {}


def lib(name):
    """name in {'oracle','ref_harris','ref_canny','ref_dlib','ref_otsu','ref_contour','ref_lsd'}; None if that .so is absent."""
    if name not in _cache:
        p = os.path.join(HERE, "liboracle.so") if name == "oracle" else os.path.join(HERE, "_ref", "lib%s.so" % name)
        _cache[name] = _load(p)
    return _cache[name]


def have_ref(which):
    return lib("ref_" + which) is not None


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


f32 = C.c_float
f64 = C.c_double

# ------------------------------------------------------------------------------------------ Harris


def harris_detect(img, k=0.06, sigma_d=1.0, sigma_i=2.5, threshold=130.0, gaussian=0, gradient=0,
                  strategy=0, Nselect=1, measure=0, Nscales=1, precision=0, cells=10, impl="oracle"):
    """img: 2-D array [ny, nx] (any numeric dtype; passed as doubles like R does).
    Returns (x, y, strength) float32 arrays.  impl: 'oracle' | 'ref'."""
    img = np.ascontiguousarray(img, dtype=np.float64)
    ny, nx = img.shape
    cap = nx * ny // 2 + 16
    x = np.zeros(cap, np.float32); y = np.zeros(cap, np.float32); s = np.zeros(cap, np.float32)
    if impl == "ref":
        fn = lib("ref_harris").ref_harris_detect
    else:
        fn = lib("oracle").orc_harris_detect
    fn.restype = C.c_int
    n = fn(_p(img), nx, ny, f32(k), f32(sigma_d), f32(sigma_i), f32(threshold), int(gaussian), int(gradient),
           int(strategy), int(Nselect), int(measure), int(Nscales), int(precision), int(cells),
           _p(x), _p(y), _p(s), cap)
    return x[:n].copy(), y[:n].copy(), s[:n].copy()


def harris_response(img, gauss=0, grad=0, measure=0, k=0.06, sigma_d=1.0, sigma_i=2.5, impl="oracle"):
    """Returns (R, blurred_I) float32 [ny,nx]."""
    I = np.ascontiguousarray(img, dtype=np.float32).copy()
    ny, nx = I.shape
    R = np.zeros((ny, nx), np.float32)
    if impl == "ref":
        lib("ref_harris").ref_harris_response(_p(I), _p(R), nx, ny, int(gauss), int(grad), int(measure), f32(k), f32(sigma_d), f32(sigma_i))
    else:
        lib("oracle").orc_harris_response(_p(I), _p(R), nx, ny, int(gauss), int(grad), int(measure), f32(k), f32(sigma_d), f32(sigma_i))
    return R, I


def harris_nms(R, Th, radius, impl="oracle", window=False):
    """impl 'ref' = reference scan; 'oracle' + window=False = restated scan; window=True = window
    predicate (returns an extra `ambiguous` uint8 array)."""
    R = np.ascontiguousarray(R, dtype=np.float32)
    ny, nx = R.shape
    cap = nx * ny // 2 + 16
    x = np.zeros(cap, np.float32); y = np.zeros(cap, np.float32); s = np.zeros(cap, np.float32)
    if impl == "ref":
        fn = lib("ref_harris").ref_harris_nms; fn.restype = C.c_int
        Rc = R.copy()
        n = fn(_p(Rc), f32(Th), int(radius), nx, ny, _p(x), _p(y), _p(s), cap)
        return x[:n].copy(), y[:n].copy(), s[:n].copy()
    if window:
        amb = np.zeros(cap, np.uint8)
        fn = lib("oracle").orc_harris_nms_window; fn.restype = C.c_int
        n = fn(_p(R), f32(Th), int(radius), nx, ny, _p(x), _p(y), _p(s), _p(amb), cap)
        return x[:n].copy(), y[:n].copy(), s[:n].copy(), amb[:n].copy()
    fn = lib("oracle").orc_harris_nms_scan; fn.restype = C.c_int
    n = fn(_p(R), f32(Th), int(radius), nx, ny, _p(x), _p(y), _p(s), cap)
    return x[:n].copy(), y[:n].copy(), s[:n].copy()


def harris_gaussian(I, sigma, type=0, impl="oracle"):
    I = np.ascontiguousarray(I, dtype=np.float32)
    ny, nx = I.shape
    out = I.copy()
    src = I.copy()
    if impl == "ref":
        lib("ref_harris").ref_harris_gaussian(_p(src), _p(out), nx, ny, f32(sigma), int(type))
    else:
        lib("oracle").orc_gaussian(_p(src), _p(out), nx, ny, f32(sigma), int(type))
    return out

# ------------------------------------------------------------------------------------------ Canny


def canny(img, s=2.0, low_thr=3.0, high_thr=10.0, accGrad=True, impl="oracle", stages=False):
    """img: [ny,nx] integer array.  Returns (edges uint8 [ny,nx], pixels_nonzero)
    (+ blurred float32 plane and class map when stages=True, oracle only)."""
    a = np.ascontiguousarray(img, dtype=np.int32)
    ny, nx = a.shape
    e = np.zeros((ny, nx), np.uint8)
    if impl == "ref":
        fn = lib("ref_canny").ref_canny; fn.restype = C.c_int
        nz = fn(_p(a), nx, ny, f64(s), f64(low_thr), f64(high_thr), int(bool(accGrad)), _p(e))
        return e, nz
    fn = lib("oracle").orc_canny; fn.restype = C.c_int
    if stages:
        b = np.zeros((ny, nx), np.float32); c = np.zeros((ny, nx), np.uint8)
        nz = fn(_p(a), nx, ny, f64(s), f64(low_thr), f64(high_thr), int(bool(accGrad)), _p(e), _p(b), _p(c))
        return e, nz, b, c
    nz = fn(_p(a), nx, ny, f64(s), f64(low_thr), f64(high_thr), int(bool(accGrad)), _p(e), None, None)
    return e, nz


def canny_blur_ref(img, s):
    """The reference's own gblur (tools.c) through the DFT shim: float-rounded doubles."""
    a = np.ascontiguousarray(img, dtype=np.float64)
    ny, nx = a.shape
    out = np.zeros((ny, nx), np.float64)
    lib("ref_canny").ref_canny_gblur(_p(a), _p(out), nx, ny, f64(s))
    return out


def canny_taps(w, s):
    cap = w
    c = np.zeros(cap, np.int32); wt = np.zeros(cap, np.float64)
    fn = lib("oracle").orc_canny_taps; fn.restype = C.c_int
    n = fn(int(w), f64(s), _p(c), _p(wt), cap)
    return c[:n].copy(), wt[:n].copy()

# ------------------------------------------------------------------------------------------ FHOG


def fhog(rgb, cell=8, frp=1, fcp=1, impl="oracle"):
    """rgb: [rows, cols, 3] integer array.  Returns float64 array [hog_nr, hog_nc, 31]
    (the R wrapper's `array(out$fhog, dim=c(hog_height, hog_width, 31))`, image_fhog.R:47)."""
    a = np.ascontiguousarray(rgb, dtype=np.int32)
    rows, cols = a.shape[:2]
    hnr = C.c_int(); hnc = C.c_int()
    fn = lib("ref_dlib").ref_fhog if impl == "ref" else lib("oracle").orc_fhog
    fn(_p(a), rows, cols, int(cell), int(frp), int(fcp), None, C.byref(hnr), C.byref(hnc))
    out = np.zeros(max(hnr.value * hnc.value * 31, 1), np.float64)
    fn(_p(a), rows, cols, int(cell), int(frp), int(fcp), _p(out), C.byref(hnr), C.byref(hnc))
    n = hnr.value * hnc.value * 31
    # glue order: y + nr*(x + nc*feat)  -> numpy [feat, x, y] -> [y, x, feat]
    return out[:n].reshape(31, hnc.value, hnr.value).transpose(2, 1, 0).copy()

# ------------------------------------------------------------------------------------------ Otsu


def otsu(x, width, height, threshold=0, impl="oracle"):
    """otsu(x, width, height, threshold) of image.Otsu: x = width*height doubles.  Returns (out doubles, threshold)."""
    v = np.ascontiguousarray(np.asarray(x, dtype=np.float64).ravel())
    out = np.zeros_like(v)
    t = C.c_int(0)
    fn = lib("ref_otsu").ref_otsu if impl == "ref" else lib("oracle").orc_otsu
    fn.restype = C.c_int
    rc = fn(_p(v), int(width), int(height), int(threshold), _p(out), C.byref(t))
    if rc != 0:
        raise ValueError("pixel values outside 0..255")
    return out, int(t.value)

# ------------------------------------------------------------------------------------------ SURF


def surf(rgb, max_points=1000, thr=30.0, impl="oracle"):
    """Returns dict(x,y,angle,pyramid_scale,score,laplacian: float64[n]; surf: float64[n,64])."""
    a = np.ascontiguousarray(rgb, dtype=np.int32)
    rows, cols = a.shape[:2]
    cap = int(max_points) + 1
    arrs = [np.zeros(cap, np.float64) for _ in range(6)]
    des = np.zeros(cap * 64, np.float64)
    fn = lib("ref_dlib").ref_surf if impl == "ref" else lib("oracle").orc_surf
    fn.restype = C.c_int
    n = fn(_p(a), rows, cols, C.c_long(int(max_points)), f64(thr), cap, *[_p(v) for v in arrs], _p(des))
    names = ["x", "y", "angle", "pyramid_scale", "score", "laplacian"]
    out = {k: v[:n].copy() for k, v in zip(names, arrs)}
    out["surf"] = des[: n * 64].reshape(n, 64).copy()
    return out

# ------------------------------------------------------------------------------------------ fixtures


# ------------------------------------------------------------------------------------------ ContourDetector front end
def contour_sigma():
    """smooth_contours.c:1466-1479: sigma_step * sqrt(dog_rate^2 - 1)."""
    return float(0.8 * np.sqrt(np.float64(1.6) * np.float64(1.6) - 1.0))


def contour_gaussian(img, sigma=None, impl="oracle"):
    """gaussian_filter (smooth_contours.c:184-262) of a [Y, X] image -> float64 [Y, X]."""
    I = np.ascontiguousarray(img, dtype=np.float64)
    Y, X = I.shape
    out = np.zeros((Y, X), np.float64)
    s = contour_sigma() if sigma is None else float(sigma)
    if impl == "ref":
        lib("ref_contour").ref_contour_gaussian(_p(I), X, Y, f64(s), _p(out))
    else:
        lib("oracle").orc_contour_gaussian(_p(I), X, Y, f64(s), _p(out))
    return out


def contour_edge_points(gauss, impl="oracle"):
    """compute_gradient + compute_edge_points on the blurred image -> dict(idx, Ex, Ey, Gx, Gy) in raster order."""
    g = np.ascontiguousarray(gauss, dtype=np.float64)
    Y, X = g.shape
    if impl == "ref":
        planes = [np.zeros((Y, X), np.float64) for _ in range(5)]
        Gx, Gy, modG, Ex, Ey = planes
        lib("ref_contour").ref_contour_edge_points(_p(g), X, Y, _p(Gx), _p(Gy), _p(modG), _p(Ex), _p(Ey))
        idx = np.flatnonzero((Ex.ravel() >= 0) & (Ey.ravel() >= 0)).astype(np.int32)
        return dict(idx=idx, Ex=Ex.ravel()[idx], Ey=Ey.ravel()[idx], Gx=Gx.ravel()[idx], Gy=Gy.ravel()[idx])
    cap = X * Y
    idx = np.zeros(cap, np.int32)
    Ex = np.zeros(cap); Ey = np.zeros(cap); Gx = np.zeros(cap); Gy = np.zeros(cap)
    fn = lib("oracle").orc_contour_edge_points
    fn.restype = C.c_int
    n = fn(_p(g), X, Y, _p(idx), _p(Ex), _p(Ey), _p(Gx), _p(Gy), cap)
    return dict(idx=idx[:n].copy(), Ex=Ex[:n].copy(), Ey=Ey[:n].copy(), Gx=Gx[:n].copy(), Gy=Gy[:n].copy())


def contour_chain_ref(Ex, Ey, Gx, Gy):
    """The reference's sequential chainer on given [Y, X] planes -> (x, y, curve_limits)."""
    planes = [np.ascontiguousarray(p, dtype=np.float64).copy() for p in (Ex, Ey, Gx, Gy)]
    Y, X = planes[0].shape
    cap = X * Y
    x = np.zeros(cap); y = np.zeros(cap)
    lim = np.zeros(cap + 1, np.int32)
    M = C.c_int(0)
    fn = lib("ref_contour").ref_contour_chain_from_planes
    fn.restype = C.c_int
    n = fn(_p(planes[0]), _p(planes[1]), _p(planes[2]), _p(planes[3]), X, Y, _p(x), _p(y), cap, _p(lim), cap, C.byref(M))
    return x[:n].copy(), y[:n].copy(), lim[:M.value + 1].copy()


def contour_planes_ref(gauss):
    """compute_gradient + compute_edge_points of the reference -> full planes (Ex, Ey, Gx, Gy)."""
    g = np.ascontiguousarray(gauss, dtype=np.float64)
    Y, X = g.shape
    Gx, Gy, modG, Ex, Ey = [np.zeros((Y, X), np.float64) for _ in range(5)]
    lib("ref_contour").ref_contour_edge_points(_p(g), X, Y, _p(Gx), _p(Gy), _p(modG), _p(Ex), _p(Ey))
    return Ex, Ey, Gx, Gy


def contour_detect_ref(img, Q=2.0):
    """The whole reference detector (smooth_contours) -> (x, y, curve_limits)."""
    I = np.ascontiguousarray(img, dtype=np.float64)
    Y, X = I.shape
    cap = X * Y
    x = np.zeros(cap); y = np.zeros(cap)
    lim = np.zeros(cap + 1, np.int32)
    M = C.c_int(0)
    fn = lib("ref_contour").ref_contour_detect
    fn.restype = C.c_int
    n = fn(_p(I), X, Y, f64(Q), _p(x), _p(y), cap, _p(lim), cap, C.byref(M))
    return x[:n].copy(), y[:n].copy(), lim[:M.value + 1].copy()


# ------------------------------------------------------------------------------------------ LSD front end
def lsd_rho(quant=2.0, ang_th=22.5):
    """lsd.c:2449-2451: gradient magnitude threshold quant / sin(pi ang_th / 180)."""
    return float(quant / np.sin(np.pi * ang_th / 180.0))


def lsd_sampler(img, scale=0.8, sigma_scale=0.6, impl="oracle"):
    """gaussian_sampler (lsd.c:603-720): [Y, X] -> float64 [ceil(Y*scale), ceil(X*scale)]."""
    I = np.ascontiguousarray(img, dtype=np.float64)
    Y, X = I.shape
    N, M = int(np.ceil(X * scale)), int(np.ceil(Y * scale))
    out = np.zeros((M, N), np.float64)
    if impl == "ref":
        n, m = C.c_int(0), C.c_int(0)
        lib("ref_lsd").ref_lsd_sampler(_p(I), X, Y, f64(scale), f64(sigma_scale), _p(out), C.byref(n), C.byref(m))
        assert (n.value, m.value) == (N, M)
    else:
        lib("oracle").orc_lsd_sampler(_p(I), X, Y, f64(scale), f64(sigma_scale), _p(out))
    return out


def lsd_ll_angle(img, threshold=None, n_bins=1024, impl="oracle"):
    """ll_angle (lsd.c:744-880) -> (angles [Y,X], modgrad [Y,X], list of linear indices x + y*X in list order)."""
    I = np.ascontiguousarray(img, dtype=np.float64)
    Y, X = I.shape
    th = lsd_rho() if threshold is None else float(threshold)
    ang = np.zeros((Y, X)); mod = np.zeros((Y, X))
    if impl == "ref":
        lx = np.zeros(X * Y, np.int32); ly = np.zeros(X * Y, np.int32)
        fn = lib("ref_lsd").ref_lsd_ll_angle
        fn.restype = C.c_int
        n = fn(_p(I), X, Y, f64(th), int(n_bins), _p(ang), _p(mod), _p(lx), _p(ly))
        return ang, mod, (lx[:n] + ly[:n] * X).astype(np.int32)
    lst = np.zeros(X * Y, np.int32)
    fn = lib("oracle").orc_lsd_ll_angle
    fn.restype = C.c_int
    n = fn(_p(I), X, Y, f64(th), int(n_bins), _p(ang), _p(mod), _p(lst))
    return ang, mod, lst[:n].copy()


def lsd_detect_ref(img):
    """The whole reference detector with the Rcpp defaults -> [n, 7] float64."""
    I = np.ascontiguousarray(img, dtype=np.float64)
    Y, X = I.shape
    cap = 200000
    out = np.zeros((cap, 7))
    fn = lib("ref_lsd").ref_lsd_detect
    fn.restype = C.c_int
    n = fn(_p(I), X, Y, _p(out), cap)
    return out[:n].copy()


def read_pgm_ascii(path):
    t = open(path).read().split()
    assert t[0] == "P2"
    w, h = int(t[1]), int(t[2])
    return np.array(t[4:4 + w * h], dtype=np.int32).reshape(h, w)
