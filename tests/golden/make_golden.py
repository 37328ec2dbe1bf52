"""Generates tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref, built in place from
/root/reference by oracle/Makefile) on the reference's own fixtures.  Run in the build container:

    python tests/golden/make_golden.py

Each file holds the input pixels and the reference outputs, so the tests need neither
/root/reference nor oracle/_ref at run time.
"""
import lzma
import os
import struct
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))


def read_building_rds():
    """image.CornerDetectionHarris/inst/extdata/building.rds: xz-compressed R serialization (v2) of an
    integer matrix; returned as R sees it: array [nrow, ncol] (column-major data)."""
    raw = lzma.decompress(open(REF + "/image.CornerDetectionHarris/inst/extdata/building.rds", "rb").read())
    assert raw[:2] == b"X\n"
    off = 2 + 12                      # version, writer version, min reader version
    flags, = struct.unpack(">i", raw[off:off + 4]); off += 4
    assert flags & 0xFF == 13         # INTSXP
    n, = struct.unpack(">i", raw[off:off + 4]); off += 4
    data = np.frombuffer(raw[off:off + 4 * n], dtype=">i4").astype(np.int32); off += 4 * n
    # attribute pairlist: dim
    tail = raw[off:]
    i = tail.find(b"dim")
    j = i + 3
    f2, ln = struct.unpack(">ii", tail[j:j + 8])
    assert f2 & 0xFF == 13 and ln == 2
    d = struct.unpack(">ii", tail[j + 8:j + 16])
    return data.reshape(d[1], d[0]).T          # [nrow, ncol]


def harris_cases(img_yx, tag):
    """img_yx: [ny, nx] grey image.  Stores reference corner lists for several argument sets."""
    out = {"image": img_yx.astype(np.uint8)}
    cases = {
        "default": dict(gaussian=0, gradient=0, measure=0, strategy=0, precision=0),          # R defaults as seen by C++
        "cpp_default": dict(gaussian=1, precision=1),                                            # Rcpp-level defaults
        "sobel_shi_sorted": dict(gaussian=0, gradient=1, measure=1, strategy=1, precision=0),
        "harmonic_quartic_top50": dict(gaussian=0, measure=2, strategy=2, Nselect=50, precision=2),
        "grid100_quadratic": dict(gaussian=0, strategy=3, Nselect=100, cells=5, precision=1),
        "two_scales": dict(gaussian=0, Nscales=2, precision=0),
        "no_gaussian": dict(gaussian=2, precision=0),
    }
    for name, kw in cases.items():
        x, y, s = po.harris_detect(img_yx, impl="ref", **kw)
        out[name + "_x"], out[name + "_y"], out[name + "_s"] = x, y, s
        out[name + "_args"] = np.array(repr(kw))
    R, _ = po.harris_response(img_yx, impl="ref")
    out["R_default_digest"] = np.array(po.digest(R))      # the float32 plane itself does not compress (1 MB)
    np.savez_compressed(os.path.join(OUT, "harris_%s.npz" % tag), **out)
    print("harris", tag, {k: len(out[k + "_x"]) for k in cases})


def canny_cases(img_yx, tag):
    out = {"image": img_yx.astype(np.uint8)}
    cases = {
        "default": dict(s=2.0, low_thr=3.0, high_thr=10.0, accGrad=True),        # R wrapper defaults (accGrad=TRUE)
        "cpp_default": dict(s=2.0, low_thr=3.0, high_thr=10.0, accGrad=False),   # Rcpp-level default
        "fractional_thr": dict(s=1.3, low_thr=2.7, high_thr=7.9, accGrad=True),
    }
    for name, kw in cases.items():
        e, nz = po.canny(img_yx, impl="ref", **kw)
        out[name + "_edges"] = np.packbits(e == 255)
        out[name + "_nonzero"] = np.array(nz)
        out[name + "_args"] = np.array(repr(kw))
    np.savez_compressed(os.path.join(OUT, "canny_%s.npz" % tag), **out)
    print("canny", tag, {k: int(out[k + "_nonzero"]) for k in cases})


if __name__ == "__main__":
    po.build(ref=True)
    chairs = po.read_pgm_ascii(REF + "/image.CannyEdges/inst/extdata/chairs.pgm")     # [512, 512], BASELINE config 1
    harris_cases(chairs, "chairs")
    canny_cases(chairs, "chairs")
    b = read_building_rds()                                                            # R matrix [600, 400] = [w, h]
    harris_cases(np.ascontiguousarray(b.T), "building")                                # as image [ny=400, nx=600]
    if len(sys.argv) > 1 and sys.argv[1] == "all":
        import make_golden_dlib  # noqa: F401
