"""Freezes the outputs of the UNMODIFIED reference (oracle/_ref, built in place by oracle/Makefile from the
reference tree) on the synthetic inputs of the parity tests, so that those tests need neither the reference
tree nor oracle/_ref at run time:

    python tests/golden/make_golden_parity.py

 * reference_digests.json   key -> oracle.digests(...) of the reference's outputs on the inputs that the
                            *_cases() generators of the test modules yield (bit-exact comparisons)
 * canny_blur_reference.npz the reference's blurred planes (float32) of the Canny frames: the test counts
                            the pixels where the oracle's blur rounds differently, so it needs the values
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
from oracle import pyoracle as po  # noqa: E402
import test_oracle_contour_lsd as tcl  # noqa: E402
import test_oracle_dlib as tdl  # noqa: E402
import test_oracle_harris_canny as thc  # noqa: E402
import test_rshim_gpu as trs  # noqa: E402


def main():
    po.build(ref=True)
    po._cache.clear()
    for which in ("harris", "canny", "dlib", "otsu", "contour", "lsd"):
        assert po.have_ref(which), "oracle/_ref/libref_%s.so was not built: is the reference tree there?" % which
    d, blur = {}, {}
    for key, img, kw in list(thc.harris_frame_cases()) + list(thc.harris_tiny_cases()):
        x, y, s = po.harris_detect(img, impl="ref", **kw)
        d[key] = po.digests(x=x, y=y, s=s)
    for key, img, acc in thc.canny_frame_cases():
        e, nz = po.canny(img, impl="ref", accGrad=acc)
        d[key] = po.digests(edges=e, nonzero=nz)
        blur[key.rsplit("_", 1)[0]] = po.canny_blur_ref(img, 2.0).astype(np.float32)
    for k, img in enumerate(tcl._frames()):
        g = po.contour_gaussian(img, impl="ref")
        d["contour_frame_%d" % k] = po.digests(gauss=g, **po.contour_edge_points(g, impl="ref"))
        s = po.lsd_sampler(img, impl="ref")
        a, m, lst = po.lsd_ll_angle(s, impl="ref")
        d["lsd_frame_%d" % k] = po.digests(scaled=s, angles=a, modgrad=m, list=lst)
    for key, im, cell, frp, fcp in tdl.fhog_frame_cases():
        d[key] = po.digests(fhog=po.fhog(im, cell, frp, fcp, impl="ref"))
    for key, img, mp, thr in tdl.surf_frame_cases():
        r = po.surf(img, mp, thr, impl="ref")
        d[key] = po.digests(points=len(r["x"]), **r)
    for key, x, ww, hh, thr in tdl.otsu_cases():
        o, t = po.otsu(x, ww, hh, thr, impl="ref")
        d[key] = po.digests(out=o, threshold=t)
    from image_b200 import synth
    seed, Y, X = trs.CONTOUR_SHIM_FRAME
    g = po.contour_gaussian(synth.frame_shapes(seed, Y, X).astype(np.float64), impl="ref")
    d["contour_shim_frame"] = po.digests(**po.contour_edge_points(g, impl="ref"))
    with open(os.path.join(HERE, "reference_digests.json"), "w") as f:
        json.dump(d, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(HERE, "canny_blur_reference.npz"), **blur)
    print("%d digest entries, %d blurred planes" % (len(d), len(blur)))


if __name__ == "__main__":
    main()
