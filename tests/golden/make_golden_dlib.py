"""Golden vectors for the dlib paths.  Run in the build container (needs /root/reference):

    python tests/golden/make_golden_dlib.py

 * fhog_dlib_face.npz — dlib's OWN regression vectors (dlib/test/fhog.cpp:156-213): the embedded face
   image and the expected 31-channel features for its two cell sizes, decoded by
   oracle/extract_dlib_fhog_golden.cpp (built in place from the reference, ~1 min).
 * fhog_boat.npz / surf_boat.npz — outputs of the unmodified reference (oracle/_ref) on its own
   fixture image.dlib/inst/extdata/cruise_boat.png.
"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402

REF = "/root/reference"
D = REF + "/image.dlib/inst/dlib-19.20"
OUT = os.path.dirname(os.path.abspath(__file__))


def dlib_face_vectors():
    exe, raw = "/tmp/extract_fhog", "/tmp/fhog_dlib_face.bin"
    if not os.path.exists(raw):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-DDLIB_NO_GUI_SUPPORT", "-I" + D, "-I" + D + "/dlib/test",
                               os.path.join(ROOT, "oracle", "extract_dlib_fhog_golden.cpp"), D + "/dlib/test/tester.cpp",
                               D + "/dlib/all/source.cpp", "-o", exe, "-lpthread"])
        subprocess.check_call([exe, raw])
    b = open(raw, "rb").read()
    nr, nc = np.frombuffer(b, np.int32, 2, 0)
    off = 8
    img = np.frombuffer(b, np.uint8, nr * nc * 3, off).reshape(nr, nc, 3); off += nr * nc * 3
    out = {"image": img}
    for k in (1, 2):
        sbin, hr, hc = np.frombuffer(b, np.int32, 3, off); off += 12
        v = np.frombuffer(b, np.float32, hr * hc * 31, off).reshape(hr, hc, 31); off += hr * hc * 31 * 4
        out["cell%d" % k] = np.array(sbin); out["hog%d" % k] = v
    np.savez_compressed(os.path.join(OUT, "fhog_dlib_face.npz"), **out)
    print("dlib face", img.shape, [(int(out["cell%d" % k]), out["hog%d" % k].shape) for k in (1, 2)])


def boat():
    from PIL import Image
    img = np.asarray(Image.open(REF + "/image.dlib/inst/extdata/cruise_boat.png").convert("RGB"))
    f = {"image": img}
    for name, kw in {"default": dict(cell=8, frp=1, fcp=1), "cell4_pad3": dict(cell=4, frp=3, fcp=3)}.items():
        f[name + "_digest"] = np.array(po.digest(po.fhog(img, impl="ref", **kw).astype(np.float32)))   # 0.4 / 1.3 MB as arrays
        f[name + "_args"] = np.array(repr(kw))
    np.savez_compressed(os.path.join(OUT, "fhog_boat.npz"), **f)
    # cell_size == 1 (dlib's separate routine): a 96 x 128 crop keeps the fixture small (31 floats per pixel)
    crop = np.ascontiguousarray(img[100:196, 200:328])
    np.savez_compressed(os.path.join(OUT, "fhog_cell1.npz"), image=crop,
                        fhog=po.fhog(crop, impl="ref", cell=1, frp=1, fcp=1).astype(np.float32))
    s = {"image": img}
    for name, kw in {"default": dict(max_points=1000, thr=30.0), "all": dict(max_points=10000, thr=5.0)}.items():
        r = po.surf(img, impl="ref", **kw)
        for k, v in r.items():
            s[name + "_" + k] = v
        s[name + "_args"] = np.array(repr(kw))
        print("surf", name, len(r["x"]))
    np.savez_compressed(os.path.join(OUT, "surf_boat.npz"), **s)


if __name__ == "__main__":
    po.build(ref=True)
    dlib_face_vectors()
    boat()
