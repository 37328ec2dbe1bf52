"""The C restatements of the ContourDetector and LSD front ends (oracle/contour_oracle.c, oracle/lsd_oracle.c) against
the UNMODIFIED reference sources compiled in place (oracle/_ref/libref_contour.so, libref_lsd.so): bit for bit, on
synthetic frames, through the reference's outputs frozen in tests/golden/reference_digests.json.  Neither package ships
tests or golden vectors, so `_ref` is the authority ("parity unpinned" beyond it)."""
import numpy as np
import pytest

from image_b200 import synth


def _frames():
    rng = np.random.default_rng(11)
    out = [synth.frame_shapes(5, 97, 131).astype(np.float64), rng.integers(0, 256, (40, 53)).astype(np.float64),
           synth.frame_shapes(6, 120, 160).astype(np.float64) + rng.random((120, 160))]
    return out


@pytest.mark.parametrize("k", range(3))
def test_contour_front_end_restatement_is_bit_identical_to_the_reference(oracle, reference_digests, k):
    img = _frames()[k]
    g_o = oracle.contour_gaussian(img)
    e_o = oracle.contour_edge_points(g_o)
    assert len(e_o["idx"]) > 50
    assert oracle.digests(gauss=g_o, **e_o) == reference_digests["contour_frame_%d" % k]


@pytest.mark.parametrize("k", range(3))
def test_lsd_front_end_restatement_is_bit_identical_to_the_reference(oracle, reference_digests, k):
    img = _frames()[k]
    s_o = oracle.lsd_sampler(img)
    assert s_o.shape == (int(np.ceil(img.shape[0] * 0.8)), int(np.ceil(img.shape[1] * 0.8)))
    a_o, m_o, l_o = oracle.lsd_ll_angle(s_o)
    assert len(l_o) == (s_o.shape[0] - 1) * (s_o.shape[1] - 1)
    assert oracle.digests(scaled=s_o, angles=a_o, modgrad=m_o, list=l_o) == reference_digests["lsd_frame_%d" % k]
