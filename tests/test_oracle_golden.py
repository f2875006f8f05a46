"""The oracle restatement (oracle/pyref.py + oracle/chains.py over the C oracle) against
(a) the committed golden vectors, which were produced by the reference's own unmodified
Python layer (tests/golden/make_golden.py), and (b) the bits that layer gave for further calls
(tests/golden/reference_*.npz, tests/golden/make_golden_reference_calls.py), re-checked against
the layer live when its tree is present."""
import os
import sys

import numpy as np
import pytest

from oracle import chains, pyref, refload
from oracle import f2py as of
from util import assert_bit_equal, rows_of

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden_reference_calls as rc  # noqa: E402
from make_golden_reference_calls import assert_pinned  # noqa: E402


def test_golden_wolter1_reproduced_by_restatement(golden):
    g = golden("wolter1")
    np.random.seed(0)
    rays = pyref.subannulus(220., 220.6, 2 * np.pi, 4000, zhat=-1.)
    assert_bit_equal(rays, rows_of(g["rays_in"]), what="subannulus")
    assert np.array_equal(g["u1"], np.random.RandomState(0).rand(8000)[:4000])
    chains.run_steps_cpu(rays, chains.wolter1_steps()[:2])
    assert_bit_equal(rays, rows_of(g["after_primary"]), what="after_primary")
    chains.run_steps_cpu(rays, chains.wolter1_steps()[2:])
    assert_bit_equal(rays, rows_of(g["rays_out"]), what="rays_out")
    w = g["weights"]
    assert pyref.hpd(rays) == g["hpd"] and pyref.rmsCentroid(rays) == g["rms"]
    assert pyref.hpd(rays, weights=w) == g["hpd_w"] and pyref.rmsCentroid(rays, weights=w) == g["rms_w"]
    assert np.array_equal(np.array(pyref.centroid(rays, weights=w)), g["centroid_w"])
    r, cdf = pyref.rhocdf(rays, weights=w)
    assert np.array_equal(r, g["rhocdf_r"]) and np.array_equal(cdf, g["rhocdf_cdf"])


def test_golden_ws_reproduced_by_restatement(golden):
    g = golden("ws_offaxis")
    a0, a1 = chains.ws_aperture()
    assert a0 == g["a0"] and a1 == g["a1"]
    assert a0 == 220.13737656836065 and a1 == 221.23348169132342       # SURVEY.md 3.2 probe
    rays = chains.ws_source(4000, 0)
    assert_bit_equal(rays, rows_of(g["rays_in"]), what="ws rays_in")
    chains.run_steps_cpu(rays, chains.ws_steps(float(g["theta"])))
    assert_bit_equal(rays, rows_of(g["after_secondary"]), what="ws after_secondary")
    assert pyref.analyticImagePlane(rays) == g["dz_analytic"]
    assert pyref.focusI(rays) == g["focus"]
    assert_bit_equal(rays, rows_of(g["rays_out"]), what="ws rays_out")
    assert pyref.hpd(rays) == g["hpd"] and pyref.rmsCentroid(rays) == g["rms"]


def test_golden_vignette_reproduced_by_restatement(golden):
    g = golden("spo_grating")
    assert_bit_equal(pyref.vignette(rows_of(g["after_evan"])), rows_of(g["vignetted_evan"]))
    assert_bit_equal(pyref.vignette(rows_of(g["after_miss"])), rows_of(g["vignetted"]))
    assert_bit_equal(pyref.vignette(rows_of(g["after_miss"]), ind=g["keep"]), rows_of(g["vignetted_mask"]))
    # masked gather/scatter idiom
    rays = rows_of(g["after_grat"])
    pyref.masked(of.transformationsf.radgrat, [rays[1], rays[2], rays[4], rays[5], rays[6]], g["evan"],
                 2.4, 160. / 11832.911, 150)
    assert_bit_equal(rays, rows_of(g["after_evan"]), what="masked radgrat")


def test_restatement_matches_live_reference_python(golden):
    """Every numpy restatement in oracle/pyref.py, and the product's mirrored host helpers, against the bits the
    reference's own functions gave for the same calls (tests/golden/reference_python.npz); where the reference tree is
    present, those functions live as well."""
    gold = golden("reference_python")
    values = rc.python_layer_values(rc.restated_python_layer())
    for f, _ in rc.CONIC_FINITE:
        assert np.all(np.isfinite(values["py.con." + f])), f
    assert_pinned(values, gold, atol=rc.PYTHON_ATOL, what="restatement")
    if refload.available():
        assert_pinned(rc.python_layer_values(rc.reference_python_layer(refload.load())), gold, atol=rc.PYTHON_ATOL,
                      what="reference")


def test_golden_southwell_reproduced_by_the_oracle(golden):
    """tests/golden/southwell.npz was written by the reference's unmodified southwell.py driving the oracle's
    ``reconstruct``; re-running the oracle through this repository's restatement of the same few lines must give
    the same bits (guards the fixture and the f2py-shaped binding)."""
    g = golden("southwell")
    for tag in ("ex", "ir"):
        gx, gy = g[tag + "_gx"].copy(), g[tag + "_gy"].copy()
        ind = np.isnan(gx) | np.isnan(gy)
        gx[ind] = 100.
        gy[ind] = 100.
        phase = np.zeros(gx.shape, order="F")
        phase[ind] = 100.

        def pad(a):
            t = np.zeros((a.shape[0] + 2, a.shape[1] + 2), order="F") + 100.
            t[1:-1, 1:-1] = a
            return t
        P, GX, GY = pad(phase), pad(gx), pad(gy)
        of.reconstruct.reconstruct(GX, GY, 1e-10, 1., P, 10000 if tag == "ex" else 300)
        assert of.reconstruct.reconstruct.sweeps == int(g[tag + "_sweeps"])
        res = P[1:-1, 1:-1]
        res[ind] = np.nan
        assert np.array_equal(-res, g[tag + "_phase"], equal_nan=True)
    for tag in ("even", "odd"):
        xd, yd, bs = g["bin_%s_dims" % tag]
        xa, ya, ph = of.reconstruct.southwellbin(g["bin_x"], g["bin_y"], g["bin_l"], g["bin_m"], bs, int(xd), int(yd))
        assert np.array_equal(xa, g["bin_%s_xang" % tag]) and np.array_equal(ph, g["bin_%s_phase" % tag])


def test_interpolatevec_and_wavefront_restatements_match_the_live_reference(golden):
    """oracle/refapi.py interpolateVec (analyses.py:189-230; both call scipy's griddata) and wavefront (:305-334)
    against the bits the reference's text gave for the same calls (tests/golden/reference_interp.npz), run with the
    two things it lacks as shipped supplied from outside (``make_golden_reference_calls.reference_interp``); where the
    reference tree is present, that text live as well."""
    pytest.importorskip("scipy.interpolate")
    gold = golden("reference_interp")
    values = rc.interp_values(*rc.restated_interp())
    for method in ("linear", "cubic"):
        assert np.isfinite(values["interp.wf.%s.0" % method]).sum() > 50, method
    assert_pinned(values, gold, what="restatement")
    if refload.available():
        assert_pinned(rc.interp_values(*rc.reference_interp(refload.load())), gold, what="reference")
