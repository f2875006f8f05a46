"""Whole-chain BASELINE configurations on the CPU oracle (no GPU): ``oracle.refapi`` -- the restatement that
travels to the GPU box -- against the committed goldens (``tests/golden/configs.npz``, produced by the reference's
own Python layer, and ``tests/golden/reference_api.npz``) and, when the reference tree is present, against that layer
live, bit for bit."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

from oracle import refapi, refload  # noqa: E402
from pyxfocus_b200 import examples as ex  # noqa: E402
from make_golden_configs import SIZES, stack  # noqa: E402
import make_golden_reference_calls as rc  # noqa: E402
from make_golden_reference_calls import assert_pinned  # noqa: E402

C4_CASES = ((-1, 4.8), (-3, 2.4), (-8, .6), (-1, "uniform"))


@pytest.fixture(scope="module")
def api():
    return ex.make_api(refapi.load(), ex.NumpyXP, "refapi")


@pytest.fixture(scope="module")
def gold(golden):
    return golden("configs")


def same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def test_config2_matches_golden(api, gold):
    ap = ex.ws_aperture(api)
    assert same(np.array(ap), gold["c2_aperture"])
    # SURVEY.md 3.2 probe: aperture radii of the default shell
    assert ap == (220.13737656836065, 221.23348169132342)
    for a in SIZES["c2_arcmin"]:
        r = ex.config2_point(api, SIZES["c2_n"], a / 60. * np.pi / 180., ap)
        tag = "c2_%02d_" % int(a)
        assert same(stack(r["rays"], (1, 2)), gold[tag + "xy"]), tag
        assert same(np.array([r["f"], r["d2"], r["d3"], r["hpd"], r["rms"], r["hpd_scan"], r["rms_scan"]]), gold[tag + "scalars"]), tag


def test_config3_matches_golden(api, gold):
    r = ex.config3(api, SIZES["c3_n"])
    assert same(stack(r["rays"], range(10)), gold["c3_rows"])
    assert same(r["idx"], gold["c3_idx"])
    assert same(np.array([r["hpd"], r["rms"]]), gold["c3_scalars"])
    assert 0 < len(r["idx"]) < SIZES["c3_n"]          # both vignettes bite


@pytest.mark.parametrize("order,wave", C4_CASES)
def test_config4_matches_golden(api, gold, order, wave):
    r = ex.config4(api, SIZES["c4_n"], SIZES["c4_M"], order=order, wave=wave)
    tag = "c4_o%d_%s_" % (-order, "w" if isinstance(wave, str) else "s")
    assert same(stack(r["rays"], range(1, 10)), gold[tag + "rows"])
    assert same(np.array([r["kept"], r["dz"], r["gratings"], r["cx"], r["cy"], r["rmsY"], r["hpdY"]]), gold[tag + "scalars"])
    assert r["gratings"] >= 20                         # the fan really is a long masked loop


def test_config5_matches_golden(api, gold):
    r = ex.config5(api, SIZES["c5_n"], SIZES["c5_shells"], offaxis=1. / 60. * np.pi / 180.)
    assert same(stack(r["rays"], range(1, 10)), gold["c5_rows"])
    assert same(r["weights"], gold["c5_weights"])
    assert same(np.array([r["kept"], r["hpd"], r["rms"], r["cx"], r["cy"], r["area"]]), gold["c5_scalars"])
    assert r["kept"] < SIZES["c5_n"] * SIZES["c5_shells"]


def test_restated_api_equals_the_live_reference_layer(api, golden):
    """Other sizes / seeds than the goldens: every configuration on the restatement against the bits the reference's own
    Python layer gave for the same calls (tests/golden/reference_api.npz); where the reference tree
    is present, that layer live as well."""
    assert_pinned(rc.api_runs(api), golden("reference_api"), what="refapi")
    if refload.available():
        assert_pinned(rc.api_runs(ex.make_api(refload.load(), ex.NumpyXP, "reference")), golden("reference_api"),
                      what="reference")
