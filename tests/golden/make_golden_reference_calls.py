"""Golden fixtures for the calls the cross-checks against the reference's own code make (tests/test_examples.py,
tests/test_oracle_golden.py, tests/test_f95_source.py), so that those checks run without the reference tree:

    reference_api.npz      every BASELINE configuration at sizes / seeds other than configs.npz
    reference_python.npz   sources, vignette, analyses, conicsolve and transformations helpers of the Python layer
    reference_interp.npz   interpolateVec and wavefront
    reference_f95.npz      the small configurations the reference ran over its own Fortran text

    python tests/golden/make_golden_reference_calls.py                 # the reference's code (needs its tree)
    python tests/golden/make_golden_reference_calls.py --restatement   # the restatement in its place

The committed fixtures were written with ``--restatement``: oracle/ and the Python helpers of pyxfocus_b200 were
then unchanged since the commit at which the same calls, run on the reference's own Python layer and Fortran text,
gave the same bits.  Where the reference tree is present the tests still run the reference and compare it with the
fixtures as well.

Arrays of more than SAMPLE entries are stored as the SHA-256 of their float64 bytes plus a fixed sample of entries
(``pinned``), which keeps every file small while the comparison stays bit for bit over every entry.
"""
import hashlib
import os
import sys
from types import SimpleNamespace

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import chains, pyref, refapi, refload  # noqa: E402

SAMPLE = 64


# ------------------------------------------------------------------------------------------------ storage
def _canonical(a):
    """float64 copy in which every NaN is the same NaN and -0 is +0: what ``==`` / ``equal_nan`` cannot tell apart
    must hash the same."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    return np.where(np.isnan(a), np.nan, a + 0.)


def _digest(a):
    return np.frombuffer(hashlib.sha256(_canonical(a).tobytes()).digest(), dtype=np.uint8)


def _sample_index(size):
    return np.sort(np.random.default_rng(0).choice(size, SAMPLE, replace=False))


def flatten(prefix, v, out):
    """Nested dicts / lists / tuples of arrays and scalars -> {dotted key: array}."""
    if isinstance(v, dict):
        for k in v:
            flatten("%s.%s" % (prefix, k), v[k], out)
    elif isinstance(v, (list, tuple)):
        for j, x in enumerate(v):
            flatten("%s.%d" % (prefix, j), x, out)
    else:
        out[prefix] = np.asarray(v)
    return out


def pinned(values):
    """Golden form of {key: array}: small arrays whole, larger ones as shape + digest + sample."""
    out = {}
    for k, v in values.items():
        a = np.asarray(v)
        if a.size <= SAMPLE:
            out[k] = a
        else:
            out[k + "__shape"] = np.array(a.shape)
            out[k + "__sha256"] = _digest(a)
            out[k + "__sample"] = _canonical(a).ravel()[_sample_index(a.size)]
    return out


def assert_pinned(values, gold, atol=None, what=""):
    """``values`` equal the fixture entry for entry (NaNs equal to NaNs); keys in ``atol`` within that absolute
    tolerance instead (they must be stored whole)."""
    atol = atol or {}
    keys = sorted({k.split("__")[0] for k in gold.files})
    assert sorted(values) == keys, "%s: keys differ: %s" % (what, sorted(set(values) ^ set(keys)))
    for k in keys:
        a = np.asarray(values[k])
        if k in gold.files:
            b = gold[k]
            assert a.shape == b.shape, "%s %s: shape %s vs %s" % (what, k, a.shape, b.shape)
            if k in atol:
                assert np.allclose(a, b, rtol=0, atol=atol[k]), (what, k)
            else:
                assert np.array_equal(a, b, equal_nan=True), "%s %s: %r vs %r" % (what, k, a, b)
            continue
        assert a.shape == tuple(gold[k + "__shape"]), "%s %s: shape %s vs %s" % (what, k, a.shape, tuple(gold[k + "__shape"]))
        got = _canonical(a).ravel()[_sample_index(a.size)]
        want = gold[k + "__sample"]
        same = (got == want) | (np.isnan(got) & np.isnan(want))
        assert same.all(), "%s %s: %d of %d sampled entries differ, first %r vs %r" % (
            what, k, (~same).sum(), SAMPLE, got[~same][0], want[~same][0])
        assert np.array_equal(_digest(a), gold[k + "__sha256"]), "%s %s: entries outside the stored sample differ" % (what, k)


# ------------------------------------------------------------------------------------------------ the calls
def api_runs(api):
    """Every configuration on an ``examples.make_api`` API, at sizes / seeds other than configs.npz."""
    from pyxfocus_b200 import examples as ex
    ap = ex.ws_aperture(api)
    return flatten("api", dict(
        aperture=ap,
        c1=ex.config1(api, 5000, 3),
        c2=ex.config2_point(api, 2000, 24. / 60. * np.pi / 180., ap, 5),
        c3=ex.config3(api, 3000, 2),
        c4=ex.config4(api, 15, 30, order=-2, wave=2.4, rng_seed=4, offX=1e-4, offY=-2e-4),
        c5=ex.config5(api, 60, 25, offaxis=2e-4, rng_seed=7)), {})


def f95_runs(api):
    """The small configurations the reference ran over its own Fortran text."""
    from pyxfocus_b200 import examples as ex
    ap = ex.ws_aperture(api)
    return flatten("f95", [ex.config1(api, 400, 3),
                           ex.config2_point(api, 150, 5. / 60. * np.pi / 180., ap, 5),
                           ex.config2_point(api, 60, 24. / 60. * np.pi / 180., ap, 6),
                           ex.config3(api, 300, 2),
                           ex.config4(api, 6, 20, order=-2, wave=2.4, rng_seed=4, offX=1e-4, offY=-2e-4),
                           ex.config5(api, 12, 20, offaxis=2e-4, rng_seed=7)], {})


def restated_python_layer():
    """The restatement of the reference's Python layer: oracle/pyref.py and the product's host helpers."""
    from pyxfocus_b200 import analyses as panal, conicsolve as pcon, transformations as ptran

    def coords():
        c = ptran.newCoords()
        ptran._update_coords_fwd(c, 1., 2., 3., .1, .2, .3)
        return c[1]
    return SimpleNamespace(sources=pyref, vignette=pyref.vignette, analyses=pyref, woltparam=pyref.woltparam,
                           focusI=pyref.focusI, radialGrad=panal.radialGrad, sellmeier=panal.sellmeier,
                           conicsolve=pcon, transformations=ptran, coords=coords)


def reference_python_layer(ref):
    """The same names on the reference's own modules (``refload.load()``)."""
    tran, con = ref.transformations, ref.conicsolve
    return SimpleNamespace(sources=ref.sources, vignette=tran.vignette, analyses=ref.analyses, woltparam=con.woltparam,
                           focusI=ref.surfaces.focusI, radialGrad=ref.analyses.radialGrad, sellmeier=ref.analyses.sellmeier,
                           conicsolve=con, transformations=tran,
                           coords=lambda: np.dot(np.dot(tran.rotationM(.1, .2, .3), tran.translationM(1., 2., 3.)),
                                                 tran.newCoords()[1]))


CONIC_EXACT = (("primrad", (8450., 220., 8400.)), ("secrad", (8350., 220., 8400.)), ("woltparam", (220., 8400.)),
               ("primfocus", (220., 8400.)), ("wsRMS", (1., 1e-3, 6e-3, 200., 1e4)), ("wsFoc", (3., 1., 200., 1e4, 6e-3)))
CONIC_FINITE = (("primsag", (8500., 220., 8400.)), ("secsag", (8300., 8400., 220., 8400.)),
                ("rGoal_to_rMax", (221., 8400., 8500.)), ("ellipsoidRad", (1e5, 1., 220., 8400., 8450.)),
                ("ehSecRad", (1e5, 1., 220., 8400., 8350.)), ("ellipsoidSag", (1e5, 1., 220., 8400., 8500., 8400.)),
                ("solveS", (8500., 9000., 30., .99, 8900., 0., 0., -1., 0., 0., 1.)))
# compared within an absolute tolerance, as the reference's matrices are (the product composes them differently)
PYTHON_ATOL = {"py.rotationM.0": 1e-16, "py.rotationM.1": 1e-16, "py.coords": 1e-15}


def python_layer_values(L):
    out = {}
    for name, args in (("subannulus", (220., 220.6, 1.3, 5001, -1.)), ("annulus", (200., 230., 5001, 1.)),
                       ("circularbeam", (12.5, 5001)), ("pointsource", (.03, 5001))):
        np.random.seed(11)
        out["py.src." + name] = np.array(getattr(L.sources, name)(*args))
    for name, args in (("xslit", (-3., 5., 257, 1.)), ("rectArray", (4., 2.5, 33)),
                       ("convergingbeam", (8400., 200., 230., -.1, .3, 4001, 1.5)),
                       ("convergingbeam2", (8400., -20., 30., 190., 240., 4001, .5)),
                       ("rectbeam", (12., 7., 4001)), ("gaussianBeam", (.01, 4001)),
                       ("fanBeam", (.02, .03, 21)), ("circFan", (.05, 7, 12))):
        np.random.seed(13)
        out["py.src." + name] = np.array(getattr(L.sources, name)(*args))
    rays = chains.wolter1_source(5001, 12)
    chains.run_steps_cpu(rays, chains.wolter1_steps())
    rays[6][::13] = np.nan
    rays[4][::17] = 0.; rays[5][::17] = 0.; rays[6][::17] = 0.
    out["py.vignette"] = np.array(L.vignette([r.copy() for r in rays]))
    good = pyref.vignette([r.copy() for r in rays])
    w = np.random.default_rng(12).uniform(.2, 3., good[1].size)
    for fn in ("centroid", "rmsCentroid", "hpd", "analyticImagePlane"):
        for tag, ww in (("", None), (".w", w)):
            out["py.%s%s" % (fn, tag)] = np.array(getattr(L.analyses, fn)(good, weights=ww))
    out["py.rhocdf.r"], out["py.rhocdf.cdf"] = L.analyses.rhocdf(good, weights=w)
    out["py.woltparam"] = np.array(L.woltparam(220., 8400.))
    a = [r.copy() for r in good]
    out["py.focusI"] = np.array(L.focusI(a))
    out["py.focusI.rays"] = np.array(a)
    xs, ys = np.linspace(-3., 4., 11), np.linspace(1., 9., 11)
    flatten("py.radialGrad", L.radialGrad(xs, ys, 2e-4, .03, 11832.), out)
    out["py.sellmeier"] = np.array(L.sellmeier([.5, .6, .7], [1.03, .23, 1.01], [6e-3, 2e-2, 103.]))
    for f, args in CONIC_EXACT + CONIC_FINITE:
        out["py.con." + f] = np.array(getattr(L.conicsolve, f)(*args))
    for inv in (False, True):
        out["py.rotationM.%d" % inv] = L.transformations.rotationM(.1, -.2, .3, inverse=inv)
    out["py.translationM"] = L.transformations.translationM(1., 2., 3.)
    out["py.coords"] = L.coords()
    return out


def interp_rays():
    rng = np.random.default_rng(4)
    n = 3000
    r, t = 12.5 * np.sqrt(rng.uniform(0, 1, n)), rng.uniform(0, 2 * np.pi, n)
    x, y = r * np.cos(t), r * np.sin(t)
    l, m = 1e-3 * np.sin(x / 5.) + 1e-5 * rng.normal(size=n), 1e-3 * np.cos(y / 7.) + 1e-5 * rng.normal(size=n)
    zero = np.zeros(n)
    return [zero.copy(), x, y, zero.copy(), l, m, np.sqrt(1 - l ** 2 - m ** 2), zero.copy(), zero.copy(), zero + 1.]


def interp_values(interpolate_vec, wavefront):
    """interpolateVec(rays, 4, 31, 23, **kw) for five argument sets and wavefront(rays, 20, 16) for two methods."""
    import warnings
    rays = interp_rays()
    out = {}
    for j, kw in enumerate((dict(method="linear"), dict(method="nearest"), dict(method="cubic"),
                            dict(method="linear", polar=True),
                            dict(method="linear", xr=[-3., 9.], yr=[-14., 2.], interpVec=rays[1] * rays[2]))):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            flatten("interp.iv%d" % j, interpolate_vec([r.copy() for r in rays], 4, 31, 23, **kw), out)
    for method in ("linear", "cubic"):
        flatten("interp.wf." + method, wavefront([r.copy() for r in rays], 20, 16, method=method), out)
    return out


def restated_interp():
    return refapi.interpolateVec, lambda rays, nx, ny, method: refapi.wavefront(rays, nx, ny, method=method, maxiter=500)


def reference_interp(ref):
    """The reference's own analyses.py, with the two things it lacks as shipped supplied from outside:
    ``man.padRect`` (un-vendored; a one-pixel NaN frame) and a ``reconstruct`` whose ``maxiter`` has a default (the
    reference omits the required argument, analyses.py:327)."""
    from oracle import f2py as of
    anal = ref.analyses

    def pad_rect(img):
        out = np.full((img.shape[0] + 2, img.shape[1] + 2), np.nan)
        out[1:-1, 1:-1] = img
        return out
    anal.man.padRect = pad_rect
    anal.reconstruct.reconstruct = lambda xa, ya, crit, h, ph, maxiter=500: of.reconstruct.reconstruct(xa, ya, crit, h, ph, maxiter)
    return anal.interpolateVec, lambda rays, nx, ny, method: anal.wavefront(rays, nx, ny, method=method)


def main():
    from pyxfocus_b200 import examples as ex
    if "--restatement" in sys.argv:
        api = ex.make_api(refapi.load(), ex.NumpyXP, "refapi")
        py, interp = restated_python_layer(), restated_interp()
        f95 = api
    else:
        from oracle import f95mods
        ref = refload.load()
        api = ex.make_api(ref, ex.NumpyXP, "reference")
        py, interp = reference_python_layer(ref), reference_interp(ref)
        f95 = ex.make_api(refload.load(f2py_modules=f95mods.modules()), ex.NumpyXP, "reference over its own Fortran")
    for name, values in (("reference_api", api_runs(api)), ("reference_python", python_layer_values(py)),
                         ("reference_interp", interp_values(*interp)), ("reference_f95", f95_runs(f95))):
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **pinned(values))
        print("%-22s %4d arrays  %7d bytes" % (name, len(values), os.path.getsize(path)))


if __name__ == "__main__":
    main()
