"""The remaining scalar surfaces as fused-program ops: cases, programs, layouts and input bundles shared by
tests/test_gpu_surface_ops.py and tests/run_surface_compare.py (host side only: numpy in, numpy out).  Input bundles are
drawn from the surfaces2.npz fixtures, so every surface meets rays of the geometry it was pinned with."""
import os

import numpy as np

from pyxfocus_b200 import conicsolve

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALPHA = float(conicsolve.woltparam(220., 1.e4)[0])
T_IN = (-0., -0., .5, -0., -0., -0.)        # the transform in front of each surface
# segments straddle the 2048-ray tile boundaries, some are empty
LAYOUT = [0, 1, 2047, 2048, 2049, 3, 0, 5001, 7]

# name: (Program method, its scalars, fixture bundle, the op behind it is a reflection)
# Sphere and cylinder radii of 15 mm are smaller than the +-20 mm bundles: part of the rays miss (zeroed, NaN normal).
SINGLE = {
    "tracesphere": ("tracesphere", (15.,), "sphere_in", False),
    "tracesphereopd": ("tracesphereopd", (15., 1.5), "sphere_in", False),
    "tracecyl": ("tracecyl", (15.,), "cyl_in", False),
    "tracecylopd": ("tracecylopd", (15., 1.2), "cyl_in", False),
    "cylconic": ("cylconic", (1. / 400., -.7), "cylconic_in", True),
    "paraxial": ("paraxial", (350.,), "paraxial_in", False),
    "paraxialy": ("paraxialy", (-120.,), "paraxial_in", False),
    "torus": ("torus", (150., 900.), "torus_in", True),
    "wsprimaryback": ("wsprimaryback", (ALPHA, 1.e4, 1., .4), "wsback_in", True),
    "wssecondaryback": ("wssecondaryback", (ALPHA, 1.e4, 1., .4), "wsback_in", True),
}
# the routine of each op in the stand-alone modules (surfacesf / woltsurf), and whether it takes the opd row
ROUTINE = {
    "tracesphere": ("surfacesf", False), "tracesphereopd": ("surfacesf", True), "tracecyl": ("surfacesf", False),
    "tracecylopd": ("surfacesf", True), "cylconic": ("surfacesf", False), "paraxial": ("surfacesf", False),
    "paraxialy": ("surfacesf", False), "torus": ("surfacesf", False), "wsprimaryback": ("woltsurf", False),
    "wssecondaryback": ("woltsurf", False),
}


def fixture():
    return np.load(os.path.join(ROOT, "tests", "golden", "surfaces2.npz"))


def source(key, num, seed=0):
    """num rays drawn from the fixture bundle ``key``, transverse positions jittered by ~1 um (host rows)."""
    g = fixture()[key]
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, g.shape[1], num)
    rows = [np.ascontiguousarray(g[k][idx]) for k in range(10)]
    rows[1] = rows[1] + rng.normal(0., 1e-3, num)
    rows[2] = rows[2] + rng.normal(0., 1e-3, num)
    rows[0] = rng.normal(0., 1., num)
    return rows


def vig_cut(rows):
    """vignette_box on y: keeps roughly the lower half of the bundle"""
    return 2, -1e300, float(np.median(rows[2]))


def single_program(pxf, name, vig_rows=None):
    """transform, [wsprimaryback, reflect for the W-S secondary], the op, [vignette on y], reflect / refract, flatopd;
    vig_rows: the bundle the cut is taken from"""
    meth, args, _, refl = SINGLE[name]
    p = pxf.Program().transform(*T_IN)
    if name == "wssecondaryback":
        p.wsprimaryback(ALPHA, 1.e4, 1., .4).reflect()
    getattr(p, meth)(*args)
    if vig_rows is not None:
        p.vignette_box(*vig_cut(vig_rows))
    p.reflect() if refl else p.refract(1., 1.5)
    return p.flatopd(1.)


def single_routines(pxf, rows, name, upto_op=False):
    """single_program(name) as stand-alone calls on ten device rows (in place); upto_op: stop behind the op"""
    meth, args, _, refl = SINGLE[name]
    tf = pxf.transformationsf
    tf.transform(*rows[1:], *T_IN)
    if name == "wssecondaryback":
        pxf.woltsurf.wsprimaryback(*rows[1:], ALPHA, 1.e4, 1., .4)
        tf.reflect(*rows[4:])
    mod, with_opd = ROUTINE[name]
    getattr(getattr(pxf, mod), meth)(*(rows if with_opd else rows[1:]), *args)
    if upto_op:
        return
    if refl:
        tf.reflect(*rows[4:])
    else:
        tf.refract(*rows[4:], 1., 1.5)
    pxf.surfacesf.flatopd(*rows[1:], rows[0], 1.)


def single_name(name, vig):
    return "%s_vig%d" % (name, int(vig))


# segmented families: the fixture bundle and the program of segment k (scalars differ per segment)
def _lens(pxf, k):
    # a refracting pair of spheres; the first radius is below the bundle's extent for some segments (misses)
    return (pxf.Program().transform(-0., -0., 5. + .1 * k, -0., -0., -0.).tracesphereopd(20. + k % 7, 1.)
            .refract(1., 1.5).transform(0., 0., -10., 0., 0., 0.).tracesphere(40. + k % 5).refract(1.5, 1.).flatopd(1.))


def _cyl(pxf, k):
    return (pxf.Program().transform(-0., -0., .5 + .01 * k, -0., -0., -0.).tracecylopd(17. + k % 4, 1.2)
            .refract(1., 1.2).paraxial(300. + k).paraxialy(-100. - k).flatopd(1.))


def _conic(pxf, k):
    return (pxf.Program().transform(-0., -0., .01 * k, -0., -0., -0.).cylconic(1. / (400. + 10. * k), -.7).reflect()
            .flat())


def _torus(pxf, k):
    return pxf.Program().transform(-0., -0., .1 * k, -0., -0., -0.).torus(150., 900. + k).reflect().flat()


def _ws(pxf, k):
    t = .4 + .01 * k
    return (pxf.Program().transform(-0., -0., .05 * k, -0., -0., -0.).wsprimaryback(ALPHA, 1.e4, 1., t).reflect()
            .wssecondaryback(ALPHA, 1.e4, 1., t).reflect().flat())


SEG = {"lens": (_lens, "sphere_in"), "cyl": (_cyl, "cyl_in"), "conic": (_conic, "cylconic_in"),
       "torus": (_torus, "torus_in"), "ws": (_ws, "wsback_in")}
