"""Cases shared by the GPU tests of conicplus, legsurf, zernphase and the rotated Zernike surface as fused-program ops,
their interpreter-vs-specialised runner and the benchmark: bundles resampled from the surfaces2 fixtures (rays at
which each routine does real work), one program per op, and segmented programs with per-segment tables."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = np.load(os.path.join(ROOT, "tests", "golden", "surfaces2.npz"))
RO, AO = G["z_rorder"], G["z_aorder"]
LEG = (25., 30., 2., G["leg_coeff"], G["leg_xo"], G["leg_yo"])
# the fixture each bundle is drawn from
KEYS = {"conicplus": "conicplus_in", "conicplusopd": "conicplus_in", "legsurf": "legsurf_in",
        "zernphase": "zernphase_in", "zernrot": "zernrot_in", "asphere": "conicplus_in", "leg_behind_sphere": "legsurf_in"}


def source(name, num, seed=0):
    """num rays of the fixture of ``name``: its rays repeated, positions jittered by 1e-6 relative"""
    g = G[KEYS[name]]
    idx = np.random.default_rng(seed).integers(0, g.shape[1], num)
    rows = [np.array(g[k][idx], dtype=np.float64) for k in range(10)]
    jit = np.random.default_rng(seed + 1).normal(0., 1e-6, (2, num))
    rows[1] = rows[1] * (1. + jit[0])
    rows[2] = rows[2] * (1. + jit[1])
    return rows


def vig_hi(name):
    """|x| below which a ray passes the vignette of the programs below: about half of the bundle"""
    return float(np.median(np.abs(G[KEYS[name]][1])))


def add_op(prog, name, k=0):
    """the op of ``name`` (k: the segment, whose terms / wave / rot differ)"""
    s = 1. + .01 * k
    if name == "conicplus":
        return prog.conicplus(800., -1.3, G["conicplus_p"] * s)
    if name == "conicplusopd":
        return prog.conicplusopd(800., -1.3, G["conicplus_p"] * s, 1.1)
    if name == "legsurf":
        return prog.legsurf(LEG[0], LEG[1], LEG[2], LEG[3] * s, LEG[4], LEG[5])
    if name == "zernphase":
        return prog.zernphase(G["z_coeff"], RO, AO, 20., 5.e-4 * s)
    if name == "zernrot":
        return prog.tracezernrot(G["z_coeff"], RO, AO, G["z_coeff2"], RO[:10], AO[:10], 20., .37 + .01 * k)
    raise KeyError(name)


def asphere_terms(n=8):
    return np.array([(-1.) ** j * 10. ** (-6 - 3 * j) for j in range(n)])


def call_surfaces(pxf, rays, name):
    """the op through pxf.surfaces (recorded when inside ``fused``, else the stand-alone routine)"""
    S = pxf.surfaces
    if name == "conicplus":
        S.conicplus(rays, 800., -1.3, G["conicplus_p"])
    elif name == "conicplusopd":
        S.conicplus(rays, 800., -1.3, G["conicplus_p"], nr=1.1)
    elif name == "legsurf":
        S.legSurf(rays, *LEG)
    elif name == "zernphase":
        S.zernphase(rays, G["z_coeff"], 20., 5.e-4, rorder=RO, aorder=AO)
    elif name == "zernrot":
        S.zernsurfrot(rays, G["z_coeff"], G["z_coeff2"], 20., .37, rorder1=RO, aorder1=AO, rorder2=RO[:10],
                      aorder2=AO[:10])
    elif name == "asphere":
        # an aspheric singlet: a sphere front, a conicplus back, refract between
        T = pxf.transformations
        T.transform(rays, 0, 0, 0, 0, 0, 0)
        S.sphere(rays, -900.)
        T.refract(rays, 1., 1.5)
        T.transform(rays, 0, 0, -2., 0, 0, 0)
        S.conicplus(rays, 800., -1.3, asphere_terms())
        T.refract(rays, 1.5, 1.)
        T.transform(rays, 0, 0, -50., 0, 0, 0)
        S.flat(rays)
    elif name == "leg_behind_sphere":
        S.sphere(rays, 1.e4)
        S.legSurf(rays, *LEG)
    else:
        raise KeyError(name)


def _program(name):
    def make(pxf, vig):
        p = pxf.Program()
        if vig:
            p.vignette_abs(1, vig_hi(name))
        add_op(p, name)
        return p
    return make


PROGRAMS = {name: _program(name) for name in ("conicplus", "conicplusopd", "legsurf", "zernphase", "zernrot")}


def segment_sizes(nseg):
    return [(k * 37) % 101 for k in range(nseg)]


def _segmented(name, tail):
    def make(pxf, nseg):
        progs = [tail(add_op(pxf.Program(), name, k)) for k in range(nseg)]
        return progs, segment_sizes(nseg), name
    return make


SEGMENTED = {
    "conicplus": _segmented("conicplus", lambda p: p.refract(1., 1.5)),
    "legsurf": _segmented("legsurf", lambda p: p.transform(0, 0, 1., 0, 0, 0).flat()),
    "zernphase": _segmented("zernphase", lambda p: p.transform(0, 0, 1., 0, 0, 0).flat()),
    "zernrot": _segmented("zernrot", lambda p: p.reflect()),
}
