"""Edge bundles of the remaining scalar surfaces (sphere, cylinder, cylconic, paraxial, torus, conicplus, legsurf and
the Wolter-Schwarzschild back surfaces), shared by tests/test_surface_edge_cases_host.py, tests/test_gpu_surface_edges.py
and tests/run_surface_edges.py.  numpy only: the same bundles feed the C oracle on a machine without a GPU.

Every bundle holds N = 50 001 rays (odd: the double2 kernels run their one-ray tail), ordinary rays mixed with rays built
to land on one edge of the routine: ties between the two roots, zero discriminants built from integers, misses, rays at
the origin or on the axis, polynomial / Legendre edges and Newton iterations that never converge and stop at the
1000-iteration cap.  ``bundle(name)`` returns the ten rows and the index set of every constructed class; the classes
are shuffled into the bundle with a seeded permutation, so they meet both lanes of a double2 pair and the tail."""
import numpy as np

from oracle import f2py as of
from oracle import pyref

N = 50_001
NEWTON_CAP = 1000                       # PXF_NEWTON_CAP (pxf_ray.cuh, oracle/pxf_oracle.c)
TOL10 = float(np.float32(1e-10))        # the Newton tolerance 1.e-10 of surfacesf.f95, a REAL*4 literal
ALPHA = float(pyref.woltparam(220., 1.e4)[0])
WS_THICK = .4                           # as in surface_cases.py
LAYOUT = [0, 1, 2, 3, 2047, 2048, 2049, 0, 5001]


class Case:
    """One routine call: ``routine`` of oracle/f2py.py's ``mod`` (and of the product's f2py-shaped module of the same
    name), with the opd row or not, its scalars, and the bundle it runs on.  ``prog``: a Program method of that name
    exists (the fused-program ops).  ``exact``: + - * / sqrt only, compared bit for bit."""

    def __init__(self, name, routine, args, make, mod="surfacesf", opd=False, exact=True, special=False):
        self.name, self.routine, self.args, self.make = name, routine, args, make
        self.mod, self.opd, self.exact, self.special = mod, opd, exact, special
        self.prog = routine in PROGRAM_OPS


PROGRAM_OPS = ("tracesphere", "tracesphereopd", "tracecyl", "tracecylopd", "cylconic", "paraxial", "paraxialy",
               "torus", "wsprimaryback", "wssecondaryback")


# ------------------------------------------------------------------ bundle assembly
class _Builder:
    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.blocks = []                # (class name or None, [x, y, z, l, m, n])

    def add(self, cls, x, y, z, l, m, n):
        arrs = np.broadcast_arrays(*[np.asarray(a, dtype=np.float64) for a in (x, y, z, l, m, n)])
        self.blocks.append((cls, [np.array(a, dtype=np.float64).ravel() for a in arrs]))

    def unit(self, k, axis=2, sign=1., spread=.1):
        """k directions near sign * e_axis"""
        d = self.rng.normal(0., spread, (3, k))
        d[axis] = sign
        return d / np.sqrt((d ** 2).sum(0))

    def finish(self, ordinary):
        """ordinary(k) -> [x, y, z, l, m, n] fills the bundle up to N; returns (rows, classes)"""
        used = sum(b[1][0].size for b in self.blocks)
        assert used < N // 2, used
        self.blocks.append((None, ordinary(N - used)))
        six = [np.concatenate([b[1][k] for b in self.blocks]) for k in range(6)]
        labels = np.concatenate([np.full(b[1][0].size, -1 if b[0] is None else i) for i, b in enumerate(self.blocks)])
        perm = self.rng.permutation(N)
        last = int(np.flatnonzero(labels[perm] >= 0)[0])       # an edge ray in the double2 tail (the last ray)
        perm[[last, N - 1]] = perm[[N - 1, last]]
        six = [np.ascontiguousarray(a[perm]) for a in six]
        labels = labels[perm]
        classes = {}
        for i, (cls, _) in enumerate(self.blocks):
            if cls is not None:
                classes[cls] = np.concatenate([classes.get(cls, np.zeros(0, np.int64)), np.flatnonzero(labels == i)])
        u = self.rng.normal(0., 1., (3, N))
        u /= np.sqrt((u ** 2).sum(0))
        rows = [self.rng.normal(0., 1., N)] + six + [np.ascontiguousarray(c) for c in u]
        return rows, classes


def _signed_zeros(rng, k):
    return np.where(rng.random(k) < .5, 0., -0.)


SPECIALS = np.array([-0., 0., np.nan, np.inf, -np.inf, 5e-324, -5e-324, 2.2e-308, -1e-310,
                     1e300, -1e305, 2. ** 1017, -(2. ** 1016)])


def salt(rows, seed):
    """test_gpu_parity.special_value_bundle's recipe on a given bundle: an eighth of every row replaced by -0, +0, NaN,
    +-Inf, denormals and huge values"""
    rng = np.random.default_rng(seed + 1000)
    rows = [np.array(r, copy=True) for r in rows]
    for r in rows:
        idx = rng.choice(N, N // 8, replace=False)
        r[idx] = rng.choice(SPECIALS, idx.size)
    return rows


# ------------------------------------------------------------------ sphere / cylinder
PYTH15 = [(0., 15.), (9., 12.), (12., 9.), (15., 0.)]         # a**2 + b**2 == 15**2 in integers


def _sphere(seed, R):
    b = _Builder(seed)
    rng = b.rng
    a = abs(R)
    # two roots of equal magnitude: the direction is an axis, the position has no component along it (dotol == 0)
    k = 600
    u = rng.uniform(-.7, .7, (2, k)) * a
    z0 = _signed_zeros(rng, k)
    s = np.where(rng.random(k) < .5, 1., -1.)
    zero = np.zeros(k)
    b.add("dotol0", u[0], u[1], z0, zero, zero, s)
    b.add("dotol0", u[0], z0, u[1], zero, s, zero)
    b.add("dotol0", z0, u[0], u[1], s, zero, zero)
    # det == 0 from integers: (p, q) on the circle of radius 15, any integer offset c along the axis direction
    for p, q in PYTH15:
        for sp in (1., -1.):
            for sq_ in (1., -1.):
                c = rng.integers(-40, 41, 40).astype(float)
                one = np.where(rng.random(40) < .5, 1., -1.)
                b.add("det0", sp * p, sq_ * q, c, 0., 0., one)
                b.add("det0", c, sp * p, sq_ * q, one, 0., 0.)
    # det slightly negative: just outside the circle, small offsets
    c = rng.integers(-3, 4, 300).astype(float)
    b.add("grazing_miss", 9., np.nextafter(12., 13.), c, 0., 0., 1.)
    b.add("grazing_miss", np.nextafter(-15., -16.), 0., c, 0., 0., -1.)
    # through the centre (position along the direction) and at the origin (zero direction: the normal is 0/0)
    t = rng.uniform(-3., 3., 300) * a
    b.add("centre", 0., 0., t, 0., 0., 1.)
    b.add("centre", t, -0., 0., -1., 0., 0.)
    d = b.unit(200)
    b.add("origin", _signed_zeros(rng, 200), _signed_zeros(rng, 200), _signed_zeros(rng, 200), d[0], d[1], d[2])
    b.add("origin_nodir", _signed_zeros(rng, 50), 0., -0., 0., -0., 0.)
    # starting inside
    p = rng.normal(0., 1., (3, 2000))
    p *= a * .9 * rng.random(2000) ** (1 / 3.) / np.sqrt((p ** 2).sum(0))
    d = b.unit(2000, spread=1.)
    b.add("inside", p[0], p[1], p[2], d[0], d[1], d[2])

    def ordinary(k):
        p = rng.normal(0., .8 * a, (3, k))
        d = b.unit(k, spread=1.)
        return [p[0], p[1], p[2], d[0], d[1], d[2]]
    return b.finish(ordinary)


def _cyl(seed, R):
    b = _Builder(seed)
    rng = b.rng
    a = abs(R)
    # b == 0 (x*l + z*n == 0 exactly): the two roots have equal magnitude
    k = 600
    u = rng.uniform(-.7, .7, k) * a
    y = rng.normal(0., 10., k)
    s = np.where(rng.random(k) < .5, 1., -1.)
    m = rng.normal(0., .3, k)
    b.add("b0", u, y, _signed_zeros(rng, k), 0., m, s)
    b.add("b0", _signed_zeros(rng, k), y, u, s, m, 0.)
    # det == 0 from integers: tangent to the circle of radius 15 in x, z
    for p, q in PYTH15:
        for sp in (1., -1.):
            c = rng.integers(-40, 41, 40).astype(float)
            yy = rng.normal(0., 10., 40)
            if q == 0.:
                b.add("det0", sp * p, yy, c, 0., 0., 1.)
            if p == 0.:
                b.add("det0", c, yy, sp * q, 1., 0., 0.)
            b.add("det0", sp * p, yy, q, 0., 0., 0.)                      # on the circle, along y: a = 0, det = 0
    c = rng.integers(-3, 4, 300).astype(float)
    b.add("grazing_miss", np.nextafter(15., 16.), rng.normal(0., 10., 300), c, 0., 0., 1.)
    # parallel to the axis (l = n = 0: a = 0) and on the axis (x = z = 0)
    b.add("axial", rng.normal(0., a, 300), rng.normal(0., 10., 300), rng.normal(0., a, 300), 0., 1., 0.)
    b.add("axial", rng.normal(0., a, 300), rng.normal(0., 10., 300), rng.normal(0., a, 300), -0., -1., -0.)
    d = b.unit(300, axis=0, spread=1.)
    b.add("on_axis", _signed_zeros(rng, 300), rng.normal(0., 10., 300), _signed_zeros(rng, 300), d[0], d[1], d[2])
    p = rng.normal(0., 1., (2, 2000))
    p *= a * .9 * np.sqrt(rng.random(2000)) / np.sqrt((p ** 2).sum(0))
    d = b.unit(2000, spread=1.)
    b.add("inside", p[0], rng.normal(0., 10., 2000), p[1], d[0], d[1], d[2])

    def ordinary(k):
        p = rng.normal(0., .8 * a, (3, k))
        d = b.unit(k, spread=1.)
        return [p[0], p[1], p[2], d[0], d[1], d[2]]
    return b.finish(ordinary)


# ------------------------------------------------------------------ cylconic (y = sag(x), rays along +y)
def _cylconic(seed, rad, K, beyond=None):
    b = _Builder(seed)
    rng = b.rng
    # Fp = 0: x = +-0 and m = 0 (Fx = 0 at the vertex)
    k = 300
    b.add("fp0", _signed_zeros(rng, k), rng.uniform(-20., 20., k), rng.normal(0., 10., k),
          rng.uniform(-.9, .9, k), _signed_zeros(rng, k), rng.uniform(-.3, .3, k))
    if beyond is not None:               # 1 - A x**2 < 0: the sag's root is NaN
        x = beyond * rng.uniform(1.01, 1.3, k) * np.where(rng.random(k) < .5, 1., -1.)
        d = b.unit(k, axis=1, spread=.05)
        b.add("root_nan", x, -5., rng.normal(0., 10., k), d[0], d[1], d[2])
    if K <= -1.:
        # a line below the vertex whose slope is too small to reach the sag (no root: Newton never converges)
        x0 = rng.uniform(-5., 5., 1000)
        y0 = -10. - rng.uniform(0., 10., 1000)
        slope = rng.uniform(-.1, .1, 1000)
        ll = np.where(rng.random(1000) < .5, 1., -1.) / np.sqrt(1. + slope ** 2)
        b.add("cap", x0, y0, rng.normal(0., 10., 1000), ll, ll * slope, 0.)

    def ordinary(k):
        d = b.unit(k, axis=1, spread=.1)
        return [rng.uniform(-40., 40., k), np.full(k, -30.), rng.normal(0., 10., k), d[0], d[1], d[2]]
    return b.finish(ordinary)


# ------------------------------------------------------------------ torus (axis of revolution: x, through z = -(rin+rout))
def _torus(seed, rin, rout):
    b = _Builder(seed)
    rng = b.rng
    k = 300
    d = b.unit(k, sign=-1., spread=.05)
    b.add("near_axis", _signed_zeros(rng, k), _signed_zeros(rng, k), rng.uniform(5., 30., k), d[0], d[1], d[2])
    b.add("on_axis", _signed_zeros(rng, k), _signed_zeros(rng, k), rng.uniform(5., 30., k), 0., 0., -1.)
    # beyond the tube's half width rin in x, travelling along z: no root, Newton never converges (the few candidates
    # that land on a root by chance are left out)
    x = (rin + rng.uniform(50., 250., 1600)) * np.where(rng.random(1600) < .5, 1., -1.)
    d = b.unit(1600, sign=-1., spread=.01)
    cand = [x, rng.uniform(-50., 50., 1600), np.full(1600, 20.), d[0], d[1], d[2]]
    keep = replay_torus([None] + cand, rin, rout) == NEWTON_CAP
    b.add("cap", *[c[keep][:1500] for c in cand])

    def ordinary(k):
        d = b.unit(k, sign=-1., spread=.05)
        w = .6 * min(rin, 100.)
        return [rng.uniform(-w, w, k), rng.uniform(-w, w, k), np.full(k, 20.), d[0], d[1], d[2]]
    return b.finish(ordinary)


# ------------------------------------------------------------------ conicplus (z = sag(rho) - poly, rays along -z)
def _conicplus(seed, R, K, cap=False, beyond=None):
    b = _Builder(seed)
    rng = b.rng
    k = 300
    d = b.unit(k, sign=-1., spread=.05)
    b.add("on_axis", _signed_zeros(rng, k), _signed_zeros(rng, k), rng.uniform(5., 30., k), d[0], d[1], d[2])
    if beyond is not None:
        phi = rng.uniform(0., 2 * np.pi, k)
        r = beyond * rng.uniform(1.01, 1.3, k)
        d = b.unit(k, sign=-1., spread=.01)
        b.add("root_nan", r * np.cos(phi), r * np.sin(phi), 10., d[0], d[1], d[2])
    if cap:
        # nearly horizontal rays on the side the sag curves away from: no root, Newton never converges
        side = 1. if R < 0 else -1.
        nn = rng.uniform(-.05, .05, 1000)
        ll = np.where(rng.random(1000) < .5, 1., -1.) * np.sqrt(1. - nn ** 2)
        b.add("cap", rng.uniform(-5., 5., 1000), rng.uniform(2., 20., 1000) * np.where(rng.random(1000) < .5, 1., -1.),
              side * rng.uniform(10., 20., 1000), ll, 0., nn)

    def ordinary(k):
        d = b.unit(k, sign=-1., spread=.05)
        return [rng.uniform(-40., 40., k), rng.uniform(-40., 40., k), np.full(k, 30.), d[0], d[1], d[2]]
    return b.finish(ordinary)


def conicplus_terms(n, seed=7, rho=40.):
    """n polynomial terms, each worth ~1e-3 at rho"""
    rng = np.random.default_rng(seed)
    return np.array([rng.choice([-1., 1.]) * rng.uniform(.5, 1.5) * 1e-3 / rho ** (2 * j) for j in range(1, n + 1)])


# ------------------------------------------------------------------ legsurf (a Legendre phase grating on x/xwidth, y/ywidth)
LEG_W = (2., 30.)          # xwidth, ywidth


def leg_terms(nc, seed=11):
    """nc terms with every order 0..15 on both axes (for nc >= 16)"""
    rng = np.random.default_rng(seed)
    j = np.arange(nc)
    xo = (j % 16).astype(np.int32)
    yo = np.where(j < 16, 15 - j % 16, (5 * j + 3) % 16).astype(np.int32)
    return rng.normal(0., 1e-3, nc), xo, yo


def _legsurf(seed):
    b = _Builder(seed)
    rng = b.rng
    xw, yw = LEG_W

    def edges(w):
        return np.array([w, -w, 0., -0., np.nextafter(w, 0.), np.nextafter(-w, 0.), np.nextafter(w, 2 * w),
                         np.nextafter(-w, -2 * w), .5 * w, -.25 * w])
    ex, ey = edges(xw), edges(yw)
    gx, gy = np.meshgrid(ex, ey)
    for rep in range(6):
        k = gx.size
        d = b.unit(k, sign=rng.choice([-1., 1.]), spread=.2)
        b.add("width_edge", gx.ravel(), gy.ravel(), rng.normal(0., 1., k), d[0], d[1], d[2])
    k = 300
    d = b.unit(k, spread=.2)
    b.add("n_zero", rng.uniform(-xw, xw, k), rng.uniform(-yw, yw, k), 0., d[0], d[1], _signed_zeros(rng, k))
    # l**2 + m**2 just below 1: the kick pushes part of them beyond (n becomes NaN)
    ll = rng.uniform(.995, .9999, 2000) * np.where(rng.random(2000) < .5, 1., -1.)
    mm = np.sqrt(1. - ll ** 2) * rng.uniform(.5, .999, 2000)
    b.add("steep", rng.uniform(-xw, xw, 2000), rng.uniform(-yw, yw, 2000), 0., ll, mm,
          np.sqrt(np.maximum(1. - ll ** 2 - mm ** 2, 0.)))

    def ordinary(k):
        d = b.unit(k, spread=.2)
        return [rng.uniform(-1.2 * xw, 1.2 * xw, k), rng.uniform(-1.2 * yw, 1.2 * yw, k), rng.normal(0., 1., k),
                d[0], d[1], d[2]]
    return b.finish(ordinary)


# ------------------------------------------------------------------ paraxial
def _paraxial(seed):
    b = _Builder(seed)
    rng = b.rng
    k = 400
    d = b.unit(k, spread=.1)
    b.add("zero_xy", _signed_zeros(rng, k), _signed_zeros(rng, k), 0., d[0], d[1], d[2])

    def ordinary(k):
        d = b.unit(k, spread=.1)
        return [rng.normal(0., 20., k), rng.normal(0., 20., k), np.zeros(k), d[0], d[1], d[2]]
    return b.finish(ordinary)


# ------------------------------------------------------------------ Wolter-Schwarzschild back surfaces
def ws_source(seed, arcmin):
    """the surfaces2.npz W-S back-surface bundle (make_golden.py) tilted by a field angle"""
    a0, a1 = _ws_aperture()
    np.random.seed(seed)
    rays = pyref.subannulus(a0 + WS_THICK, a1 + WS_THICK, .3, N, zhat=-1.)
    th = arcmin / 60. * np.pi / 180.
    rays[4][:] = rays[4] + np.sin(th)
    rays[6][:] = -np.sqrt(1. - rays[4] ** 2 - rays[5] ** 2)
    pyref.transform(rays, 0, 0, -1.e4, 0, 0, 0)
    return rays


def _ws_aperture():
    from oracle import chains
    return chains.ws_aperture(220., 1.e4, 1., 200.)


def _ws(arcmin, secondary):
    rays = ws_source(28 + int(arcmin), arcmin)
    if secondary:                  # the secondary sees what the primary and a reflection made of the bundle
        of.woltsurf.wsprimaryback(*rays[1:], ALPHA, 1.e4, 1., WS_THICK)
        of.transformationsf.reflect(*rays[4:])
    return rays, {}


# ------------------------------------------------------------------ the cases
def _cases():
    c = {}

    def add(case):
        c[case.name] = case
    for R in (15., -15.):
        tag = "p" if R > 0 else "m"
        add(Case("tracesphere_R%s" % tag, "tracesphere", (R,), lambda R=R: _sphere(1, R)))
        add(Case("tracesphereopd_R%s" % tag, "tracesphereopd", (R, 1.5), lambda R=R: _sphere(2, R), opd=True))
        add(Case("tracecyl_R%s" % tag, "tracecyl", (R,), lambda R=R: _cyl(3, R)))
        add(Case("tracecylopd_R%s" % tag, "tracecylopd", (R, 1.2), lambda R=R: _cyl(4, R), opd=True))
    add(Case("cylconic_Km1", "cylconic", (1. / 400., -1.), lambda: _cylconic(5, 1. / 400., -1.)))
    add(Case("cylconic_K0", "cylconic", (1. / 100., 0.), lambda: _cylconic(6, 1. / 100., 0., beyond=100.)))
    add(Case("cylconic_Km3", "cylconic", (1. / 400., -3.), lambda: _cylconic(7, 1. / 400., -3.)))
    add(Case("cylconic_K2", "cylconic", (1. / 400., 2.), lambda: _cylconic(8, 1. / 400., 2., beyond=400. / np.sqrt(3.))))
    add(Case("torus_in_lt_out", "torus", (150., 900.), lambda: _torus(9, 150., 900.)))
    add(Case("torus_in_gt_out", "torus", (900., 150.), lambda: _torus(10, 900., 150.)))
    cp = [("conicplus_0_Rm_Km1", (-500., -1., conicplus_terms(0)), dict(cap=True)),
          ("conicplus_1", (800., -1.3, conicplus_terms(1)), {}),
          ("conicplus_3_rootnan", (300., .5, conicplus_terms(3)), dict(beyond=300. / np.sqrt(1.5))),
          ("conicplus_16_Km1", (800., -1., conicplus_terms(16)), {})]
    for k, (name, args, kw) in enumerate(cp):
        add(Case(name, "conicplus", args, lambda kw=kw, a=args, k=k: _conicplus(12 + k, a[0], a[1], **kw)))
        add(Case(name.replace("conicplus", "conicplusopd"), "conicplusopd", args + (1.1,),
                 lambda kw=kw, a=args, k=k: _conicplus(20 + k, a[0], a[1], **kw), opd=True))
    for nc in (0, 5, 48):
        co, xo, yo = leg_terms(nc)
        add(Case("legsurf_%d" % nc, "legsurf", LEG_W + (2., co, xo, yo), lambda: _legsurf(30)))
    for tag, F in (("350", 350.), ("-120", -120.), ("p0", 0.), ("m0", -0.), ("1e308", 1e308), ("-1e308", -1e308)):
        add(Case("paraxial_F%s" % tag, "paraxial", (F,), lambda: _paraxial(40)))
        add(Case("paraxialy_F%s" % tag, "paraxialy", (F,), lambda: _paraxial(41)))
    for arcmin in (0., 5., 10., 15.):
        for sec in (False, True):
            r = "wssecondaryback" if sec else "wsprimaryback"
            add(Case("%s_%d" % (r, arcmin), r, (ALPHA, 1.e4, 1., WS_THICK),
                     lambda a=arcmin, s=sec: _ws(a, s), mod="woltsurf", exact=False))
    # special-value variants of the algebraic routines
    for base in ("tracesphere_Rp", "tracesphereopd_Rm", "tracecyl_Rp", "tracecylopd_Rm", "cylconic_Km1", "torus_in_lt_out",
                 "conicplus_3_rootnan", "conicplusopd_16_Km1", "legsurf_48", "paraxial_F350", "paraxialy_F-120"):
        b = c[base]
        add(Case(base + "_sv", b.routine, b.args, lambda b=b, s=len(c): (salt(b.make()[0], s), {}), opd=b.opd,
                 special=True))
    return c


CASES = _cases()
EXACT = sorted(n for n, c in CASES.items() if c.exact)
WS = sorted(n for n, c in CASES.items() if not c.exact)
PROGRAM = sorted(n for n, c in CASES.items() if c.prog)
_memo = {}


def bundle(name):
    """(rows, classes) of a case: fresh copies of the ten rows, and the index array of every constructed class"""
    if name not in _memo:
        _memo[name] = CASES[name].make()
    rows, classes = _memo[name]
    return [np.array(r, copy=True) for r in rows], classes


def call_args(case, rows):
    """positional arguments of the f2py-shaped call on ten rows"""
    return (list(rows) if case.opd else list(rows[1:])) + list(case.args)


def oracle(case, rows):
    """the case's routine on the C oracle, in place"""
    getattr(getattr(of, case.mod), case.routine)(*call_args(case, rows))


def oracle_flat(rows):
    of.surfacesf.flat(*rows[1:])


# ------------------------------------------------------------------ Newton replays with an iteration counter
def _loop(step, state, tol=TOL10):
    """while (fabs(delt) > tol && it++ < CAP) step(): returns the number of passes of each ray"""
    delt = np.full(state[0].shape, 100.)
    it = np.zeros(state[0].shape, np.int64)
    with np.errstate(all="ignore"):
        for _ in range(NEWTON_CAP):
            go = np.abs(delt) > tol
            if not go.any():
                break
            it += go
            d = step(state)
            delt = np.where(go, d, delt)
            for k in range(3):
                state[k] = np.where(go, state[k] + state[3 + k] * d, state[k])
    return it


def replay_cylconic(rows, rad, K):
    A = (1 + K) * rad * rad

    def step(s):
        x, y = s[0], s[1]
        root = np.sqrt(1 - A * x * x)
        low, high = 1 + root, rad * (x * x)
        dL, dH = -(A * x / root), 2 * rad * x
        F = y - high / low
        Fx = (high * dL - low * dH) / (low * low)
        return -F / (Fx * s[3] + 1. * s[4])
    return _loop(step, [np.array(rows[k], copy=True) for k in (1, 2, 3, 4, 5, 6)])


def replay_torus(rows, rin, rout):
    def step(s):
        x, y, z = s[0], s[1], s[2]
        t = z + rin + rout
        F = (t * t + y * y + x * x + rout * rout - rin * rin) ** 2 - 4 * rout * rout * (y * y + t * t)
        S = rin + rout + z
        Fx = 4 * x * (-rin * rin + S * S + rout * rout + x * x + y * y)
        G = 2 * rin * (rout + z) + 2 * rout * z + z * z + y * y + x * x
        return -F / (Fx * s[3] + 4 * y * G * s[4] + 4 * S * G * s[5])
    return _loop(step, [np.array(rows[k], copy=True) for k in (1, 2, 3, 4, 5, 6)])


def replay_conicplus(rows, R, K, p):
    c = 1 / R

    def step(s):
        x, y, z = s[0], s[1], s[2]
        rad = np.sqrt(x * x + y * y)
        a0 = sum(p[j - 1] * rad ** (2 * j) for j in range(1, len(p) + 1))
        a1 = sum(p[j - 1] * (2 * j) * rad ** (2 * j - 1) for j in range(1, len(p) + 1))
        root = np.sqrt(1 - (K + 1) * c * c * rad * rad)
        denom = root + 1
        F = z - c * rad * rad / denom + a0
        Fr = -(2 * c * rad / denom + (K + 1) * rad ** 3 * c ** 3 / (denom * denom * root)) + a1
        return -F / (Fr * x / rad * s[3] + Fr * y / rad * s[4] + s[5])
    return _loop(step, [np.array(rows[k], copy=True) for k in (1, 2, 3, 4, 5, 6)])


def replay(case, rows):
    """iteration count of every ray of a cylconic / torus / conicplus case"""
    if case.routine == "cylconic":
        return replay_cylconic(rows, *case.args)
    if case.routine == "torus":
        return replay_torus(rows, *case.args)
    return replay_conicplus(rows, *case.args[:3])


# ------------------------------------------------------------------ segmented families (per-segment scalars at the edges)
def seg_sphere_scalars(k):
    # radius 1e-3: every ray of the segment misses (no ordinary ray passes within 1e-3 of the centre)
    return ((15., -15., 1e-3, 15., 1e-3, -40., 15., 7., 1e-3)[k], 1. + .1 * k)


def seg_paraxial_scalars(k):
    return ((350., -0., 0., -120., -0., 1e308, -1e308, 5., -0.)[k], (-120., 0., -0., -0., 350., -1e308, 2., -0., 80.)[k])


def seg_torus_scalars(k):
    return ((150., 900.), (900., 150.))[k % 2]


SEG = {
    "sphere": ("tracesphere_Rp", lambda P, k: P().tracesphereopd(*seg_sphere_scalars(k)),
               lambda rows, k: of.surfacesf.tracesphereopd(*rows, *seg_sphere_scalars(k))),
    "paraxial": ("paraxial_F350", lambda P, k: P().paraxial(seg_paraxial_scalars(k)[0]).paraxialy(seg_paraxial_scalars(k)[1]),
                 lambda rows, k: (of.surfacesf.paraxial(*rows[1:], seg_paraxial_scalars(k)[0]),
                                  of.surfacesf.paraxialy(*rows[1:], seg_paraxial_scalars(k)[1]))),
    "torus": ("torus_in_lt_out", lambda P, k: P().torus(*seg_torus_scalars(k)),
              lambda rows, k: of.surfacesf.torus(*rows[1:], *seg_torus_scalars(k))),
}


def seg_bundle(family):
    """sum(LAYOUT) rays of the family's edge bundle in bundle order, except that the sphere segments of radius 1e-3
    get ordinary rays only (no edge ray through the centre): every ray of those segments misses"""
    rows, classes = bundle(SEG[family][0])
    edge = np.zeros(N, bool)
    for v in classes.values():
        edge[v] = True
    plain = list(np.flatnonzero(~edge)[::-1])
    taken = np.zeros(N, bool)
    parts = [None] * len(LAYOUT)
    for k, size in enumerate(LAYOUT):
        if family == "sphere" and seg_sphere_scalars(k)[0] == 1e-3:
            parts[k] = np.array([plain.pop() for _ in range(size)], dtype=np.int64)
            taken[parts[k]] = True
    rest = iter(np.flatnonzero(~taken))
    for k, size in enumerate(LAYOUT):
        if parts[k] is None:
            parts[k] = np.array([next(rest) for _ in range(size)], dtype=np.int64)
    idx = np.concatenate(parts)
    where = np.full(N, -1)
    where[idx] = np.arange(idx.size)
    return [np.ascontiguousarray(r[idx]) for r in rows], {k: np.sort(where[v][where[v] >= 0]) for k, v in classes.items()}


def seg_oracle(family, rows):
    """segment k of the layout through the oracle with segment k's scalars, in place"""
    start = np.concatenate([[0], np.cumsum(LAYOUT)])
    for k in range(len(LAYOUT)):
        a, b = int(start[k]), int(start[k + 1])
        if a == b:
            continue
        part = [np.ascontiguousarray(r[a:b]) for r in rows]
        SEG[family][2](part, k)
        for r, p in zip(rows, part):
            r[a:b] = p


# ------------------------------------------------------------------ host-buffer path: a closing flat, then a surface op
HOST = {
    "paraxial": ("paraxial_F350", lambda P: P().flat().paraxial(350.), lambda r: of.surfacesf.paraxial(*r[1:], 350.)),
    "tracecyl": ("tracecyl_Rp", lambda P: P().flat().tracecyl(15.), lambda r: of.surfacesf.tracecyl(*r[1:], 15.)),
    "cylconic": ("cylconic_Km1", lambda P: P().flat().cylconic(1. / 400., -1.),
                 lambda r: of.surfacesf.cylconic(*r[1:], 1. / 400., -1.)),
    "tracesphere": ("tracesphere_Rp", lambda P: P().flat().tracesphere(15.),
                    lambda r: of.surfacesf.tracesphere(*r[1:], 15.)),
}


def host_oracle(name, rows):
    oracle_flat(rows)
    HOST[name][2](rows)
