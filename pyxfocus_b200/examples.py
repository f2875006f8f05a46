"""The BASELINE configurations, written the way the reference's example scripts are written.

Every ``configN(api, ...)`` below is plain PyXFocus script text -- ``sources.*`` / ``tran.*`` / ``surf.*`` /
``anal.*`` calls on a ten-row ray list plus array arithmetic for masks -- following the example scripts cited in
each docstring.  ``api`` bundles the five modules and the array namespace, so the SAME text runs on

* the reference's own Python layer (``oracle.refload``, build container only: produces ``tests/golden/config*.npz``),
* the CPU oracle's restatement of that layer (``oracle.refapi``: what the GPU parity tests compare against), and
* this package (``product_api()``): the drop-in claim, exercised call for call.

``configN_fast`` is the same computation arranged for the GPU: whole chains recorded into ONE fused program,
nested shells as ONE segmented launch, vignettes as in-kernel predicates + one compaction, sources drawn on
the device.  ``tests/test_gpu_examples.py`` holds ``fast == script == oracle`` (bit for bit where the routines
are algebraic, 1e-12 / 1e-9 otherwise); ``bench.py`` times the fast forms at the BASELINE sizes.

Nothing here imports ``oracle/``.
"""
import math
from types import SimpleNamespace

import numpy as np


# =============================================================================== back ends
class NumpyXP:
    """Array namespace of the reference scripts (numpy itself, plus the few spellings used below)."""
    sqrt, abs, arcsin, sign = np.sqrt, np.abs, np.arcsin, np.sign
    logical_and, logical_or, invert = np.logical_and, np.logical_or, np.invert
    concatenate = staticmethod(np.concatenate)

    @staticmethod
    def copy(a):
        return np.copy(a)

    @staticmethod
    def count(mask):
        return int(np.sum(mask))

    @staticmethod
    def repeat(v, n):
        return np.repeat(float(v), int(n))

    @staticmethod
    def arange(n):
        return np.arange(int(n))

    @staticmethod
    def asarray(a):
        return np.asarray(a, dtype=np.float64)

    @staticmethod
    def uniform(lo, hi, n):
        return np.random.uniform(lo, hi, size=int(n))

    @staticmethod
    def tonumpy(a):
        return np.asarray(a)


class TorchXP:
    """The same spellings over CUDA tensors: what a user's script does with the rows between library calls."""

    def __init__(self, device=None):
        import torch
        self.t = torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.sqrt, self.abs, self.arcsin, self.sign = torch.sqrt, torch.abs, torch.arcsin, torch.sign
        self.logical_and, self.logical_or, self.invert = torch.logical_and, torch.logical_or, torch.logical_not

    def concatenate(self, parts):
        return self.t.cat(list(parts))

    def copy(self, a):
        return a.clone()

    def count(self, mask):
        return int(mask.sum())

    def repeat(self, v, n):
        return self.t.full((int(n),), float(v), dtype=self.t.float64, device=self.device)

    def arange(self, n):
        return self.t.arange(int(n), device=self.device)

    def asarray(self, a):
        return self.t.as_tensor(np.asarray(a, dtype=np.float64), device=self.device)

    def uniform(self, lo, hi, n):
        # host MT19937 draw, uploaded: the same numbers as the numpy back ends
        return self.asarray(np.random.uniform(lo, hi, size=int(n)))

    def tonumpy(self, a):
        return a.detach().cpu().numpy()


def make_api(mods, xp, name):
    """mods: namespace with sources / transformations / surfaces / analyses / conicsolve."""
    return SimpleNamespace(sources=mods.sources, tran=mods.transformations, surf=mods.surfaces, anal=mods.analyses,
                           conic=mods.conicsolve, xp=xp, name=name)


def product_api(device=None):
    import pyxfocus_b200 as pxf
    return make_api(pxf, TorchXP(device), "pyxfocus_b200")


def seed(s):
    """The reference's sources draw from numpy's global MT19937 stream (sources.py:157-158)."""
    np.random.seed(int(s))


def findimageplane(api, rays, zscan, num, weights=None):
    """Legacy ``PyTrace.findimageplane(zscan,num)`` as the reference's examples call it
    (examples/axro/WSverify.py:74-77,161-164); the reference ships no definition (SURVEY.md 8c: parity unpinned).
    Literal scan: for each dz in linspace(-zscan,zscan,num): move the plane, trace to it, rmsCentroid; best dz.
    Back ends that define ``analyses.findimageplane`` (the product: one pass, exact quadratic) use their own."""
    if hasattr(api.anal, "findimageplane"):
        return api.anal.findimageplane(rays, zscan, num, weights=weights)
    scan = np.linspace(-zscan, zscan, int(num))
    rms = []
    for dz in scan:
        t = [api.xp.copy(r) for r in rays]
        api.tran.transform(t, 0, 0, dz, 0, 0, 0)
        api.surf.flat(t)
        rms.append(api.anal.rmsCentroid(t, weights=weights))
    return float(scan[int(np.argmin(rms))])


# =============================================================================== config 1
def config1(api, n=100_000, rng_seed=0):
    """Wolter-I pair, on-axis annular source at infinity, to the focal plane; HPD
    (examples/axro/singlePassAlignment.py:246-269 with secalign = 0; SURVEY.md 3.1 / 8d)."""
    src, tran, surf, anal = api.sources, api.tran, api.surf, api.anal
    seed(rng_seed)
    rays = src.subannulus(220., 220.6, 2 * np.pi, n, zhat=-1.)
    tran.transform(rays, 0, 0, -8400., 0, 0, 0)
    surf.wolterprimary(rays, 220., 8400.)
    tran.reflect(rays)
    surf.woltersecondary(rays, 220., 8400.)
    tran.reflect(rays)
    surf.flat(rays)
    return dict(rays=rays, hpd=anal.hpd(rays), rms=anal.rmsCentroid(rays))


# =============================================================================== config 2
WS = dict(R0=220., Z0=1.e4, psi=1., L=200., az=100., pmin=1.e4 + 25.)


def wsPrimrad(api, z, r0, z0, psi=1.):
    """Radius of the W-S primary at height z: one horizontal ray traced to the surface
    (examples/axro/axialHeights.py:51-62)."""
    ray = api.sources.pointsource(0., 1)
    api.tran.transform(ray, 0, 0, 0, 0, -np.pi / 2, 0)
    api.tran.transform(ray, -r0 - 2., 0, -z, 0, 0, 0)
    api.surf.wsPrimary(ray, r0, z0, psi)
    return float(ray[1][0])


def ws_aperture(api, R0=WS["R0"], Z0=WS["Z0"], psi=WS["psi"], L=WS["L"], pmin=WS["pmin"]):
    """axialHeights.py:86-87"""
    return wsPrimrad(api, pmin, R0, Z0, psi), wsPrimrad(api, pmin + L, R0, Z0, psi)


def config2_point(api, n, offaxis, aperture, rng_seed=0, R0=WS["R0"], Z0=WS["Z0"], psi=WS["psi"], az=WS["az"]):
    """One field point of the W-S sweep: the chain of ``traceZeta`` (examples/axro/axialHeights.py:77-113) to the
    nominal focal plane, the two-stage plane scan of the legacy sweep (examples/axro/WSverify.py:150-167:
    flat, findimageplane(20,100), findimageplane(1,100), flat) with its hpd / rms, then traceZeta's own
    refinement (focusI) and merit functions.  The scans come first on purpose: scanned from the best focus itself
    the two grid points next to zero tie and the literal scan picks one from rounding noise."""
    src, tran, surf, anal = api.sources, api.tran, api.surf, api.anal
    a0, a1 = aperture
    seed(rng_seed)
    rays = src.subannulus(a0, a1, az / R0, n)
    tran.transform(rays, 0, 0, -Z0, 0, 0, 0)
    surf.wsPrimary(rays, R0, Z0, psi)
    rays[4] = rays[4] + np.sin(offaxis)
    rays[6] = -api.xp.sqrt(1. - rays[4] ** 2)
    tran.reflect(rays)
    surf.wsSecondary(rays, R0, Z0, psi)
    tran.reflect(rays)
    surf.flat(rays)
    d2 = findimageplane(api, rays, 20., 100)
    tran.transform(rays, 0, 0, d2, 0, 0, 0)
    d3 = findimageplane(api, rays, 1., 100)
    tran.transform(rays, 0, 0, d3, 0, 0, 0)
    surf.flat(rays)
    hpd_scan, rms_scan = anal.hpd(rays), anal.rmsCentroid(rays)
    f = surf.focusI(rays)
    return dict(rays=rays, f=f, d2=d2, d3=d3, hpd_scan=hpd_scan, rms_scan=rms_scan, hpd=anal.hpd(rays),
                rms=anal.rmsCentroid(rays))


def config2(api, n=10_000_000, arcmin=None, aperture=None, rng_seed=0):
    """The field sweep: theta = linspace(0,30,31) arcmin (WSverify.py:194), seed reset per field point."""
    arcmin = np.linspace(0., 30., 31) if arcmin is None else arcmin
    aperture = ws_aperture(api) if aperture is None else aperture
    return [config2_point(api, n, a / 60. * np.pi / 180., aperture, rng_seed) for a in arcmin]


# =============================================================================== config 3
def zernike_orders(nmax=7):
    """Explicit (rorder, aorder), radial order ascending, |m| ascending, cosine (+m) before sine (-m): 36 terms for
    nmax = 7.  (The reference's default ordering lives in an un-vendored module, SURVEY.md 8c.)"""
    ro, ao = [], []
    for n in range(nmax + 1):
        for m in range(n % 2, n + 1, 2):
            ro.append(n); ao.append(m)
            if m:
                ro.append(n); ao.append(-m)
    return np.array(ro, dtype=np.int64), np.array(ao, dtype=np.int64)


def zernike_coeff(nterms=36, rng_seed=0, sigma=1.e-4):
    c = np.random.default_rng(rng_seed).normal(0., sigma, nterms)
    c[:3] = 0.          # piston / tilts zeroed (SURVEY.md 8d)
    return c


def config3(api, n=100_000_000, rng_seed=0):
    """Zernike figure error (36 terms) on a flat, relayed through a Wolter-I pair with two vignettes
    (examples/axro/singlePassAlignment.py:22-56 createWavefront, :133-187 traceThroughPair; the z / |y| aperture
    mask of examples/axro/slf.py:145-147; SURVEY.md 8d).  Returns the surviving bundle and ``idx``, the indices
    of the surviving rays in the launched bundle."""
    src, tran, surf, anal, xp = api.sources, api.tran, api.surf, api.anal, api.xp
    ro, ao = zernike_orders(7)
    coeff = zernike_coeff(len(ro), rng_seed)
    seed(rng_seed)
    rays = src.subannulus(220., 220.6, 100. / 220., n, zhat=-1.)
    idx = xp.arange(n)
    tran.transform(rays, 220.3, 0, -100., 0, 0, 0)
    surf.zernsurf(rays, coeff, 62.5, rorder=ro, aorder=ao, nr=1.)
    tran.reflect(rays)
    tran.transform(rays, 0, 0, 0, np.pi, 0, 0)
    surf.flat(rays, nr=1.)
    tran.transform(rays, -220.3, 0, -8600., 0, 0, 0)
    surf.wolterprimary(rays, 220., 8400.)
    tran.reflect(rays)
    ind = xp.logical_and(xp.logical_and(rays[3] > 8426., rays[3] < 8526.), xp.abs(rays[2]) < 50.)
    rays = tran.vignette(rays, ind=ind)
    idx = idx[ind]
    surf.woltersecondary(rays, 220., 8400.)
    tran.reflect(rays)
    ind = (rays[4] ** 2 + rays[5] ** 2 + rays[6] ** 2) > .1
    rays = tran.vignette(rays)
    idx = idx[ind]
    surf.flat(rays)
    return dict(rays=rays, idx=idx, hpd=anal.hpd(rays), rms=anal.rmsCentroid(rays))


# =============================================================================== config 4
def arcus_geometry(M=72):
    """Outermost SPO module row of the Arcus layout (examples/arcus/cat.py:59-132: module radii, widths and
    angles; the reflectivity / efficiency tables are private data, so weights are geometric area only)."""
    rin, rout, span, ang_deg = 755.807, 811.607, 82.053, 3.597
    R = np.arange(rin, rout, .775)[:M]
    tg = .25 * np.arctan((R + .775 / 2) / 12e3)
    L = .775 / np.tan(tg)
    focVec = np.sqrt(12e3 ** 2 - R ** 2)
    spanv = 2 * np.arcsin(span / 2 / R)
    area = ((R + .605) ** 2 - R ** 2) * spanv / 2 / 100.
    gap, lgrat, inc = 50., 95., 1.5 * np.pi / 180
    H = focVec[-1] - (L.max() + gap + 95.)                  # plane of the outermost grating above the focus
    outerrad = 798.895210199 + 2.                           # sector.py:40
    return SimpleNamespace(R=R, L=L, focVec=focVec, spanv=spanv, area=area, ang=ang_deg * np.pi / 180, H=H,
                           outerrad=outerrad, hubdist=math.sqrt(outerrad ** 2 + H ** 2),
                           angle=math.atan(outerrad / H), inc=inc, lgrat=lgrat, blazeYaw=0.022509613654884453,
                           dpermm_num=160.)


def traceSPO(api, g, N, offX=0., offY=0.):
    """examples/arcus/cat.py:203-288: shell by shell; positions and directions are collected into the master
    arrays (rows 1-6: opd and the normals stay zero)."""
    src, tran, surf, xp = api.sources, api.tran, api.surf, api.xp
    parts = []
    for i in range(len(g.R)):
        rays = src.subannulus(g.R[i], g.R[i] + .605, g.spanv[i], N, zhat=-1.)
        tran.transform(rays, 0, 0, 0, 0, 0, g.ang)
        surf.spoPrimary(rays, g.R[i], g.focVec[i])
        rays = [rays[0], rays[1], rays[2], rays[3], rays[4] + offX, rays[5] + offY,
                -xp.sqrt(rays[6] ** 2 - offX ** 2 - offY ** 2), rays[7], rays[8], rays[9]]
        tran.reflect(rays)
        surf.spoSecondary(rays, g.R[i], g.focVec[i])
        tran.reflect(rays)
        tran.transform(rays, 0, 0, -g.focVec[i], 0, 0, 0)
        parts.append(rays)
    zero = xp.repeat(0., N * len(g.R))
    cat = [xp.concatenate([p[t] for p in parts]) for t in range(1, 7)]
    return [xp.copy(zero)] + cat + [xp.copy(zero), xp.copy(zero), xp.copy(zero)]


def gratArray(api, rays, g, order, wave, weights=None, offX=0., max_gratings=2000):
    """examples/arcus/sector.py:636-757: the fanned CAT-grating array.  Every op in the loop is masked
    (``ind=``); the loop runs until every ray has met a grating.  Returns (focusY offset, gratings visited)."""
    tran, surf, xp = api.tran, api.surf, api.xp
    outerrad, hubdist, angle, inc, l = g.outerrad, g.hubdist, g.angle, g.inc, g.lgrat
    tran.transform(rays, outerrad, 0, 0, 0, 0, 0)
    tran.transform(rays, 0, 0, 0, 0, 0, -np.pi / 2)
    tran.transform(rays, 0, 0, 0, -np.pi / 2 - angle + inc, 0, 0)
    tran.transform(rays, 0, 0, 0, 0, 0, g.blazeYaw)
    tran.transform(rays, 0, hubdist, 0, 0, 0, 0)
    indg = xp.abs(xp.arcsin(rays[6])) > .001
    surf.flat(rays, ind=indg)
    rho = -xp.sqrt(rays[1] ** 2 + rays[2] ** 2) * xp.sign(rays[2])
    ind = xp.logical_and(rho > hubdist, rho < l + hubdist)
    ind2 = xp.copy(ind)
    ang = l * np.sin(inc - offX) / hubdist * .95
    i = 0
    prev = xp.copy(ind)
    num = rays[1].shape[0]
    while xp.count(prev) < num:
        i = i + 1
        if i > max_gratings:
            raise RuntimeError("gratArray: rays left after %d gratings (they never meet the array)" % max_gratings)
        if xp.count(ind2) > 0:
            tran.reflect(rays, ind=ind2)
            tran.radgrat(rays, g.dpermm_num / hubdist, order, wave, ind=ind2)
        tran.transform(rays, 0, 0, 0, ang, 0, 0)
        indg = xp.abs(xp.arcsin(rays[6])) > .001
        indg = xp.logical_and(xp.invert(prev), indg)
        surf.flat(rays, ind=indg)
        rho = -xp.sqrt(rays[1] ** 2 + rays[2] ** 2) * xp.sign(rays[2])
        ind = xp.logical_and(rho > hubdist, rho < l + hubdist)
        ind2 = xp.logical_and(xp.invert(prev), ind)
        prev = xp.logical_or(prev, ind)
    tran.reflect(rays, ind=ind2)
    tran.radgrat(rays, g.dpermm_num / hubdist, order, wave, ind=ind2)
    tran.transform(rays, 0, 0, 0, -ang * i, 0, 0)
    tran.transform(rays, 0, -hubdist, 0, 0, 0, 0)
    tran.transform(rays, 0, 0, 0, 0, 0, -g.blazeYaw)
    tran.transform(rays, 0, 0, 0, np.pi / 2 + angle - inc, 0, 0)
    tran.transform(rays, 0, 0, 0, 0, 0, np.pi / 2)
    tran.transform(rays, -outerrad, 0, 0, 0, 0, 0)
    surf.flat(rays)
    return surf.focusY(rays, weights=weights), i


def config4(api, n_per_shell=1000, M=72, order=-3, wave=2.4, rng_seed=0, offX=0., offY=0.):
    """Arcus: one SPO module row (M shells) -> fanned radial-grating array -> line focus
    (examples/arcus/cat.py:59-288, sector.py:253-389 traceArcus, :636-757 gratArray; SURVEY.md 3.4 / 8d).
    ``wave``: scalar [nm] -> radgrat; the string 'uniform' -> a per-ray wavelength array drawn from
    uniform(3.6, 7.2) -> radgratW.  Analysis as sector.py:372-389: drop |y - <y>| >= 10, weighted centroid."""
    tran, surf, anal, xp = api.tran, api.surf, api.anal, api.xp
    g = arcus_geometry(M)
    N = int(n_per_shell)
    seed(rng_seed)
    rays = traceSPO(api, g, N, offX, offY)
    weights = xp.concatenate([xp.repeat(a / N, N) for a in g.area])
    if isinstance(wave, str):
        wave = xp.uniform(3.6, 7.2, N * M)
    # to the plane of the outermost grating (cat.py:189-191)
    tran.transform(rays, 0, 0, g.H, 0, 0, 0)
    surf.flat(rays)
    dz, ngrat = gratArray(api, rays, g, order, wave, weights=weights, offX=offX)
    ind = xp.abs(rays[2] - anal.centroid(rays)[1]) < 10.
    surv = tran.vignette(rays, ind=ind)
    w = weights[ind]
    cx, cy = anal.centroid(surv, weights=w)
    return dict(rays=rays, surv=surv, kept=int(surv[1].shape[0]), dz=dz, gratings=ngrat, cx=cx, cy=cy,
                rmsY=anal.rmsY(surv, weights=w), hpdY=anal.hpdY(surv, weights=w))


# =============================================================================== config 5
def nested_geometry(nshell=260, L=200., nodegap=50.):
    """Nested Wolter-I assembly on a spherical principal surface: node radii r in [200,1500], z = sqrt(1e4^2 - r^2)
    (examples/axro/axialHeights.py:222-240, SMARTX.py:179-180; SURVEY.md 8d)."""
    r = np.linspace(200., 1500., int(nshell))
    z = np.sqrt(1.e4 ** 2 - r ** 2)
    return SimpleNamespace(r=r, z=z, L=L, nodegap=nodegap)


def config5(api, n_per_shell=1000, nshell=260, offaxis=0., rng_seed=0):
    """``tracePerfectXRS`` (examples/axro/axialHeights.py:215-322) with the Wolter-I prescription per shell that
    SURVEY.md 8d names: per shell annulus -> primary -> field kick -> reflect -> secondary -> reflect ->
    vignette(z range) -> exit aperture -> vignette(rho > back of the previous shell) -> focal plane; area
    weights follow the rays through both vignettes; weighted hpd / rms / centroid of the accumulated bundle."""
    src, tran, surf, anal, conic, xp = api.sources, api.tran, api.surf, api.anal, api.conic, api.xp
    g = nested_geometry(nshell)
    L, nodegap, N = g.L, g.nodegap, int(n_per_shell)
    seed(rng_seed)
    previousrho = 0.
    mparts, wparts = [], []
    for r, z in zip(g.r, g.z):
        r, z = float(r), float(z)
        a0 = float(conic.primrad(z + nodegap / 2., r, z))
        a1 = float(conic.primrad(z + nodegap / 2. + L, r, z))
        rays = src.annulus(a0, a1, N)
        tran.transform(rays, 0, 0, -z, 0, 0, 0)
        weights = xp.repeat((a1 ** 2 - a0 ** 2) * np.pi / 100. / N, N)
        surf.wolterprimary(rays, r, z)
        rays[4] = rays[4] + np.sin(offaxis)
        rays[6] = -xp.sqrt(1. - rays[4] ** 2)
        tran.reflect(rays)
        surf.woltersecondary(rays, r, z)
        tran.reflect(rays)
        ind = xp.logical_and(rays[3] > z - nodegap / 2. - L, rays[3] < z - nodegap / 2.)
        rays = tran.vignette(rays, ind=ind)
        weights = weights[ind]
        tran.transform(rays, 0, 0, z - nodegap / 2 - L, 0, 0, 0)
        surf.flat(rays)
        rho = xp.sqrt(rays[1] ** 2 + rays[2] ** 2)
        ind = rho > previousrho
        rays = tran.vignette(rays, ind=ind)
        weights = weights[ind]
        previousrho = float(conic.secrad(z - nodegap / 2 - L, r, z)) + .4
        tran.transform(rays, 0, 0, -z + nodegap / 2 + L, 0, 0, 0)
        surf.flat(rays)
        mparts.append(rays)
        wparts.append(weights)
    mrays = [xp.concatenate([p[t] for p in mparts]) for t in range(10)]
    mweights = xp.concatenate(wparts)
    cx, cy = anal.centroid(mrays, weights=mweights)
    return dict(rays=mrays, weights=mweights, kept=int(mrays[1].shape[0]),
                hpd=anal.hpd(mrays, weights=mweights), rms=anal.rmsCentroid(mrays, weights=mweights), cx=cx, cy=cy,
                area=float(mweights.sum()))


# =============================================================================== the same configurations, GPU-arranged
# Same arithmetic, same order per ray; what changes is the packaging: whole chains are recorded into one fused
# program (``with pxf.fused(rays)``), mask expressions become in-kernel predicates followed by ONE order-preserving
# compaction, the Python loops over shells become ONE segmented launch, and the grating fan becomes a per-ray loop
# inside the kernel.  ``rng='numpy'`` draws the uniforms exactly as the scripts above do (parity tests);
# ``rng='philox'`` draws them on the device (throughput at the BASELINE sizes, where host MT19937 would dominate).
def _pxf():
    import pyxfocus_b200 as pxf
    return pxf


def _source_kw(rng, rng_seed, device, first=0):
    if rng == "numpy":
        return dict(device=device)
    return dict(rng="philox", seed=rng_seed, first=first, device=device)


def config1_fast(n=100_000, rng="numpy", rng_seed=0, device=None, sources=None):
    pxf = _pxf()
    src = sources or pxf.sources
    tran, surf, anal = pxf.transformations, pxf.surfaces, pxf.analyses
    seed(rng_seed)
    rays = src.subannulus(220., 220.6, 2 * np.pi, n, zhat=-1., **_source_kw(rng, rng_seed, device))
    with pxf.fused(rays):
        tran.transform(rays, 0, 0, -8400., 0, 0, 0)
        surf.wolterprimary(rays, 220., 8400.)
        tran.reflect(rays)
        surf.woltersecondary(rays, 220., 8400.)
        tran.reflect(rays)
        surf.flat(rays)
    return dict(rays=rays, hpd=anal.hpd(rays), rms=anal.rmsCentroid(rays))


def config2_point_fast(n, offaxis, aperture, rng="numpy", rng_seed=0, device=None,
                       R0=WS["R0"], Z0=WS["Z0"], psi=WS["psi"], az=WS["az"], sources=None):
    pxf = _pxf()
    src = sources or pxf.sources
    tran, surf, anal = pxf.transformations, pxf.surfaces, pxf.analyses
    a0, a1 = aperture
    seed(rng_seed)
    rays = src.subannulus(a0, a1, az / R0, n, **_source_kw(rng, rng_seed, device))
    with pxf.fused(rays):
        tran.transform(rays, 0, 0, -Z0, 0, 0, 0)
        surf.wsPrimary(rays, R0, Z0, psi)
        pxf.program.recorder_for(rays).kick(np.sin(offaxis), 0., -1.)      # the two row assignments of the script
        tran.reflect(rays)
        surf.wsSecondary(rays, R0, Z0, psi)
        tran.reflect(rays)
        surf.flat(rays)
    # both scans from ONE pass over the bundle: moving the frame by d2 only shifts the sums
    s9 = anal.imageplane_sums(rays, at_z0=True)
    d2 = anal.findimageplane(rays, 20., 100, sums=s9)
    d3 = anal.findimageplane(rays, 1., 100, sums=s9, moved=d2)
    with pxf.fused(rays):
        tran.transform(rays, 0, 0, d2, 0, 0, 0)
        tran.transform(rays, 0, 0, d3, 0, 0, 0)
        surf.flat(rays)
    hpd_scan, rms_scan = anal.hpd(rays), anal.rmsCentroid(rays)
    f = surf.focusI(rays)
    return dict(rays=rays, f=f, d2=d2, d3=d3, hpd_scan=hpd_scan, rms_scan=rms_scan, hpd=anal.hpd(rays),
                rms=anal.rmsCentroid(rays))


def config2_fast(n=10_000_000, arcmin=None, aperture=None, rng="numpy", rng_seed=0, device=None):
    arcmin = np.linspace(0., 30., 31) if arcmin is None else arcmin
    aperture = ws_aperture(product_api(device)) if aperture is None else aperture
    return [config2_point_fast(n, a / 60. * np.pi / 180., aperture, rng, rng_seed, device) for a in arcmin]


def config2_sweep_fast(n=10_000_000, arcmin=None, aperture=None, rng="numpy", rng_seed=0, device=None,
                       R0=WS["R0"], Z0=WS["Z0"], psi=WS["psi"], az=WS["az"], sources=None):
    """``config2_fast`` as ONE bundle: the source is drawn once and replicated per field point (config2_fast reuses
    the same draws at every point), one segmented launch traces all points with a per-segment kick, and every
    analysis runs per segment (``segments=``) in a number of launches that does not depend on the point count.
    Returns the same list of per-point dicts; ``rays`` is each point's view of the joint bundle."""
    pxf = _pxf()
    from pyxfocus_b200._call import bundle_alloc, bundle_split
    anal = pxf.analyses
    arcmin = np.linspace(0., 30., 31) if arcmin is None else np.asarray(arcmin, dtype=np.float64)
    aperture = ws_aperture(product_api(device)) if aperture is None else aperture
    a0, a1 = aperture
    K = len(arcmin)
    seed(rng_seed)
    src = (sources or pxf.sources).subannulus(a0, a1, az / R0, n, **_source_kw(rng, rng_seed, device))
    dev = src[1].device
    rays = bundle_alloc(K * n, dev)
    for r, s_ in zip(rays, src):
        r.view(K, n).copy_(s_.unsqueeze(0).expand(K, n))
    del src
    segs = pxf.Segments([n] * K, device=dev)
    alpha = pxf.conicsolve.woltparam(R0, Z0)[0]
    # the recorded form of config2_point_fast's chain (transform arguments negated, as transformations.transform does)
    progs = [pxf.Program().transform(-0., -0., Z0, -0., -0., -0.).wsprimary(alpha, Z0, psi)
             .kick(np.sin(a / 60. * np.pi / 180.), 0., -1.).reflect().wssecondary(alpha, Z0, psi).reflect().flat()
             for a in arcmin]
    pxf.SegmentedProgram(progs, segs.sizes(), device=dev).run(rays)
    s9 = anal.imageplane_sums(rays, at_z0=True, segments=segs)
    d2 = anal.findimageplane(rays, 20., 100, sums=s9, segments=segs)
    d3 = anal.findimageplane(rays, 1., 100, sums=s9, moved=d2, segments=segs)
    pxf.SegmentedProgram([pxf.Program().transform(-0., -0., -d2[k], -0., -0., -0.)
                          .transform(-0., -0., -d3[k], -0., -0., -0.).flat() for k in range(K)],
                         segs.sizes(), device=dev).run(rays)
    hpd_scan, rms_scan = anal.hpd(rays, segments=segs), anal.rmsCentroid(rays, segments=segs)
    f = pxf.surfaces.focusI(rays, segments=segs)
    hpd, rms = anal.hpd(rays, segments=segs), anal.rmsCentroid(rays, segments=segs)
    views = bundle_split(rays, [n] * K)
    return [dict(rays=views[k], f=float(f[k]), d2=float(d2[k]), d3=float(d3[k]), hpd_scan=float(hpd_scan[k]),
                 rms_scan=float(rms_scan[k]), hpd=float(hpd[k]), rms=float(rms[k])) for k in range(K)]


def config3_fast(n=100_000_000, rng="numpy", rng_seed=0, device=None, want_idx=True, sources=None, coeff=None):
    """``coeff``: the 36 Zernike coefficients (default: ``zernike_coeff(36, rng_seed)``, as ``config3``)."""
    pxf = _pxf()
    src = sources or pxf.sources
    tran, surf, anal = pxf.transformations, pxf.surfaces, pxf.analyses
    ro, ao = zernike_orders(7)
    coeff = zernike_coeff(len(ro), rng_seed) if coeff is None else coeff
    seed(rng_seed)
    rays = src.subannulus(220., 220.6, 100. / 220., n, zhat=-1., **_source_kw(rng, rng_seed, device))
    with pxf.fused(rays):
        prog = pxf.program.recorder_for(rays)
        tran.transform(rays, 220.3, 0, -100., 0, 0, 0)
        surf.zernsurf(rays, coeff, 62.5, rorder=ro, aorder=ao, nr=1.)
        tran.reflect(rays)
        tran.transform(rays, 0, 0, 0, np.pi, 0, 0)
        surf.flat(rays, nr=1.)
        tran.transform(rays, -220.3, 0, -8600., 0, 0, 0)
        surf.wolterprimary(rays, 220., 8400.)
        tran.reflect(rays)
        prog.vignette_box(3, 8426., 8526.).vignette_abs(2, 50.)
        surf.woltersecondary(rays, 220., 8400.)
        tran.reflect(rays)
        prog.vignette_mag()
        surf.flat(rays)
    alive = pxf.program.last_alive(rays)
    surv = tran.compact(rays, alive)
    out = dict(rays=surv, hpd=anal.hpd(surv), rms=anal.rmsCentroid(surv))
    if want_idx:
        out["idx"] = tran.surviving_indices(alive)
    return out


def config3_program(coeff):
    """The 14-op program ``config3_fast`` records, written out (transform arguments negated, as
    ``transformations.transform`` passes them on): the same ops with the same scalars, so the same bits."""
    pxf = _pxf()
    ro, ao = zernike_orders(7)
    return (pxf.Program().transform(-220.3, 0., 100., 0., 0., 0.).zernsurf(coeff, ro, ao, 62.5, 1.).reflect()
            .transform(0., 0., 0., -np.pi, 0., 0.).flatopd(1.).transform(220.3, 0., 8600., 0., 0., 0.)
            .wolterprimary(220., 8400., 1.).reflect().vignette_box(3, 8426., 8526.).vignette_abs(2, 50.)
            .woltersecondary(220., 8400., 1.).reflect().vignette_mag().flat())


def config3_tolerance_fast(n, coeffs, rng="numpy", rng_seed=0, device=None, sources=None):
    """A figure-error Monte Carlo of config 3 as ONE bundle: one realisation per coefficient vector in ``coeffs``
    (e.g. ``zernike_coeff(36, seed_k)``).  The source is drawn once and replicated per realisation (the loop of
    ``config3_fast(coeff=c_k)`` draws the same rays every time), one segmented launch traces every realisation
    through its own Zernike surface, one compaction drops the vignetted rays, and ``hpd`` / ``rmsCentroid`` run per
    segment.  Returns one dict per realisation with the keys of ``config3_fast``: ``rays`` is the realisation's view
    of the compacted bundle, ``idx`` the surviving indices within its own n rays."""
    pxf = _pxf()
    from pyxfocus_b200._call import bundle_alloc, bundle_split
    tran, anal = pxf.transformations, pxf.analyses
    K = len(coeffs)
    seed(rng_seed)
    src = (sources or pxf.sources).subannulus(220., 220.6, 100. / 220., n, zhat=-1.,
                                               **_source_kw(rng, rng_seed, device))
    dev = src[1].device
    rays = bundle_alloc(K * n, dev)
    for r, s_ in zip(rays, src):
        r.view(K, n).copy_(s_.unsqueeze(0).expand(K, n))
    del src
    segs = pxf.Segments([n] * K, device=dev)
    alive = pxf.SegmentedProgram([config3_program(c) for c in coeffs], segs.sizes(), device=dev).run(rays)
    after = segs.after(alive)
    surv = tran.compact(rays, alive)
    idx = tran.surviving_indices(alive)
    hpd, rms = anal.hpd(surv, segments=after), anal.rmsCentroid(surv, segments=after)
    kept = after.sizes()
    views = bundle_split(surv, kept)
    return [dict(rays=views[k], hpd=float(hpd[k]), rms=float(rms[k]),
                 idx=idx[after.start[k]:after.start[k + 1]] - k * n) for k in range(K)]


# ------------------------------------------------------------------ Legendre-Legendre Wolter-I pair
# The geometry of the reference fixture for the LL shells (tests/golden/make_golden.py, singlePassAlignment.py style):
# a 220 mm Wolter-I pair at 8400 mm, 0.25 rad of azimuth, the primary's figure on 8400..8500 mm, the secondary's on
# 8300..8400 mm.
def ll_orders(nmax=5):
    """(axial, az) of every Legendre-Legendre term up to order ``nmax`` in both directions: (nmax+1)**2 terms."""
    ax, az = np.meshgrid(np.arange(nmax + 1), np.arange(nmax + 1), indexing="ij")
    return ax.ravel(), az.ravel()


def ll_coeff(nterms=36, rng_seed=0, sigma=2.e-4):
    """Random LL figure coefficients [mm] (one realisation of a figure error)."""
    return np.random.default_rng(rng_seed).normal(0., sigma, nterms)


def llpair_program(coeff_p, coeff_s, axial, az):
    """The LL pair ``llpair_fast`` records, written out (transform arguments negated, as ``transformations.transform``
    passes them on): the same ops with the same scalars, so the same bits."""
    pxf = _pxf()
    return (pxf.Program().transform(-0., -0., 8400., -0., -0., -0.)
            .wolterprimll(220., 8400., 8500., 8400., .25, coeff_p, axial, az).reflect()
            .woltersecll(220., 8400., 1., 8400., 8300., .25, coeff_s, axial, az).reflect().flat())


def llpair_fast(n, coeff_p, coeff_s, axial, az, rng="numpy", rng_seed=0, device=None, sources=None):
    """A Wolter-I pair whose primary and secondary carry Legendre-Legendre figure terms, traced to the focal plane
    inside ``fused``: one launch for orders <= 7."""
    pxf = _pxf()
    src = sources or pxf.sources
    tran, surf, anal = pxf.transformations, pxf.surfaces, pxf.analyses
    seed(rng_seed)
    rays = src.subannulus(220., 220.6, .25, n, zhat=-1., **_source_kw(rng, rng_seed, device))
    with pxf.fused(rays):
        tran.transform(rays, 0, 0, -8400., 0, 0, 0)
        surf.primaryLL(rays, 220., 8400., 8500., 8400., .25, coeff_p, axial, az)
        tran.reflect(rays)
        surf.secondaryLL(rays, 220., 8400., 1., 8400., 8300., .25, coeff_s, axial, az)
        tran.reflect(rays)
        surf.flat(rays)
    return dict(rays=rays, hpd=anal.hpd(rays), rms=anal.rmsCentroid(rays))


def ll_tolerance_fast(n, realisations, axial, az, rng="numpy", rng_seed=0, device=None, sources=None):
    """A figure-error Monte Carlo of the LL pair as ONE bundle: one realisation per (coeff_p, coeff_s) pair in
    ``realisations``.  The source is drawn once and replicated per realisation (the loop of ``llpair_fast`` draws the
    same rays every time), one segmented launch traces every realisation through its own pair of figures, and
    ``hpd`` / ``rmsCentroid`` run per segment.  Returns one dict per realisation with the keys of ``llpair_fast``:
    ``rays`` is the realisation's view of the joint bundle."""
    pxf = _pxf()
    from pyxfocus_b200._call import bundle_alloc, bundle_split
    anal = pxf.analyses
    K = len(realisations)
    seed(rng_seed)
    src = (sources or pxf.sources).subannulus(220., 220.6, .25, n, zhat=-1., **_source_kw(rng, rng_seed, device))
    dev = src[1].device
    rays = bundle_alloc(K * n, dev)
    for r, s_ in zip(rays, src):
        r.view(K, n).copy_(s_.unsqueeze(0).expand(K, n))
    del src
    segs = pxf.Segments([n] * K, device=dev)
    pxf.SegmentedProgram([llpair_program(cp, cs, axial, az) for cp, cs in realisations], segs.sizes(),
                         device=dev).run(rays)
    hpd, rms = anal.hpd(rays, segments=segs), anal.rmsCentroid(rays, segments=segs)
    views = bundle_split(rays, [n] * K)
    return [dict(rays=views[k], hpd=float(hpd[k]), rms=float(rms[k])) for k in range(K)]


def _arcus_spo_fast(pxf, src, g, N, M, rng, rng_seed, dev, offX, offY):
    """The M SPO shells of ``config4_fast`` in one segmented launch, traced to the plane of the outermost grating.
    Returns the bundle and the per-ray area weights."""
    import torch
    from pyxfocus_b200._call import bundle_alloc, bundle_split
    per = [N] * M
    seed(rng_seed)
    rays = bundle_alloc(N * M, dev, zero=True)
    if rng == "numpy":
        for i, seg in enumerate(bundle_split(rays, per)):
            src.subannulus(g.R[i], g.R[i] + .605, g.spanv[i], N, zhat=-1., out=seg)
    else:
        pxf.sources.segments("subannulus", [(g.R[i], g.R[i] + .605, g.spanv[i], -1.) for i in range(M)], per,
                             seed=rng_seed, out=rays)
    weights = torch.cat([torch.full((N,), a / N, dtype=torch.float64, device=dev) for a in g.area])
    # one launch for the M shells: SPO pair, to the focus frame, to the plane of the outermost grating
    # (Program.* take the scalars as the Fortran routine sees them: transform arguments negated, transformations.py:29)
    shells = [pxf.Program().transform(0, 0, 0, 0, 0, -g.ang)
              .spocone(g.R[i], .25 * np.arctan((g.R[i] + .605 / 2) / g.focVec[i])).kickn(offX, offY).reflect()
              .spocone(g.R[i], .75 * np.arctan((g.R[i] + .605 / 2) / g.focVec[i])).reflect()
              .transform(0, 0, g.focVec[i], 0, 0, 0).transform(0, 0, -g.H, 0, 0, 0).flat() for i in range(M)]
    pxf.SegmentedProgram(shells, per, device=dev).run(rays)
    return rays, weights


def _uniform_wave(num, rng, rng_seed, dev):
    """config4's ``wave='uniform'``: per-ray wavelengths [nm] from uniform(3.6, 7.2)."""
    import torch
    if rng == "numpy":
        return torch.as_tensor(np.random.uniform(3.6, 7.2, size=num), device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(int(rng_seed))
    return 3.6 + 3.6 * torch.rand(num, dtype=torch.float64, device=dev, generator=gen)


def config4_fast(n_per_shell=1000, M=72, order=-3, wave=2.4, rng="numpy", rng_seed=0, device=None, offX=0., offY=0.,
                 sources=None):
    pxf = _pxf()
    src = sources or pxf.sources
    tran, surf, anal = pxf.transformations, pxf.surfaces, pxf.analyses
    g = arcus_geometry(M)
    N = int(n_per_shell)
    dev = pxf.sources._device(device)
    rays, weights = _arcus_spo_fast(pxf, src, g, N, M, rng, rng_seed, dev, offX, offY)
    if isinstance(wave, str):
        wave = _uniform_wave(N * M, rng, rng_seed, dev)
    # the grating fan: frame changes + per-ray loop over the gratings (sector.py:650-707)
    outerrad, hubdist, angle, inc, l = g.outerrad, g.hubdist, g.angle, g.inc, g.lgrat
    ang = l * np.sin(inc - offX) / hubdist * .95
    aux = pxf.FanAux(N * M, dev)
    (pxf.Program().transform(-outerrad, 0, 0, 0, 0, 0).transform(0, 0, 0, 0, 0, np.pi / 2)
     .transform(0, 0, 0, -(-np.pi / 2 - angle + inc), 0, 0).transform(0, 0, 0, 0, 0, -g.blazeYaw)
     .transform(0, -hubdist, 0, 0, 0, 0)
     .gratfan(ang, hubdist, l, g.dpermm_num / hubdist, order, wave)).run(rays, aux=aux)
    i = aux.gratings()                                    # the one host round trip of the loop
    (pxf.Program().rotx_remaining(ang, i).transform(0, 0, 0, ang * i, 0, 0).transform(0, hubdist, 0, 0, 0, 0)
     .transform(0, 0, 0, 0, 0, g.blazeYaw).transform(0, 0, 0, -(np.pi / 2 + angle - inc), 0, 0)
     .transform(0, 0, 0, 0, 0, -np.pi / 2).transform(outerrad, 0, 0, 0, 0, 0).flat()).run(rays, aux=aux)
    dz = surf.focusY(rays, weights=weights)
    alive = pxf.Program().vignette_abs(2, 10., anal.centroid(rays)[1]).run(rays)
    surv, (w,) = tran.compact(rays, alive, extra=[weights])
    cx, cy = anal.centroid(surv, weights=w)
    return dict(rays=rays, surv=surv, kept=int(surv[1].shape[0]), dz=dz, gratings=i, cx=cx, cy=cy,
                rmsY=anal.rmsY(surv, weights=w), hpdY=anal.hpdY(surv, weights=w))


def config4_spectrum_fast(n_per_shell=1000, M=72, order=-3, rng="numpy", rng_seed=0, device=None, offX=0., offY=0.,
                          sources=None, fuse=True):
    """The SPO shells of ``config4_fast`` followed by a straight grating stage driven by a sampled spectrum: per-ray
    wavelengths drawn as config4's ``wave='uniform'``, a radial grating (radgratW) in the plane of the outermost
    grating with the CAT period (``dpermm_num`` = 160 nm) at the outermost module radius, back down to the focal
    plane and ``flat``.  Inside ``fused`` the grating stage is one launch; ``fuse=False`` runs the same calls one by
    one.  Returns the rays, the wavelengths, the best line focus in y and the weighted y RMS there."""
    pxf = _pxf()
    src = sources or pxf.sources
    tran, surf, anal = pxf.transformations, pxf.surfaces, pxf.analyses
    g = arcus_geometry(M)
    N = int(n_per_shell)
    dev = pxf.sources._device(device)
    rays, weights = _arcus_spo_fast(pxf, src, g, N, M, rng, rng_seed, dev, offX, offY)
    wave = _uniform_wave(N * M, rng, rng_seed, dev)

    def grating_stage():
        tran.radgrat(rays, g.dpermm_num / g.outerrad, order, wave)
        tran.transform(rays, 0, 0, -g.H, 0, 0, 0)
        surf.flat(rays)
    if fuse:
        with pxf.fused(rays):
            grating_stage()
    else:
        grating_stage()
    dz = surf.focusY(rays, weights=weights)
    return dict(rays=rays, wave=wave, dz=dz, rmsY=anal.rmsY(rays, weights=weights))


def config5_fast(n_per_shell=1000, nshell=260, offaxis=0., rng="numpy", rng_seed=0, device=None, first=0,
                 sources=None, analyses=None):
    """``analyses``: module for the closing weighted statistics -- ``pxf.dist`` when the bundle is one shard of a
    multi-GPU run (every rank traces its own rays of every shell, ``first`` = its offset in the Philox stream; only
    the analyses communicate)."""
    pxf = _pxf()
    src = sources or pxf.sources
    import torch
    from pyxfocus_b200._call import bundle_alloc, bundle_split
    tran, anal, conic = pxf.transformations, pxf.analyses, pxf.conicsolve
    g = nested_geometry(nshell)
    L, nodegap, N = g.L, g.nodegap, int(n_per_shell)
    dev = pxf.sources._device(device)
    per = [N] * len(g.r)
    aper, progs, wts = [], [], []
    previousrho = 0.
    for r, z in zip(g.r, g.z):
        r, z = float(r), float(z)
        a0 = float(conic.primrad(z + nodegap / 2., r, z))
        a1 = float(conic.primrad(z + nodegap / 2. + L, r, z))
        aper.append((a0, a1, 0., -1.))
        wts.append((a1 ** 2 - a0 ** 2) * np.pi / 100. / N)
        progs.append(pxf.Program().transform(0, 0, z, 0, 0, 0).wolterprimary(r, z, 1.).kick(np.sin(offaxis), 0., -1.)
                     .reflect().woltersecondary(r, z, 1.).reflect()
                     .vignette_box(3, z - nodegap / 2. - L, z - nodegap / 2.)
                     .transform(0, 0, -(z - nodegap / 2 - L), 0, 0, 0).flat().vignette_rhogt(previousrho)
                     .transform(0, 0, -(-z + nodegap / 2 + L), 0, 0, 0).flat())
        previousrho = float(conic.secrad(z - nodegap / 2 - L, r, z)) + .4
    seed(rng_seed)
    rays = bundle_alloc(N * len(per), dev, zero=True)
    if rng == "numpy":
        for k, sgm in enumerate(bundle_split(rays, per)):
            src.annulus(aper[k][0], aper[k][1], N, out=sgm)
    else:
        pxf.sources.segments("annulus", aper, per, seed=rng_seed, first=first, out=rays)
    weights = torch.repeat_interleave(torch.as_tensor(np.array(wts), device=dev), N)
    alive = pxf.SegmentedProgram(progs, per, device=dev).run(rays)
    mrays, (mweights,) = tran.compact(rays, alive, extra=[weights])
    if analyses is not None:
        anal = analyses
    cx, cy = anal.centroid(mrays, weights=mweights)
    return dict(rays=mrays, weights=mweights, kept=int(mrays[1].shape[0]),
                hpd=anal.hpd(mrays, weights=mweights), rms=anal.rmsCentroid(mrays, weights=mweights), cx=cx, cy=cy,
                area=float(mweights.sum()))


# =============================================================================== kernel pre-compilation
def baseline_programs():
    """The op lists the GPU-arranged configurations above hand to the library that are not among its built-in chains
    -- only the opcode sequence (and predicate rows) matters for the kernel, not the scalars."""
    import pyxfocus_b200 as pxf
    P = pxf.Program
    ro, ao = zernike_orders(7)
    progs = [
        # config 2: W-S pair to the nominal focal plane; move the plane twice and trace to it
        (P().transform(0, 0, 1, 0, 0, 0).wsprimary(5e-3, 1e4, 1.).kick(0, 0, -1).reflect().wssecondary(5e-3, 1e4, 1.).reflect().flat(), False),
        (P().transform(0, 0, 1, 0, 0, 0).transform(0, 0, 1, 0, 0, 0).flat(), False),
        # config 3: the 14-op program with the Zernike surface and three predicates
        (P().transform(1, 0, 1, 0, 0, 0).zernsurf(zernike_coeff(len(ro)), ro, ao, 62.5, 1.).reflect().transform(0, 0, 0, 1, 0, 0)
         .flatopd(1.).transform(1, 0, 1, 0, 0, 0).wolterprimary(220., 8400., 1.).reflect().vignette_box(3, 0, 1).vignette_abs(2, 1.)
         .woltersecondary(220., 8400., 1.).reflect().vignette_mag().flat(), False),
        # config 3 as a figure-error Monte Carlo: one Zernike surface per segment (segmented)
        (config3_program(zernike_coeff(len(ro))), True),
        # the Legendre-Legendre Wolter-I pair (36 terms per mirror), single and as a figure-error Monte Carlo
        (llpair_program(ll_coeff(36), ll_coeff(36, 1), *ll_orders(5)), False),
        (llpair_program(ll_coeff(36), ll_coeff(36, 1), *ll_orders(5)), True),
        # config 4: SPO shells (segmented), the grating fan, the way back, the outlier cut
        (P().transform(0, 0, 0, 0, 0, 1).spocone(700., .01).kickn(0, 0).reflect().spocone(700., .03).reflect()
         .transform(0, 0, 1, 0, 0, 0).transform(0, 0, 1, 0, 0, 0).flat(), True),
        (P().transform(1, 0, 0, 0, 0, 0).transform(0, 0, 0, 0, 0, 1).transform(0, 0, 0, 1, 0, 0).transform(0, 0, 0, 0, 0, 1)
         .transform(0, 1, 0, 0, 0, 0).gratfan(1e-4, 1e4, 95., .01, -1, 1.), False),
        (P().rotx_remaining(1e-4, 1).transform(0, 0, 0, 1, 0, 0).transform(0, 1, 0, 0, 0, 0).transform(0, 0, 0, 0, 0, 1)
         .transform(0, 0, 0, 1, 0, 0).transform(0, 0, 0, 0, 0, 1).transform(1, 0, 0, 0, 0, 0).flat(), False),
        (P().vignette_abs(2, 10., 1.), False),
        # config 5: one nested shell (segmented)
        (P().transform(0, 0, 1, 0, 0, 0).wolterprimary(220., 8400., 1.).kick(0, 0, -1).reflect().woltersecondary(220., 8400., 1.)
         .reflect().vignette_box(3, 0, 1).transform(0, 0, 1, 0, 0, 0).flat().vignette_rhogt(1.).transform(0, 0, 1, 0, 0, 0).flat(), True),
    ]
    return progs


def precompile():
    """Compile (NVRTC; no GPU needed) and cache the specialised kernels of ``baseline_programs``.  Returns
    (kernels available, programs): 0 kernels means NVRTC is unavailable and the interpreter will run instead."""
    have = 0
    progs = baseline_programs()
    for prog, segmented in progs:
        have += prog.precompile(segmented=segmented)
    return have, len(progs)
