"""Mirror of the hot-path part of the reference's ``surfaces.py`` on the device ray bundle:
``flat`` (surfaces.py:14-29), ``zernsurf`` (:31-47), ``conic`` (:104-113),
``wolterprimary`` (:219-227), ``wolterprimarynode`` (:229-236), ``woltersecondary``
(:238-243), ``woltersine`` (:265-270), ``wsPrimary`` (:331-347), ``wsSecondary`` (:367-383),
``spoCone/spoPrimary/spoSecondary`` (:403-441), ``focus/focusI`` (:502-519); and the
Legendre-Legendre shells ``primaryLL`` (:300-306), ``secondaryLL`` (:291-298),
``ellipsoidPrimary/Secondary(LL)`` (:443-500); and the rest of the file's surface wrappers:
``zernphase`` (:49-61), ``zernsurfrot`` (:63-80), ``sphere``/``tanSphere`` (:82-103), ``conicplus``
(:115-124), ``oapCollimate`` (:126-158), ``torus`` (:160-166), ``cyl`` (:168-180), ``cylconic``
(:182-186), ``paraxial``/``paraxialY`` (:188-206), ``legSurf`` (:208-217), the tangent-plane
placements ``wolterprimtan``/``woltersinetan``/``primaryLLtan`` (:245-263, :272-290, :308-329),
``wsPrimaryB``/``wsSecondaryB`` (:349-365, :385-401), ``focusX``/``focusY`` (:512-516).

Same names, argument order and results; ``ind=`` masks run as in-kernel predicates, and inside
``with program.fused(rays):`` unmasked calls are recorded into one fused kernel.
"""
import numpy as np
import torch

from . import conicsolve as con
from . import surfacesf as surf
from . import transformations as tran
from . import woltsurf as wolt
from . import zernsurf as zern
from .analyses import analyticImagePlane, analyticXPlane, analyticYPlane
from .program import (ARRAY_OPS, CONICPLUS_MAX_TERMS, LEGSURF_MAX_ORDER, LEGSURF_MAX_TERMS, LL_MAX_OPS, LL_MAX_ORDER,
                      OP, SURFACE_OPS, ZERN_MAX_ORDER, flush, recorder_for)


def flat(rays, ind=None, nr=None):
    """Trace rays to the XY plane.  As in the reference, ``ind`` takes precedence over ``nr``
    (the masked branch calls the non-OPD routine, surfaces.py:17-24)."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    if ind is not None:
        flush(rays)
        surf.flat(x, y, z, l, m, n, ux, uy, uz, mask=ind)
        return
    prog = recorder_for(rays)
    if nr is not None:
        if prog is not None:
            prog.flatopd(nr)
        else:
            surf.flatopd(x, y, z, l, m, n, ux, uy, uz, opd, nr)
    else:
        if prog is not None:
            prog.flat()
        else:
            surf.flat(x, y, z, l, m, n, ux, uy, uz)
    return


def zernsurf(rays, coeff, rad, rorder=None, aorder=None, nr=None):
    """Zernike sag surface, theta = arctan2(y,x).  ``rorder``/``aorder`` must be given: the
    reference's default comes from the un-vendored ``utilities.imaging.zernikemod.zmodes``
    (surfaces.py:10,36-37), whose ordering is not pinned anywhere in the reference tree."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    if rorder is None or aorder is None:
        raise NotImplementedError("pass rorder/aorder explicitly: the reference's default ordering lives in "
                                  "the third-party module utilities.imaging.zernikemod (not vendored)")
    prog = recorder_for(rays)
    if _zernsurf_recorder(prog, rorder):
        prog.zernsurf(coeff, rorder, aorder, rad, nr)       # radial orders <= 7: stays in the fused program
        return
    flush(rays)
    if nr is None:
        zern.tracezern(x, y, z, l, m, n, ux, uy, uz, coeff, np.array(rorder), np.array(aorder), rad)
    else:
        zern.tracezernopd(opd, x, y, z, l, m, n, ux, uy, uz, coeff, np.array(rorder), np.array(aorder), rad, nr)
    return


def conic(rays, R, K, nr=None):
    """Conic with radius of curvature R and conic constant K."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = recorder_for(rays)
    if nr is not None:
        if prog is not None:
            prog.conicopd(R, K, nr)
        else:
            surf.conicopd(opd, x, y, z, l, m, n, ux, uy, uz, R, K, nr)
    else:
        if prog is not None:
            prog.conic(R, K)
        else:
            surf.conic(x, y, z, l, m, n, ux, uy, uz, R, K)
    return


def wolterprimary(rays, r0, z0, psi=1., nr=None):
    """Wolter-I primary (paraboloid), no vignetting."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = recorder_for(rays)
    if nr is None:
        if prog is not None:
            prog.wolterprimary(r0, z0, psi)
        else:
            wolt.wolterprimary(x, y, z, l, m, n, ux, uy, uz, r0, z0, psi)
    else:
        if prog is not None:
            prog.wolterprimaryopd(r0, z0, psi, nr)
        else:
            wolt.wolterprimaryopd(opd, x, y, z, l, m, n, ux, uy, uz, r0, z0, psi, nr)
    return


def wolterprimarynode(rays, r0, z0, psi=1.):
    """Wolter node at the current origin, focus at (-r0,0,-z0)."""
    tran.transform(rays, -r0, 0, -z0, 0, 0, 0)
    wolterprimary(rays, r0, z0, psi)
    tran.itransform(rays, -r0, 0, -z0, 0, 0, 0)
    return


def woltersecondary(rays, r0, z0, psi=1.):
    """Wolter-I secondary (hyperboloid), no vignetting."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = recorder_for(rays)
    if prog is not None:
        prog.woltersecondary(r0, z0, psi)
    else:
        wolt.woltersecondary(x, y, z, l, m, n, ux, uy, uz, r0, z0, psi)
    return


def woltersine(rays, r0, z0, amp, freq):
    """Wolter-I primary with an axial sinusoid."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = recorder_for(rays)
    if prog is not None:
        prog.woltersine(r0, z0, amp, freq)
    else:
        wolt.woltersine(x, y, z, l, m, n, ux, uy, uz, r0, z0, amp, freq)
    return


def _ws(rays, which, r0, z0, psi, check, thick=None):
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    a, p, d, e = con.woltparam(r0, z0)
    if thick is not None:
        prog = _surface_recorder(rays) if check is not True else None
        if prog is not None:
            getattr(prog, which)(a, z0, psi, thick)
            return
        flush(rays)
        if check is True:
            x0, y0, zz0 = x.clone(), y.clone(), z.clone()
        getattr(wolt, which)(x, y, z, l, m, n, ux, uy, uz, a, z0, psi, thick)
        if check is True:
            return torch.logical_and(x0 == x, torch.logical_and(y0 == y, zz0 == z))
        return
    if check is True:
        # The reference's check=True path overwrites the scalar z0 with an array before the
        # Fortran call (surfaces.py:340-342) and cannot run; here it does what its docstring says.
        flush(rays)
        x0, y0, zz0 = x.clone(), y.clone(), z.clone()
    prog = recorder_for(rays)
    if prog is not None and check is not True:
        getattr(prog, which)(a, z0, psi)
        return
    getattr(wolt, which)(x, y, z, l, m, n, ux, uy, uz, a, z0, psi)
    if check is True:
        return torch.logical_and(x0 == x, torch.logical_and(y0 == y, zz0 == z))
    return


def wsPrimary(rays, r0, z0, psi, check=False):
    """Wolter-Schwarzschild primary; alpha from ``conicsolve.woltparam``."""
    return _ws(rays, "wsprimary", r0, z0, psi, check)


def wsSecondary(rays, r0, z0, psi, check=False):
    """Wolter-Schwarzschild secondary."""
    return _ws(rays, "wssecondary", r0, z0, psi, check)


def wsPrimaryB(rays, r0, z0, psi, thick, check=False):
    """Back surface of a Wolter-Schwarzschild primary of thickness ``thick``."""
    return _ws(rays, "wsprimaryback", r0, z0, psi, check, thick)


def wsSecondaryB(rays, r0, z0, psi, thick, check=False):
    """Back surface of a Wolter-Schwarzschild secondary of thickness ``thick``."""
    return _ws(rays, "wssecondaryback", r0, z0, psi, check, thick)


def spoCone(rays, R0, tg, ind=None):
    """SPO cone with intersection radius R0 and slope angle tg."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = recorder_for(rays) if ind is None else None
    if prog is not None:
        prog.spocone(R0, tg)
        return
    flush(rays)
    wolt.spocone(x, y, z, l, m, n, ux, uy, uz, R0, tg, mask=ind)
    return


def spoPrimary(rays, R0, F, d=.605, ind=None):
    """SPO primary: tg = atan((R0+d/2)/F)/4."""
    tg = .25 * np.arctan((R0 + d / 2) / F)
    spoCone(rays, R0, tg, ind=ind)
    return


def spoSecondary(rays, R0, F, d=.605, ind=None):
    """SPO secondary: tg = 3 atan((R0+d/2)/F)/4."""
    tg = .75 * np.arctan((R0 + d / 2) / F)
    spoCone(rays, R0, tg, ind=ind)
    return


def _zernsurf_recorder(prog, *rorders):
    """Whether ``prog`` (a recording program or None) can hold one more Zernike surface of these radial orders."""
    return (prog is not None and max(np.max(np.asarray(r)) for r in rorders) <= ZERN_MAX_ORDER and
            not any(c in (OP["ZERNSURF"], OP["LLSURF"], OP["ZERNPHASE"]) + SURFACE_OPS + ARRAY_OPS for c, _ in prog.ops))


def _surface_recorder(rays):
    """The program recording for ``rays`` when it can hold one of the remaining scalar surfaces (sphere, cylinder,
    cylconic, paraxial lenses, torus, W-S back surfaces: no Zernike surface, LL shell or grating fan in it), else None."""
    prog = recorder_for(rays)
    return prog if prog is not None and prog.can_hold_surface() else None


def _ll_recorder(rays, coeff, axial, az):
    """The program recording for ``rays`` when it can hold one more Legendre-Legendre shell with these terms (orders
    <= 7, fewer than two shells so far, no Zernike surface, grating fan or remaining scalar surface), else None."""
    prog = recorder_for(rays)
    if prog is None:
        return None
    try:
        c, ax, a = (np.asarray(v).ravel() for v in (coeff, axial, az))
        ok = (c.shape[0] > 0 and c.shape == ax.shape == a.shape and np.all(np.equal(np.mod(ax, 1), 0))
              and np.all(np.equal(np.mod(a, 1), 0)) and ax.min() >= 0 and a.min() >= 0
              and max(ax.max(), a.max()) <= LL_MAX_ORDER)
    except (TypeError, ValueError):
        ok = False
    codes = [code for code, _ in prog.ops]
    if not ok or codes.count(OP["LLSURF"]) >= LL_MAX_OPS or any(
            code in codes for code in (OP["ZERNSURF"], OP["ZERNPHASE"], OP["GRATFAN"], OP["ROTX_REMAINING"]) + SURFACE_OPS
            + ARRAY_OPS):
        return None
    return prog


def secondaryLL(rays, r0, z0, psi, zmax, zmin, dphi, coeff, axial, az):
    """Wolter-I secondary with Legendre-Legendre figure terms, placed at the focus."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = _ll_recorder(rays, coeff, axial, az)
    if prog is not None:
        prog.woltersecll(r0, z0, psi, zmax, zmin, dphi, coeff, axial, az)
        return
    flush(rays)
    wolt.woltersecll(x, y, z, l, m, n, ux, uy, uz, r0, z0, psi, zmax, zmin, dphi, coeff, axial, az)
    return


def primaryLL(rays, r0, z0, zmax, zmin, dphi, coeff, axial, az):
    """Wolter-I primary with Legendre-Legendre figure terms, placed at the focus."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = _ll_recorder(rays, coeff, axial, az)
    if prog is not None:
        prog.wolterprimll(r0, z0, zmax, zmin, dphi, coeff, axial, az)
        return
    flush(rays)
    wolt.wolterprimll(x, y, z, l, m, n, ux, uy, uz, r0, z0, zmax, zmin, dphi, coeff, axial, az)
    return


def ellipsoidPrimary(rays, R0, F, S, psi):
    """Primary of an ellipsoid-hyperboloid telescope (a conic placed at its vertex)."""
    P, a, b, e, f = con.ellipsoidFunction(S, psi, R0, F)
    R = b ** 2 / a
    tran.transform(rays, 0, 0, F + f - P - a, 0, 0, 0)
    conic(rays, R, -e ** 2)
    tran.itransform(rays, 0, 0, F + f - P - a, 0, 0, 0)
    return


def ellipsoidSecondary(rays, R0, F, S, psi):
    """Secondary of an ellipsoid-hyperboloid telescope (a Wolter secondary with an effective psi)."""
    P, a, b, e, f = con.ellipsoidFunction(S, psi, R0, F)
    psi_eff = np.arctan(R0 / P) / (np.arctan(R0 / F) - np.arctan(R0 / P))
    woltersecondary(rays, R0, F, psi=psi_eff)
    return


def ellipsoidPrimaryLL(rays, R0, F, S, psi, zmax, zmin, dphi, coeff, axial, az):
    """Ellipsoid primary with Legendre-Legendre figure terms."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = _ll_recorder(rays, coeff, axial, az)
    if prog is not None:
        prog.ellipsoidwoltll(R0, F, psi, S, zmax, zmin, dphi, coeff, axial, az)
        return
    flush(rays)
    wolt.ellipsoidwoltll(x, y, z, l, m, n, ux, uy, uz, R0, F, psi, S, zmax, zmin, dphi, coeff, axial, az)
    return


def ellipsoidSecondaryLL(rays, R0, F, S, psi, zmax, zmin, dphi, coeff, axial, az):
    """Hyperboloid secondary of an ellipsoid-hyperboloid telescope with L-L figure terms."""
    P, a, b, e, f = con.ellipsoidFunction(S, psi, R0, F)
    psi_eff = np.arctan(R0 / P) / (np.arctan(R0 / F) - np.arctan(R0 / P))
    secondaryLL(rays, R0, F, psi_eff, zmax, zmin, dphi, coeff, axial, az)
    return


def _move_segments(rays, dz, segments, nr):
    # every segment by its own dz: transform(rays, 0, 0, dz[k], 0, 0, 0) + flat, as the recorder would record them
    from .program import Program, SegmentedProgram
    progs = []
    for d in dz:
        p = Program().transform(-0., -0., -float(d), -0., -0., -0.)
        progs.append(p.flatopd(nr) if nr is not None else p.flat())
    SegmentedProgram(progs, segments.sizes(), device=rays[1].device).run(rays)


def focus(rays, fn, weights=None, nr=None, coords=None, segments=None):
    """Two-pass best focus (surfaces.py:502-510).  Each "move the plane, trace to it" pair runs as one fused
    kernel (same bits as the two calls).  ``segments``: every segment is moved by its own dz (one segmented launch
    per pass) and the dz of every segment is returned (np.ndarray[nseg]); not with ``coords``."""
    from .program import fused, flush, recorder_for
    if segments is not None:
        if coords is not None:
            raise ValueError("focus: coords= cannot follow per-segment moves")
        flush(rays)
        dz1 = fn(rays, weights=weights, segments=segments)
        _move_segments(rays, dz1, segments, nr)
        dz2 = fn(rays, weights=weights, segments=segments)
        _move_segments(rays, dz2, segments, nr)
        return dz1 + dz2
    own = recorder_for(rays) is None
    dz1 = fn(rays, weights=weights)
    if own:
        with fused(rays):
            tran.transform(rays, 0, 0, dz1, 0, 0, 0, coords=coords)
            flat(rays, nr=nr)
    else:
        tran.transform(rays, 0, 0, dz1, 0, 0, 0, coords=coords)
        flat(rays, nr=nr)
    dz2 = fn(rays, weights=weights)
    if own:
        with fused(rays):
            tran.transform(rays, 0, 0, dz2, 0, 0, 0, coords=coords)
            flat(rays, nr=nr)
    else:
        tran.transform(rays, 0, 0, dz2, 0, 0, 0, coords=coords)
        flat(rays, nr=nr)
    return dz1 + dz2


def focusI(rays, weights=None, nr=None, coords=None, segments=None):
    """Best focus from the analytic image plane (surfaces.py:518-519)."""
    return focus(rays, analyticImagePlane, weights=weights, nr=nr, coords=coords, segments=segments)


def focusY(rays, weights=None, nr=None, coords=None, segments=None):
    """Best line focus in y (surfaces.py:512-513)."""
    return focus(rays, analyticYPlane, weights=weights, nr=nr, coords=coords, segments=segments)


def focusX(rays, weights=None, nr=None, coords=None, segments=None):
    """Best line focus in x (surfaces.py:515-516)."""
    return focus(rays, analyticXPlane, weights=weights, nr=nr, coords=coords, segments=segments)


def _need_orders(rorder, aorder):
    if rorder is None or aorder is None:
        raise NotImplementedError("pass rorder/aorder explicitly: the reference's default ordering lives in "
                                  "the third-party module utilities.imaging.zernikemod (not vendored)")


def zernphase(rays, coeff, rad, wave, rorder=None, aorder=None):
    """Zernike phase surface: wavelength in mm, radius in mm, coeff in mm."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    _need_orders(rorder, aorder)
    prog = recorder_for(rays)
    if (prog is not None and np.max(np.asarray(rorder)) <= ZERN_MAX_ORDER and prog.can_hold_surface()
            and not any(c in SURFACE_OPS for c, _ in prog.ops)):
        prog.zernphase(coeff, rorder, aorder, rad, wave)    # radial orders <= 7: stays in the fused program
        return
    flush(rays)
    zern.zernphase(opd, x, y, z, l, m, n, ux, uy, uz, coeff, np.array(rorder), np.array(aorder), rad, wave)
    return


def zernsurfrot(rays, coeff1, coeff2, rad, rot, rorder1=None, aorder1=None, rorder2=None, aorder2=None):
    """Zernike surface made of two sets, the second rotated by ``rot`` (theta = arctan2(y,x))."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    _need_orders(rorder1, aorder1)
    _need_orders(rorder2, aorder2)
    prog = recorder_for(rays)
    if _zernsurf_recorder(prog, rorder1, rorder2):
        prog.tracezernrot(coeff1, rorder1, aorder1, coeff2, rorder2, aorder2, rad, rot)
        return
    flush(rays)
    zern.tracezernrot(x, y, z, l, m, n, ux, uy, uz, coeff1, np.array(rorder1), np.array(aorder1),
                      coeff2, np.array(rorder2), np.array(aorder2), rad, rot)
    return


def sphere(rays, rad, nr=None):
    """Sphere centred on the origin; the closer intersection is taken."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = _surface_recorder(rays)
    if prog is not None:
        if nr is not None:
            prog.tracesphereopd(rad, nr)
        else:
            prog.tracesphere(rad)
        return
    flush(rays)
    if nr is not None:
        surf.tracesphereopd(opd, x, y, z, l, m, n, ux, uy, uz, rad, nr)
    else:
        surf.tracesphere(x, y, z, l, m, n, ux, uy, uz, rad)
    return


def tanSphere(rays, rad, nr=None):
    """Sphere tangent to the XY plane; positive radius curves toward +z."""
    tran.transform(rays, 0, 0, rad, 0, 0, 0)
    sphere(rays, rad, nr=nr)
    tran.transform(rays, 0, 0, -rad, 0, 0, 0)
    return


def conicplus(rays, R, K, p, nr=None):
    """Conic of curvature radius R and conic constant K plus even polynomial terms p."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = _surface_recorder(rays)
    if prog is not None and np.size(p) <= CONICPLUS_MAX_TERMS:
        if nr is not None:
            prog.conicplusopd(R, K, p, nr)
        else:
            prog.conicplus(R, K, p)
        return
    flush(rays)
    if nr is not None:
        surf.conicplusopd(opd, x, y, z, l, m, n, ux, uy, uz, R, K, p, nr)
    else:
        surf.conicplus(x, y, z, l, m, n, ux, uy, uz, R, K, p)
    return


def oapCollimate(rays, efl, oapangle, nr=None):
    """Collimating off-axis paraboloid; returns the bundle back in the entry frame (new arrays)."""
    fp = efl * (1 + np.cos(oapangle)) / 2
    coords = tran.newCoords()
    tran.transform(rays, 0, 0, -efl, 0, 0, 0, coords=coords)
    tran.transform(rays, 0, 0, 0, np.pi - oapangle, 0, 0, coords=coords)
    tran.transform(rays, 0, 0, -fp, 0, 0, 0, coords=coords)
    conic(rays, fp * 2, -1, nr=nr)
    tran.reflect(rays)
    return tran.applyT(rays, coords, inverse=True)


def torus(rays, rin, rout):
    """Torus: outer radius in the xy plane, inner radius orthogonal."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = _surface_recorder(rays)
    if prog is not None:
        prog.torus(rin, rout)
        return
    flush(rays)
    surf.torus(x, y, z, l, m, n, ux, uy, uz, rin, rout)
    return


def cyl(rays, rad, nr=None):
    """Cylinder about the y axis through the origin."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = _surface_recorder(rays)
    if prog is not None:
        if nr is not None:
            prog.tracecylopd(rad, nr)
        else:
            prog.tracecyl(rad)
        return
    flush(rays)
    if nr is not None:
        surf.tracecylopd(opd, x, y, z, l, m, n, ux, uy, uz, rad, nr)
    else:
        surf.tracecyl(x, y, z, l, m, n, ux, uy, uz, rad)
    return


def cylconic(rays, rad, k):
    """Cylindrical conic (sag in y, cylinder axis z)."""
    opd, x, y, z, l, m, n, ux, uy, uz = rays
    prog = _surface_recorder(rays)
    if prog is not None:
        prog.cylconic(rad, k)
        return
    flush(rays)
    surf.cylconic(x, y, z, l, m, n, ux, uy, uz, rad, k)


def paraxial(rays, F):
    """Ideal paraxial lens in the xy plane, optical axis z."""
    x, y, z, l, m, n, ux, uy, uz = rays[1:]
    prog = _surface_recorder(rays)
    if prog is not None:
        prog.paraxial(F)
        return
    flush(rays)
    surf.paraxial(x, y, z, l, m, n, ux, uy, uz, F)
    return


def paraxialY(rays, F):
    """Ideal paraxial cylinder lens acting on y only."""
    x, y, z, l, m, n, ux, uy, uz = rays[1:]
    prog = _surface_recorder(rays)
    if prog is not None:
        prog.paraxialy(F)
        return
    flush(rays)
    surf.paraxialy(x, y, z, l, m, n, ux, uy, uz, F)
    return


def legSurf(rays, xwidth, ywidth, order, coeff, xo, yo):
    """Diffract from a phase surface given by 2-D Legendre coefficients (rays already on the xy plane)."""
    x, y, z, l, m, n, ux, uy, uz = rays[1:]
    prog = _surface_recorder(rays)
    if prog is not None and _legsurf_terms_ok(coeff, xo, yo):
        prog.legsurf(xwidth, ywidth, order, coeff, xo, yo)
        return
    flush(rays)
    surf.legsurf(x, y, z, l, m, n, ux, uy, uz, xwidth, ywidth, order,
                 np.asarray(coeff).flatten(), np.asarray(xo).flatten(), np.asarray(yo).flatten())
    return


def _legsurf_terms_ok(coeff, xo, yo):
    """Whether the term list is one the table fill takes (else the stand-alone routine reports the error)."""
    c, a, b = (np.asarray(v).ravel() for v in (coeff, xo, yo))
    if c.shape != a.shape or c.shape != b.shape or c.shape[0] > LEGSURF_MAX_TERMS:
        return False
    orders = np.concatenate([a, b]).astype(np.int32)
    return orders.size == 0 or (orders.min() >= 0 and orders.max() <= LEGSURF_MAX_ORDER)


# The reference's three tangent-plane placements still use its pre-`rays` module-global call style
# (bare transform(...), wolterprimary(r0,z0): surfaces.py:254-262) and raise NameError as shipped;
# these do what their comments say, with the bundle passed through.
def _to_tangent(rays, r0, z0, alpha):
    tran.transform(rays, 0, 0, 0, -np.pi / 2 - alpha, 0, 0)
    tran.transform(rays, 0, con.primrad(z0 + 75., r0, z0), -z0 - 75., 0, 0, 0)


def _from_tangent(rays, r0, z0, alpha):
    tran.transform(rays, 0, -con.primrad(z0 + 75., r0, z0), z0 + 75., 0, 0, 0)
    tran.transform(rays, 0, 0, 0, np.pi / 2 + alpha, 0, 0)


def wolterprimtan(rays, r0, z0):
    """Wolter primary placed at its tangent point: +z surface normal, +y to the sky, +x azimuthal."""
    alpha, p, d, e = con.woltparam(r0, z0)
    _to_tangent(rays, r0, z0, alpha)
    wolterprimary(rays, r0, z0)
    _from_tangent(rays, r0, z0, alpha)
    return


def woltersinetan(rays, r0, z0, amp, freq):
    """Sinusoidal Wolter primary placed at its tangent point."""
    alpha, p, d, e = con.woltparam(r0, z0)
    _to_tangent(rays, r0, z0, alpha)
    woltersine(rays, r0, z0, amp, freq)
    _from_tangent(rays, r0, z0, alpha)
    return


def primaryLLtan(rays, r0, z0, zmax, zmin, dphi, coeff, axial, az):
    """Legendre-Legendre Wolter primary placed at its tangent point."""
    alpha, p, d, e = con.woltparam(r0, z0)
    _to_tangent(rays, r0, z0, alpha)
    tran.transform(rays, 0, 0, 0, 0, 0, -np.pi / 2)
    primaryLL(rays, r0, z0, zmax, zmin, dphi, coeff, axial, az)
    tran.transform(rays, 0, 0, 0, 0, 0, np.pi / 2)
    _from_tangent(rays, r0, z0, alpha)
    return
