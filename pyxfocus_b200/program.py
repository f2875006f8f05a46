"""Fused per-ray programs: a whole chain of f2py routines in ONE kernel launch.

The reference runs a trace as a sequence of Fortran calls, each a full pass over the
bundle in memory (SURVEY.md 3.1: ~7 passes for a Wolter-I pair).  ``Program`` records the
same routines -- same names and argument meaning as the f2py modules -- and
``pxf_trace_program`` executes the list per ray in registers: rows are read from HBM once
and written once.  The arithmetic is the same device code as the per-routine kernels, so the
result is bit-identical to issuing the routines one by one.

Two ways to use it:

* explicitly::

      prog = Program().transform(0, 0, 8400., 0, 0, 0).wolterprimary(220., 8400., 1.).reflect()
      prog.run(rays)

* transparently, with the reference's own call sequence::

      with fused(rays):
          tran.transform(rays, 0, 0, -8400., 0, 0, 0)
          surf.wolterprimary(rays, 220., 8400.)
          tran.reflect(rays)
      # one kernel launch happens on exit (or as soon as something needs the rays)
"""
import ctypes

import torch

from . import _lib
from ._call import stream_ptr

OP = dict(TRANSFORM=1, ITRANSFORM=2, REFLECT=3, REFRACT=4, RADGRAT=5, FLAT=6, FLATOPD=7, CONIC=8,
          CONICOPD=9, WOLTERPRIMARY=10, WOLTERPRIMARYOPD=11, WOLTERSECONDARY=12, WOLTERSINE=13,
          WSPRIMARY=14, WSSECONDARY=15, SPOCONE=16, VIGNETTE_MAG=17, VIGNETTE_BOX=18,
          VIGNETTE_ABS=19, KICK=20, ZERNSURF=21, KICKN=22, VIGNETTE_RHOGT=23, GRATFAN=24, ROTX_REMAINING=25,
          LLSURF=26, TRACESPHERE=27, TRACESPHEREOPD=28, TRACECYL=29, TRACECYLOPD=30, CYLCONIC=31, PARAXIAL=32,
          PARAXIALY=33, TORUS=34, WSPRIMARYBACK=35, WSSECONDARYBACK=36, ZERNPHASE=37, CONICPLUS=38, CONICPLUSOPD=39,
          LEGSURF=40, RADGRATW=41, GRAT=42)
MAX_OPS = 24
LL_MAX_ORDER = 7       # Legendre orders a fused program holds (higher orders run the stand-alone routines)
LL_MAX_OPS = 2         # Legendre-Legendre shells per program
_VIGNETTES = (OP["VIGNETTE_MAG"], OP["VIGNETTE_BOX"], OP["VIGNETTE_ABS"], OP["VIGNETTE_RHOGT"])
_AUX_OPS = (OP["GRATFAN"], OP["ROTX_REMAINING"])
# the surfaces read through a device table of their own (conicplus, legsurf)
TABLE_SURFACE_OPS = (OP["CONICPLUS"], OP["CONICPLUSOPD"], OP["LEGSURF"])
# the surface family (sphere .. W-S back surfaces, conicplus, legsurf) shares no program with a table or side-array op
SURFACE_OPS = tuple(range(OP["TRACESPHERE"], OP["WSSECONDARYBACK"] + 1)) + TABLE_SURFACE_OPS
# the gratings with per-ray arrays (radgratW, grat): the device address of each array travels in the op, at these p
# slots, and is indexed by the ray's index in the bundle
ARRAY_OPS = (OP["RADGRATW"], OP["GRAT"])
_ARRAY_SLOTS = {OP["RADGRATW"]: (0,), OP["GRAT"]: (1, 2)}
TABLE_AUX_OPS = (OP["ZERNSURF"], OP["LLSURF"]) + _AUX_OPS + (OP["ZERNPHASE"],) + ARRAY_OPS
ZERN_MAX_ORDER = 7     # Zernike radial orders a fused program holds
CONICPLUS_MAX_TERMS = 16   # polynomial terms of conicplus (surfacesf.f95:514-638)
LEGSURF_MAX_TERMS = 48     # Legendre terms of legsurf ...
LEGSURF_MAX_ORDER = 15     # ... and their orders (surfacesf.f95:642-668)


def _host_array(a, dtype):
    import numpy as np
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(np.asarray(a).ravel(), dtype=dtype)


def _per_ray(v, what, scalar_ok):
    """A per-ray array of a grating op as the program keeps it: a 1-D float64 CUDA tensor or numpy array (used as
    given), or -- where ``scalar_ok`` -- a float, broadcast to the bundle when the program runs."""
    import numpy as np
    if isinstance(v, torch.Tensor):
        if not v.is_cuda or v.dtype != torch.float64 or v.dim() != 1 or not v.is_contiguous():
            raise ValueError("%s must be a contiguous 1-D float64 CUDA tensor" % what)
        return v
    if isinstance(v, np.ndarray):
        if v.dtype != np.float64 or v.ndim != 1:
            raise ValueError("%s must be a 1-D float64 array" % what)
        return np.ascontiguousarray(v)
    if scalar_ok and np.ndim(v) == 0:
        return float(v)
    raise ValueError("%s must be a CUDA float64 tensor or a numpy float64 array with one entry per ray" % what)


def _zern_terms(coeff, rorder, aorder):
    import numpy as np
    c = np.ascontiguousarray(coeff, dtype=np.float64)
    r = np.ascontiguousarray(rorder, dtype=np.int32)
    a = np.ascontiguousarray(aorder, dtype=np.int32)
    if not (c.shape == r.shape == a.shape) or c.ndim != 1 or c.shape[0] == 0:
        raise ValueError("coeff, rorder, aorder must be 1-D arrays of one length")
    return c, r, a


class Program:
    """An ordered list of per-ray operations (arguments as the Fortran routine sees them)."""

    def __init__(self):
        self.ops = []
        self._tables = {}        # op index -> host table (uint8 tensor) of a ZERNSURF or LLSURF op
        self._dev_tables = {}    # (op index, device) -> its device copy
        self._arrays = {}        # op index -> per-ray arrays of a RADGRATW / GRAT op, in the order of _ARRAY_SLOTS
        self._dev_arrays = {}    # (op index, slot, device[, num]) -> the device copy of a host array / a broadcast scalar

    def __len__(self):
        return len(self.ops)

    def add(self, code, *p):
        if len(p) > 6:
            raise ValueError("an op carries at most 6 scalars")
        self.ops.append((int(code), [float(v) for v in p]))
        return self

    # --- transformationsf ---
    def transform(self, tx, ty, tz, rx, ry, rz):
        return self.add(OP["TRANSFORM"], tx, ty, tz, rx, ry, rz)

    def itransform(self, tx, ty, tz, rx, ry, rz):
        return self.add(OP["ITRANSFORM"], tx, ty, tz, rx, ry, rz)

    def reflect(self):
        return self.add(OP["REFLECT"])

    def refract(self, n1, n2):
        return self.add(OP["REFRACT"], n1, n2)

    def radgrat(self, wave, dpermm, order):
        return self.add(OP["RADGRAT"], wave, dpermm, order)

    def radgratw(self, wave, dpermm, order):
        """radgratW (transformationsf.f95:242-272): the radial grating with one wavelength per ray, the sign of n taken
        from y.  ``wave``: a float64 CUDA tensor or numpy array with one entry per ray of the bundle the program runs
        on (of the whole bundle in a ``SegmentedProgram``).  The program keeps a reference and reads it when it runs;
        a host array is uploaded once per device."""
        w = _per_ray(wave, "wave", False)
        self._check_arrays("radgratw")
        self._arrays[len(self.ops)] = [w]
        return self.add(OP["RADGRATW"], 0., dpermm, order)

    def grat(self, d, order, wave):
        """grat (transformationsf.f95:277-305): the linear grating with grooves along +y, with a per-ray order and
        wavelength (arrays as for ``radgratw``; a scalar is broadcast to every ray, as ``transformations.grat`` does)."""
        o, w = _per_ray(order, "order", True), _per_ray(wave, "wave", True)
        self._check_arrays("grat")
        self._arrays[len(self.ops)] = [o, w]
        return self.add(OP["GRAT"], d, 0., 0.)

    def can_hold_arrays(self):
        """Whether ``radgratw`` / ``grat`` may join this program: they run in the side-array interpreter, which holds
        no Zernike surface or phase, LL shell or op of the surface family (``SURFACE_OPS``)."""
        return not any(c in SURFACE_OPS or c in (OP["ZERNSURF"], OP["ZERNPHASE"], OP["LLSURF"]) for c, _ in self.ops)

    def _check_arrays(self, what):
        if not self.can_hold_arrays():
            raise NotImplementedError("%s cannot share a program with a Zernike surface or phase, an LL shell or the "
                                      "sphere / cylinder / cylconic / paraxial / torus / W-S back-surface / conicplus / "
                                      "legsurf ops" % what)

    def _refuse_with_arrays(self, what):
        if any(c in ARRAY_OPS for c, _ in self.ops):
            raise NotImplementedError("%s cannot share a program with radgratw / grat" % what)

    def device_arrays(self, num, device):
        """{op index: device tensors} of the per-ray arrays for a bundle of ``num`` rays on ``device``: CUDA tensors
        as given, host arrays uploaded and scalars broadcast (each once per device).  Raises ValueError for an array
        with another length or on another device."""
        device = torch.device(device)
        for k, vals in self._arrays.items():
            for j in range(len(vals)):
                self._check_array(k, j, num, device)
        return {k: [self._device_array(k, j, num, device) for j in range(len(vals))]
                for k, vals in self._arrays.items()}

    def _check_array(self, k, j, num, device):
        v = self._arrays[k][j]
        code = self.ops[k][0]
        what = "%s op %d, p[%d]" % ("radgratw" if code == OP["RADGRATW"] else "grat", k, _ARRAY_SLOTS[code][j])
        if isinstance(v, float):
            return
        if v.shape[0] != num:
            raise ValueError("%s: the array has %d entries, the bundle %d rays" % (what, v.shape[0], num))
        if isinstance(v, torch.Tensor) and v.device != device:
            raise ValueError("%s: the array lives on %s, the bundle on %s" % (what, v.device, device))

    def _device_array(self, k, j, num, device):
        v = self._arrays[k][j]
        if isinstance(v, torch.Tensor):
            return v
        key = (k, j, str(device)) if not isinstance(v, float) else (k, j, str(device), int(num))
        if key not in self._dev_arrays:
            self._dev_arrays[key] = (torch.full((int(num),), v, dtype=torch.float64, device=device)
                                     if isinstance(v, float) else torch.from_numpy(v).to(device))
        return self._dev_arrays[key]

    # --- surfacesf ---
    def flat(self):
        return self.add(OP["FLAT"])

    def flatopd(self, nr):
        return self.add(OP["FLATOPD"], nr)

    def conic(self, r, k):
        return self.add(OP["CONIC"], r, k)

    def conicopd(self, r, k, nr):
        return self.add(OP["CONICOPD"], r, k, nr)

    # --- woltsurf ---
    def wolterprimary(self, r0, z0, psi):
        return self.add(OP["WOLTERPRIMARY"], r0, z0, psi)

    def wolterprimaryopd(self, r0, z0, psi, nr):
        return self.add(OP["WOLTERPRIMARYOPD"], r0, z0, psi, nr)

    def woltersecondary(self, r0, z0, psi):
        return self.add(OP["WOLTERSECONDARY"], r0, z0, psi)

    def woltersine(self, r0, z0, amp, freq):
        return self.add(OP["WOLTERSINE"], r0, z0, amp, freq)

    def wsprimary(self, alpha, z0, psi):
        return self.add(OP["WSPRIMARY"], alpha, z0, psi)

    def wssecondary(self, alpha, z0, psi):
        return self.add(OP["WSSECONDARY"], alpha, z0, psi)

    def spocone(self, r0, tg):
        return self.add(OP["SPOCONE"], r0, tg)

    # --- the remaining scalar surfaces (surfacesf.f95:57-246, :251-296, :423-508; woltsurf.f95:726-933) ---
    def tracesphere(self, rad):
        return self._surface(OP["TRACESPHERE"], rad)

    def tracesphereopd(self, rad, nr):
        return self._surface(OP["TRACESPHEREOPD"], rad, nr)

    def tracecyl(self, rad):
        return self._surface(OP["TRACECYL"], rad)

    def tracecylopd(self, rad, nr):
        return self._surface(OP["TRACECYLOPD"], rad, nr)

    def cylconic(self, rad, k):
        return self._surface(OP["CYLCONIC"], rad, k)

    def paraxial(self, F):
        return self._surface(OP["PARAXIAL"], F)

    def paraxialy(self, F):
        return self._surface(OP["PARAXIALY"], F)

    def torus(self, rin, rout):
        return self._surface(OP["TORUS"], rin, rout)

    def wsprimaryback(self, alpha, z0, psi, thick):
        return self._surface(OP["WSPRIMARYBACK"], alpha, z0, psi, thick)

    def wssecondaryback(self, alpha, z0, psi, thick):
        return self._surface(OP["WSSECONDARYBACK"], alpha, z0, psi, thick)

    # --- surfaces with a folded table (surfacesf.f95:514-668): the table is uploaded once per device and read by
    # the kernel through its address ---
    def conicplus(self, R, K, p):
        return self._table_surface(OP["CONICPLUS"], self._conicplus_table(R, K, p, 0, 0.))

    def conicplusopd(self, R, K, p, nr):
        return self._table_surface(OP["CONICPLUSOPD"], self._conicplus_table(R, K, p, 1, nr))

    def legsurf(self, xwidth, ywidth, order, coeff, xo, yo):
        c, a, b = _host_array(coeff, "float64"), _host_array(xo, "int32"), _host_array(yo, "int32")
        if not (c.shape == a.shape == b.shape):
            raise ValueError("coeff, xo, yo must have one length")
        L = _lib.lib()
        tab = torch.empty(int(L.pxf_legsurf_table_bytes()), dtype=torch.uint8)
        if int(L.pxf_legsurf_table_fill(float(xwidth), float(ywidth), float(order), c.ctypes.data, a.ctypes.data,
                                        b.ctypes.data, c.shape[0], tab.data_ptr())) < 0:
            raise ValueError(L.pxf_last_error().decode())
        return self._table_surface(OP["LEGSURF"], tab)

    @staticmethod
    def _conicplus_table(R, K, p, opd, nr):
        pp = _host_array(p, "float64")
        L = _lib.lib()
        tab = torch.empty(int(L.pxf_conicplus_table_bytes()), dtype=torch.uint8)
        if int(L.pxf_conicplus_table_fill(float(R), float(K), pp.ctypes.data, pp.shape[0], opd, float(nr),
                                          tab.data_ptr())) < 0:
            raise ValueError(L.pxf_last_error().decode())
        return tab

    def _table_surface(self, code, tab):
        self._check_surface()
        self._tables[len(self.ops)] = tab
        return self.add(code, 0.)

    def can_hold_surface(self):
        """Whether one of the ops above may join this program (none of ``TABLE_AUX_OPS`` is in it)."""
        return not any(c in TABLE_AUX_OPS for c, _ in self.ops)

    def _check_surface(self):
        if any(c in ARRAY_OPS for c, _ in self.ops):
            raise NotImplementedError("the sphere / cylinder / cylconic / paraxial / torus / W-S back-surface / "
                                      "conicplus / legsurf ops cannot share a program with radgratw / grat")
        if not self.can_hold_surface():
            raise NotImplementedError("the sphere / cylinder / cylconic / paraxial / torus / W-S back-surface / "
                                      "conicplus / legsurf ops cannot share a program with a Zernike surface or phase, "
                                      "an LL shell or a grating fan")

    def _surface(self, code, *p):
        self._check_surface()
        return self.add(code, *p)

    def _refuse_with_surfaces(self, what):
        if any(c in SURFACE_OPS for c, _ in self.ops):
            raise NotImplementedError("%s cannot share a program with the sphere / cylinder / cylconic / paraxial / "
                                      "torus / W-S back-surface / conicplus / legsurf ops" % what)
        if any(c == OP["ZERNPHASE"] for c, _ in self.ops):
            raise NotImplementedError("%s cannot share a program with a Zernike phase surface" % what)

    # --- zernsurf ---
    def zernsurf(self, coeff, rorder, aorder, rad, nr=None):
        """tracezern / tracezernOPD (zernsurf.f95:8-203) inside the program; radial orders <= 7, one Zernike surface
        per program.  The term list is folded on the host exactly as for the stand-alone routine; the table is
        uploaded once per device and staged in shared memory by the kernel."""
        c, r, a = _zern_terms(coeff, rorder, aorder)
        self._check_zernsurf()
        L = _lib.lib()
        tab = torch.empty(int(L.pxf_zern_table_bytes()), dtype=torch.uint8)
        nmax = int(L.pxf_zern_table_fill(c.ctypes.data, r.ctypes.data, a.ctypes.data, c.shape[0], float(rad),
                                         0 if nr is None else 1, 0. if nr is None else float(nr), tab.data_ptr()))
        return self._zern_op(OP["ZERNSURF"], tab, nmax, 0. if nr is None else 1.)

    def tracezernrot(self, coeff1, rorder1, aorder1, coeff2, rorder2, aorder2, rad, rot):
        """tracezernrot (zernsurf.f95:257-359) inside the program: both sets fold into one Zernike table, the second
        rotated by ``rot``, and the program holds it as a ``zernsurf`` (the same rules apply)."""
        c1, r1, a1 = _zern_terms(coeff1, rorder1, aorder1)
        c2, r2, a2 = _zern_terms(coeff2, rorder2, aorder2)
        self._check_zernsurf()
        L = _lib.lib()
        tab = torch.empty(int(L.pxf_zern_table_bytes()), dtype=torch.uint8)
        nmax = int(L.pxf_zern_table_fill_rot(c1.ctypes.data, r1.ctypes.data, a1.ctypes.data, c1.shape[0],
                                             c2.ctypes.data, r2.ctypes.data, a2.ctypes.data, c2.shape[0], float(rad),
                                             float(rot), tab.data_ptr()))
        return self._zern_op(OP["ZERNSURF"], tab, nmax, 0.)

    def zernphase(self, coeff, rorder, aorder, rad, wave):
        """zernphase (zernsurf.f95:206-250) inside the program; radial orders <= 7.  A program's only Zernike-table
        op: it shares no program with a Zernike surface, an LL shell, a grating fan or the surface family."""
        c, r, a = _zern_terms(coeff, rorder, aorder)
        if not self.can_hold_surface() or any(code in SURFACE_OPS for code, _ in self.ops):
            raise NotImplementedError("a Zernike phase surface cannot share a program with another Zernike surface or "
                                      "phase, an LL shell, a grating fan or the sphere .. legsurf surface ops")
        L = _lib.lib()
        tab = torch.empty(int(L.pxf_zern_table_bytes()), dtype=torch.uint8)
        nmax = int(L.pxf_zern_table_fill(c.ctypes.data, r.ctypes.data, a.ctypes.data, c.shape[0], float(rad), 0, 0.,
                                         tab.data_ptr()))
        return self._zern_op(OP["ZERNPHASE"], tab, nmax, float(wave))

    def _check_zernsurf(self):
        if any(code == OP["ZERNSURF"] for code, _ in self.ops):
            raise ValueError("a program carries at most one Zernike surface")
        if any(code == OP["LLSURF"] for code, _ in self.ops):
            raise NotImplementedError("a Zernike surface and Legendre-Legendre shells in one program are not supported")
        self._refuse_with_surfaces("a Zernike surface")
        self._refuse_with_arrays("a Zernike surface")

    def _zern_op(self, code, tab, nmax, p1):
        if nmax < 0:
            raise ValueError("invalid Zernike term list")
        if nmax > ZERN_MAX_ORDER:
            raise NotImplementedError("fused Zernike surfaces support radial orders <= %d" % ZERN_MAX_ORDER)
        self._tables[len(self.ops)] = tab
        return self.add(code, 0., p1, float(nmax))

    # --- Legendre-Legendre shells (woltsurf.f95:219-379, :643-718) ---
    def wolterprimll(self, r0, z0, zmax, zmin, dphi, coeff, axial, az):
        """wolterprimLL inside the program (arguments as ``woltsurf.wolterprimll``)."""
        return self._ll(0, r0, z0, 1., 0., zmax, zmin, dphi, coeff, axial, az)

    def woltersecll(self, r0, z0, psi, zmax, zmin, dphi, coeff, axial, az):
        """woltersecLL inside the program (arguments as ``woltsurf.woltersecll``)."""
        return self._ll(1, r0, z0, psi, 0., zmax, zmin, dphi, coeff, axial, az)

    def ellipsoidwoltll(self, r0, z0, psi, S, zmax, zmin, dphi, coeff, axial, az):
        """ellipsoidWoltLL inside the program (arguments as ``woltsurf.ellipsoidwoltll``)."""
        return self._ll(2, r0, z0, psi, S, zmax, zmin, dphi, coeff, axial, az)

    def _ll(self, kind, r0, z0, psi, S, zmax, zmin, dphi, coeff, axial, az):
        # Legendre orders <= 7, at most two shells per program, none with a Zernike surface.  The term list is folded
        # on the host exactly as for the stand-alone routine; the table is uploaded once per device and staged in
        # shared memory by the kernel.
        import numpy as np
        c = np.ascontiguousarray(np.asarray(coeff, dtype=np.float64).ravel())
        ax = np.asarray(axial).ravel()
        a = np.asarray(az).ravel()
        if not (c.shape == ax.shape == a.shape) or c.shape[0] == 0:
            raise ValueError("coeff, axial, az must be 1-D arrays of one length")
        if not (np.all(np.equal(np.mod(ax, 1), 0)) and np.all(np.equal(np.mod(a, 1), 0))) or ax.min() < 0 or a.min() < 0:
            raise ValueError("Legendre orders must be non-negative integers")
        ax, a = np.ascontiguousarray(ax, dtype=np.int32), np.ascontiguousarray(a, dtype=np.int32)
        if max(ax.max(), a.max()) > LL_MAX_ORDER:
            raise NotImplementedError("fused Legendre-Legendre shells support orders <= %d" % LL_MAX_ORDER)
        if sum(code == OP["LLSURF"] for code, _ in self.ops) >= LL_MAX_OPS:
            raise NotImplementedError("a program carries at most %d Legendre-Legendre shells" % LL_MAX_OPS)
        if any(code == OP["ZERNSURF"] for code, _ in self.ops):
            raise NotImplementedError("a Zernike surface and Legendre-Legendre shells in one program are not supported")
        self._refuse_with_surfaces("a Legendre-Legendre shell")
        self._refuse_with_arrays("a Legendre-Legendre shell")
        L = _lib.lib()
        tab = torch.empty(int(L.pxf_ll_table_bytes()), dtype=torch.uint8)
        top = int(L.pxf_ll_table_fill(kind, float(r0), float(z0), float(psi), float(S), float(zmax), float(zmin),
                                      float(dphi), c.ctypes.data, ax.ctypes.data, a.ctypes.data, c.shape[0],
                                      tab.data_ptr()))
        if top < 0:
            raise ValueError("invalid Legendre-Legendre term list: " + L.pxf_last_error().decode())
        self._tables[len(self.ops)] = tab
        return self.add(OP["LLSURF"], 0., float(top))

    # --- per-ray predicates (the ray stops at the op; use with ``alive``) ---
    def vignette_mag(self):
        """keep rays with l^2+m^2+n^2 > .1 (transformations.py:220-223)"""
        return self.add(OP["VIGNETTE_MAG"])

    def vignette_box(self, row, lo, hi):
        """keep rays with lo < rays[row] < hi"""
        return self.add(OP["VIGNETTE_BOX"], row, lo, hi)

    def vignette_abs(self, row, hi, centre=0.):
        """keep rays with |rays[row] - centre| < hi"""
        return self.add(OP["VIGNETTE_ABS"], row, hi, centre)

    def vignette_rhogt(self, rho0):
        """keep rays with sqrt(x^2+y^2) > rho0 (examples/axro/axialHeights.py:285-286)"""
        return self.add(OP["VIGNETTE_RHOGT"], rho0)

    def kickn(self, dl, dm):
        """l += dl, m += dm, n = -sqrt(n^2-dl^2-dm^2) (pointing offsets, examples/arcus/cat.py:246-249)"""
        return self.add(OP["KICKN"], dl, dm)

    def gratfan(self, ang, hubdist, l, dpermm, order, wave):
        """The fanned radial-grating array of examples/arcus/sector.py:681-707 as one per-ray loop: each ray is
        rotated about the hub axis by ``ang`` per grating (traced to the grating plane when steep enough) until it
        lands between ``hubdist`` and ``l + hubdist`` from the hub, then reflected and diffracted.  ``wave``: a
        float [nm] (radgrat) or a per-ray CUDA tensor (radgratW).  ``run`` needs ``aux=FanAux(...)``: the per-ray
        grating index and its maximum come back there."""
        self._refuse_with_surfaces("a grating fan")
        if isinstance(wave, torch.Tensor):
            self._wave = wave
            w = float("nan")
        else:
            w = float(wave)
        return self.add(OP["GRATFAN"], ang, hubdist, l, dpermm, order, w)

    def rotx_remaining(self, ang, total):
        """transform(0,0,0,ang,0,0) applied (total - count[i]) times: the whole-bundle fan rotations a ray still
        receives after it met its grating (sector.py:693), with ``count`` from a previous ``gratfan``."""
        self._refuse_with_surfaces("rotx_remaining")
        return self.add(OP["ROTX_REMAINING"], ang, total)

    def kick(self, dl, dm, sn):
        """l += dl, m += dm, n = sn*sqrt(1-l^2-m^2) (field-angle kick, axialHeights.py:94-95)"""
        return self.add(OP["KICK"], dl, dm, sn)

    # --- execution ---
    def has_vignette(self):
        return any(c in _VIGNETTES for c, _ in self.ops)

    def c_ops(self, device=None, arrays=None):
        """The ops as the C ABI takes them; ``arrays``: ``device_arrays`` of the bundle, whose addresses the RADGRATW /
        GRAT ops carry."""
        import struct
        arr = (_lib.pxf_op * len(self.ops))()
        for k, (code, p) in enumerate(self.ops):
            arr[k].code = code
            for j, v in enumerate(p):
                arr[k].p[j] = v
            if k in self._tables:
                if device is None:
                    raise ValueError("a program with an op that carries a table needs a device")
                key = (k, str(device))
                if key not in self._dev_tables:
                    self._dev_tables[key] = self._tables[k].to(device)
                # the table's device address travels bit-cast in p[0] (include/pxf.h, PXF_OP_ZERNSURF, LLSURF, ...)
                arr[k].p[0] = struct.unpack("d", struct.pack("Q", self._dev_tables[key].data_ptr()))[0]
            if k in self._arrays:
                if arrays is None:
                    raise ValueError("a program with radgratw / grat needs the bundle's arrays (Program.device_arrays)")
                for slot, t in zip(_ARRAY_SLOTS[code], arrays[k]):
                    arr[k].p[slot] = struct.unpack("d", struct.pack("Q", t.data_ptr()))[0]
        return arr

    def precompile(self, segmented=False):
        """Compile the run-time specialised kernels this program will want (no GPU needed; cached on disk under
        ``pyxfocus_b200/_jit``).  Returns the number of kernels available (0: NVRTC unavailable -- the interpreter
        will be used)."""
        import struct
        arr = (_lib.pxf_op * len(self.ops))()
        for k, (code, p) in enumerate(self.ops):
            arr[k].code = code
            for j, v in enumerate(p):
                arr[k].p[j] = v
            if k in self._tables:
                arr[k].p[0] = struct.unpack("d", struct.pack("Q", 8))[0]      # any non-null table address
            for slot in _ARRAY_SLOTS.get(code, ()):
                arr[k].p[slot] = struct.unpack("d", struct.pack("Q", 8))[0]   # ... and array address
        n = int(_lib.lib().pxf_jit_compile(arr, len(self.ops), 1 if segmented else 0, None))
        if n < 0:
            _lib.check(1)
        return n

    def run(self, rays, alive=None, out=None, sums=None, aux=None):
        """Execute on a bundle (list of ten CUDA fp64 rows).  Returns the ``alive`` uint8
        tensor when the program contains a vignette predicate (allocated if not given).
        ``out``: optional second bundle -- rows are read from ``rays`` and every row the program
        touches is written to ``out``; ``rays`` is left untouched.
        ``sums``: optional CUDA float64 tensor (>= 16 entries) that receives, from the same
        kernel, {count, sum x, sum y, count} of the final bundle over the surviving rays --
        pass it on to ``analyses.hpd(..., sums=sums)`` to skip the centroid pass."""
        if not self.ops:
            return alive
        if len(self.ops) > MAX_OPS:
            # split into several launches; still one HBM round trip per <=24 elements
            head, tail = Program(), Program()
            head.ops, tail.ops = self.ops[:MAX_OPS], self.ops[MAX_OPS:]
            head._tables = {k: v for k, v in self._tables.items() if k < MAX_OPS}
            tail._tables = {k - MAX_OPS: v for k, v in self._tables.items() if k >= MAX_OPS}
            head._arrays = {k: v for k, v in self._arrays.items() if k < MAX_OPS}
            tail._arrays = {k - MAX_OPS: v for k, v in self._arrays.items() if k >= MAX_OPS}
            if head.has_vignette() or tail.has_vignette():
                raise ValueError("programs with vignette predicates are limited to %d ops" % MAX_OPS)
            if out is not None:
                # the head stores only the rows it touches: give `out` every row first, then run both parts in place
                for k in range(10):
                    if rays[k] is not None and out[k] is not None:
                        out[k].copy_(rays[k])
                rays = out
            head.run(rays)
            return tail.run(rays, sums=sums)
        dev = rays[1].device
        num = rays[1].shape[0]
        for r in rays:
            if r is not None and (not r.is_cuda or r.dtype != torch.float64 or not r.is_contiguous()
                                  or r.shape[0] != num):
                raise ValueError("ray rows must be contiguous 1-D float64 CUDA tensors of equal length")
        if self.has_vignette() and alive is None:
            alive = torch.empty(num, dtype=torch.uint8, device=dev)
        ptrs = (ctypes.c_void_p * 10)(*[(r.data_ptr() if r is not None else None) for r in rays])
        arrays = self.device_arrays(num, dev) if self._arrays else None
        if arrays is not None and num == 0:
            return alive             # (an empty array has no address for the op to carry, and there is nothing to do)
        ops = self.c_ops(dev, arrays)
        ap = alive.data_ptr() if alive is not None else None
        optrs = None
        if out is not None:
            optrs = (ctypes.c_void_p * 10)(*[(r.data_ptr() if r is not None else None) for r in out])
        uses_aux = any(c in _AUX_OPS for c, _ in self.ops)
        if uses_aux and aux is None:
            raise ValueError("programs with gratfan / rotx_remaining need aux=FanAux(...)")
        with torch.cuda.device(dev):
            L = _lib.lib()
            if uses_aux:
                if sums is not None and (not sums.is_cuda or sums.dtype != torch.float64 or sums.numel() < 16):
                    raise ValueError("sums must be a contiguous CUDA float64 tensor with >= 16 entries")
                scratch = (torch.empty(int(L.pxf_sums_scratch_bytes()), dtype=torch.uint8, device=dev)
                           if sums is not None else None)
                wave = getattr(self, "_wave", None)
                if wave is not None and (not wave.is_cuda or wave.dtype != torch.float64 or not wave.is_contiguous()
                                         or wave.shape[0] != num):
                    raise ValueError("wave must be a contiguous CUDA float64 tensor with one entry per ray")
                ca = aux.c_struct(num, dev, wave)
                rc = L.pxf_trace_program_aux(ptrs, optrs, num, ops, len(self.ops), ap, ctypes.byref(ca),
                                             sums.data_ptr() if sums is not None else None,
                                             scratch.data_ptr() if scratch is not None else None, stream_ptr(dev))
            elif sums is not None:
                if not sums.is_cuda or sums.dtype != torch.float64 or sums.numel() < 16 or not sums.is_contiguous():
                    raise ValueError("sums must be a contiguous CUDA float64 tensor with >= 16 entries")
                scratch = torch.empty(int(L.pxf_sums_scratch_bytes()), dtype=torch.uint8, device=dev)
                rc = L.pxf_trace_program_sums(ptrs, optrs, num, ops, len(self.ops), ap, sums.data_ptr(),
                                              scratch.data_ptr(), stream_ptr(dev))
            elif out is None:
                rc = L.pxf_trace_program(ptrs, num, ops, len(self.ops), ap, stream_ptr(dev))
            else:
                rc = L.pxf_trace_program_to(ptrs, optrs, num, ops, len(self.ops), ap, stream_ptr(dev))
        _lib.check(rc)
        return alive


class FanAux:
    """Side arrays of a grating-fan program (include/pxf.h, pxf_program_aux): ``count`` int32[num] = gratings passed
    per ray (-1: none met), ``count_max`` int32[1] = the largest (cap + 1 if some ray met none)."""

    def __init__(self, num, device, cap=4096):
        self.count = torch.empty(int(num), dtype=torch.int32, device=device)
        self.count_max = torch.zeros(1, dtype=torch.int32, device=device)
        self.cap = int(cap)

    def c_struct(self, num, dev, wave):
        if self.count.shape[0] != num or self.count.device != dev:
            raise ValueError("FanAux was made for another bundle")
        a = _lib.pxf_program_aux()
        a.wave = wave.data_ptr() if wave is not None else None
        a.count = self.count.data_ptr()
        a.count_max = self.count_max.data_ptr()
        a.cap = self.cap
        return a

    def gratings(self):
        """Largest grating index of the launch (one 4-byte read-back); raises if some ray met no grating."""
        k = int(self.count_max.item())
        if k > self.cap:
            raise RuntimeError("gratfan: rays left after %d gratings (they never meet the array)" % self.cap)
        return k


class Segments:
    """Layout of a segmented bundle: segment k is rays ``start[k]:start[k+1]`` (``start`` host int64, nseg+1 entries,
    ``start[0] == 0``) with a device copy ``start_dev``.  The per-segment analyses (``segments=`` of ``analyses`` and
    ``surfaces.focus*``) take one; ``SegmentedProgram.segments`` is the layout a segmented trace ran with."""

    def __init__(self, sizes, device=None):
        import numpy as np
        sz = np.asarray(sizes)
        if sz.ndim != 1 or sz.shape[0] < 1:
            raise ValueError("segments need a 1-D list of at least one size")
        if not np.issubdtype(sz.dtype, np.integer) and not np.all(np.equal(np.mod(sz, 1), 0)):
            raise ValueError("segment sizes must be integers")
        sz = sz.astype(np.int64)
        if (sz < 0).any():
            raise ValueError("segment sizes must be non-negative")
        start = np.zeros(sz.shape[0] + 1, dtype=np.int64)
        start[1:] = np.cumsum(sz)
        self.start = start
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)
        self.device = torch.device(device)
        self._dev = None

    @classmethod
    def _from(cls, start, start_dev):
        seg = cls.__new__(cls)
        seg.start, seg._dev, seg.device = start, start_dev, start_dev.device
        return seg

    @property
    def start_dev(self):
        if self._dev is None:
            self._dev = torch.from_numpy(self.start).to(self.device)
        return self._dev

    @property
    def nseg(self):
        return self.start.shape[0] - 1

    @property
    def num(self):
        return int(self.start[-1])

    def sizes(self):
        import numpy as np
        return np.diff(self.start)

    def check(self, num, device):
        """Raise ValueError unless these segments describe a bundle of ``num`` rays on ``device``."""
        if num != self.num:
            raise ValueError("bundle has %d rays, the segments add up to %d" % (num, self.num))
        if torch.device(device) != self.device:
            raise ValueError("segments live on %s, the bundle on %s" % (self.device, device))

    def after(self, alive):
        """The segments of ``transformations.compact(rays, alive)``: survivors counted per segment on the device, one
        read-back of nseg int64; compaction keeps the order, so the new starts are their exclusive scan."""
        import numpy as np
        if not isinstance(alive, torch.Tensor) or alive.dtype != torch.uint8 or alive.dim() != 1:
            raise ValueError("alive must be a 1-D uint8 tensor")
        self.check(alive.shape[0], alive.device)
        counts = torch.empty(self.nseg, dtype=torch.int64, device=alive.device)
        with torch.cuda.device(alive.device):
            _lib.check(_lib.lib().pxf_segment_counts(alive.contiguous().data_ptr(), alive.shape[0], self.start_dev.data_ptr(),
                                                     self.nseg, counts.data_ptr(), stream_ptr(alive.device)))
        return Segments(counts.cpu().numpy(), device=alive.device)


class SegmentedProgram:
    """One launch for a bundle made of segments that run the same routines with different scalars -- a nested
    mirror assembly, one shell per segment (the reference loops over shells in Python,
    examples/axro/axialHeights.py:215-322, SMARTX.py:163-259)::

        progs = [Program().transform(0, 0, z0[k], 0, 0, 0).wolterprimary(r0[k], z0[k], 1.).reflect() ... for k]
        seg = SegmentedProgram(progs, sizes)      # sizes[k] = rays of shell k, concatenated in this order
        seg.run(bundle)

    The per-segment op tables are folded once on the host and uploaded once; ``run`` is a single kernel.

    Every program may carry one ``zernsurf`` at the same position, each with its own terms, ``rad`` and ``nr`` (a
    Monte Carlo over figure-error realisations, or a shell assembly with a measured figure per shell); the segment's
    Zernike table is staged with its op table.  ``nr`` must be given for all segments or for none.

    Likewise every program may carry one or two Legendre-Legendre shells (``wolterprimll`` / ``woltersecll`` /
    ``ellipsoidwoltll``) at the same positions, each segment with its own kind, terms and orders (<= 7).

    The remaining scalar surfaces (``tracesphere`` .. ``wssecondaryback``) take their own scalars per segment (a
    tolerance sweep over the radii of a lens pair, say); they share no program with a Zernike surface or an LL shell.
    So do ``conicplus`` / ``conicplusopd`` / ``legsurf``, each segment with its own table (a tolerance Monte Carlo over
    aspheric coefficients); the device copies of those tables are kept alive here.

    ``zernphase`` may take the place of ``zernsurf`` (the same op in every segment, each with its own terms and
    ``wave``), and a clocking sweep is a ``tracezernrot`` per segment whose ``rot`` differs.

    ``radgratw`` / ``grat`` take their scalars per segment; their arrays hold one entry per ray of the WHOLE bundle and
    segment k reads entries ``start[k]:start[k+1]`` (a program may give its own array or share one; a scalar ``order``
    / ``wave`` of ``grat`` is broadcast).  The arrays must live on the segmented program's device and are read when it
    runs."""

    def __init__(self, programs, sizes, device=None):
        import struct

        import numpy as np
        if len(programs) != len(sizes) or not programs:
            raise ValueError("one program per segment")
        nops = len(programs[0])
        if nops < 1 or nops > MAX_OPS:
            raise ValueError("segmented programs carry 1..%d ops" % MAX_OPS)
        for p in programs:
            if [c for c, _ in p.ops] != [c for c, _ in programs[0].ops]:
                raise ValueError("every segment must run the same routine sequence")
        self.nseg, self.nops = len(programs), nops
        self.has_vignette = programs[0].has_vignette()
        start = np.zeros(self.nseg + 1, dtype=np.int64)
        start[1:] = np.cumsum(np.asarray(sizes, dtype=np.int64))
        self.seg_start = start
        self.num = int(start[-1])
        arr = (_lib.pxf_op * (self.nseg * nops))()
        for sgm, prog in enumerate(programs):
            for k, (code, p) in enumerate(prog.ops):
                o = arr[sgm * nops + k]
                o.code = code
                for j, v in enumerate(p):
                    o.p[j] = v
        # (the device is looked up after the fill, which refuses a bad list first, unless tables go there before)
        dev = None if device is None else torch.device(device)
        # the tables of conicplus / legsurf ops are uploaded in one piece, kept here, and each segment's op carries the
        # device address of its own (16-byte aligned)
        tpos = [k for k, (c, _) in enumerate(programs[0].ops) if c in TABLE_SURFACE_OPS]
        self._op_tables = None
        if tpos:
            if any(k not in prog._tables for prog in programs for k in tpos):
                raise ValueError("a conicplus / legsurf op needs the table Program.conicplus / legsurf records")
            if dev is None:
                dev = torch.device("cuda", torch.cuda.current_device())
            parts, offs = [], []
            for prog in programs:
                for k in tpos:
                    t = prog._tables[k]
                    offs.append(sum(p.numel() for p in parts))
                    parts.append(torch.cat([t, torch.zeros(-t.numel() % 16, dtype=torch.uint8)]))
            self._op_tables = torch.cat(parts).to(dev)
            base = self._op_tables.data_ptr()
            for j, off in enumerate(offs):
                sgm, k = divmod(j, len(tpos))
                arr[sgm * nops + tpos[k]].p[0] = struct.unpack("d", struct.pack("Q", base + off))[0]
        # the per-ray arrays of radgratw / grat ops: each segment's op carries the addresses of its own program's arrays,
        # which hold one entry per ray of the whole bundle (segment s reads entries start[s]:start[s+1])
        apos = [k for k, (c, _) in enumerate(programs[0].ops) if c in ARRAY_OPS]
        self._arrays = []
        if apos:
            if any(k not in prog._arrays for prog in programs for k in apos):
                raise ValueError("a radgratw / grat op needs the arrays Program.radgratw / grat records")
            if dev is None:
                dev = torch.device("cuda", torch.cuda.current_device())
            shared = {}        # (op index, array) -> one bundle-long array for the segments that give a scalar there
            for sgm, prog in enumerate(programs):
                for k in apos:
                    for j, slot in enumerate(_ARRAY_SLOTS[prog.ops[k][0]]):
                        prog._check_array(k, j, self.num, dev)
                        v = prog._arrays[k][j]
                        if isinstance(v, float):
                            if (k, j) not in shared:
                                shared[k, j] = torch.zeros(self.num, dtype=torch.float64, device=dev)
                            t = shared[k, j]
                            t[int(start[sgm]):int(start[sgm + 1])] = v
                        else:
                            t = prog._device_array(k, j, self.num, dev)
                        self._arrays.append(t)
                        arr[sgm * nops + k].p[slot] = struct.unpack("d", struct.pack("Q", t.data_ptr()))[0]
        L = _lib.lib()
        zpos = [k for k, (c, _) in enumerate(programs[0].ops) if c in (OP["ZERNSURF"], OP["ZERNPHASE"])]
        lpos = [k for k, (c, _) in enumerate(programs[0].ops) if c == OP["LLSURF"]]
        if lpos:
            for p in programs:
                if any(k not in p._tables for k in lpos):
                    raise ValueError("an LL op needs the table Program.wolterprimll / woltersecll / ellipsoidwoltll "
                                     "records")
            # the LL tables of every segment, segment-major and in op order (include/pxf.h, pxf_segmented_table_fill_ll)
            lt = torch.cat([p._tables[k] for p in programs for k in lpos])
            nbytes = int(L.pxf_segmented_table_bytes_ll(nops, self.nseg))
            self.table_host = torch.empty(nbytes, dtype=torch.uint8)
            _lib.check(L.pxf_segmented_table_fill_ll(arr, nops, self.nseg, start.ctypes.data, lt.data_ptr(),
                                                     self.table_host.data_ptr()))
        elif zpos:
            kz = zpos[0]
            for p in programs:
                if kz not in p._tables:
                    raise ValueError("a zernsurf / zernphase op needs the table Program.zernsurf / zernphase records")
                if p.ops[kz][0] == OP["ZERNSURF"] and p.ops[kz][1][1] != programs[0].ops[kz][1][1]:
                    raise ValueError("every segment's zernsurf must give nr, or none may (tracezernOPD vs tracezern)")
            # one host table per segment, back to back (include/pxf.h, pxf_segmented_table_fill_zern)
            zt = torch.cat([p._tables[kz] for p in programs])
            nbytes = int(L.pxf_segmented_table_bytes_zern(nops, self.nseg))
            self.table_host = torch.empty(nbytes, dtype=torch.uint8)
            _lib.check(L.pxf_segmented_table_fill_zern(arr, nops, self.nseg, start.ctypes.data, zt.data_ptr(),
                                                       self.table_host.data_ptr()))
        else:
            nbytes = int(L.pxf_segmented_table_bytes(nops, self.nseg))
            self.table_host = torch.empty(nbytes, dtype=torch.uint8)
            _lib.check(L.pxf_segmented_table_fill(arr, nops, self.nseg, start.ctypes.data, self.table_host.data_ptr()))
        if dev is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.table_dev = self.table_host.to(dev)
        self.seg_start_dev = torch.from_numpy(start).to(dev)
        self.segments = Segments._from(start, self.seg_start_dev)

    def run(self, rays, alive=None, out=None):
        dev = rays[1].device
        num = rays[1].shape[0]
        if num != self.num:
            raise ValueError("bundle has %d rays, the segments add up to %d" % (num, self.num))
        if dev != self.table_dev.device:
            raise ValueError("segment table lives on %s, rays on %s" % (self.table_dev.device, dev))
        for r in rays:
            if r is not None and (not r.is_cuda or r.dtype != torch.float64 or not r.is_contiguous()
                                  or r.shape[0] != num):
                raise ValueError("ray rows must be contiguous 1-D float64 CUDA tensors of equal length")
        if self.has_vignette and alive is None:
            alive = torch.empty(num, dtype=torch.uint8, device=dev)
        ptrs = (ctypes.c_void_p * 10)(*[(r.data_ptr() if r is not None else None) for r in rays])
        optrs = None
        if out is not None:
            optrs = (ctypes.c_void_p * 10)(*[(r.data_ptr() if r is not None else None) for r in out])
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().pxf_trace_program_segmented(
                ptrs, optrs, num, self.table_host.data_ptr(), self.table_dev.data_ptr(),
                alive.data_ptr() if alive is not None else None, stream_ptr(dev)))
        return alive


# ------------------------------------------------------------------ transparent recording
_active = {}     # id(rays list) -> (rays, Program)


def recorder_for(rays):
    """Program currently recording for this bundle, or None."""
    ent = _active.get(id(rays))
    return ent[1] if ent is not None and ent[0] is rays else None


_alive = {}      # id(rays list) -> (rays, uint8 flags) left by the vignette predicates of the last recording


def last_alive(rays):
    """uint8 flag row written by the vignette predicates recorded for this bundle (1 = the ray passed every
    predicate), or None when the recording had none.  ``transformations.compact(rays, flags)`` removes the rest."""
    ent = _alive.get(id(rays))
    return ent[1] if ent is not None and ent[0] is rays else None


def flush(rays):
    """Execute whatever is pending for this bundle (called by anything that reads the rays)."""
    prog = recorder_for(rays)
    if prog is not None and len(prog):
        todo = Program()
        todo.ops, prog.ops = prog.ops, []
        todo._tables, prog._tables = prog._tables, {}
        todo._arrays, prog._arrays = prog._arrays, {}
        alive = todo.run(rays)
        if alive is not None:
            prev = last_alive(rays)
            # (a ray stopped in an earlier launch of the same recording stays stopped)
            _alive[id(rays)] = (rays, alive if prev is None else torch.minimum(prev, alive))


class fused:
    """Context manager: calls of the ``transformations``/``surfaces`` API on ``rays`` inside the
    block are recorded and executed as one kernel on exit."""

    def __init__(self, rays):
        self.rays = rays

    def __enter__(self):
        if id(self.rays) in _active:
            raise RuntimeError("bundle is already recording")
        _active[id(self.rays)] = (self.rays, Program())
        _alive.pop(id(self.rays), None)
        return self.rays

    def __exit__(self, et, ev, tb):
        try:
            if et is None:
                flush(self.rays)
        finally:
            _active.pop(id(self.rays), None)
        return False
