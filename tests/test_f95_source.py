"""The C oracle against the reference's Fortran SOURCE TEXT (SURVEY.md 8c).

There is no Fortran compiler in the image, so ``oracle/f95run.py`` executes the ``.f95`` files themselves: a translator for the
Fortran subset they use, with gfortran's arithmetic rules (REAL*4 literals and implicit typing, kind promotion, integer division,
``__powidf2`` powers, glibc libm).  ``tests/golden/make_f95_golden.py`` ran EVERY subroutine of transformationsf / surfacesf /
woltsurf / zernsurf / reconstruct on seeded rays and committed inputs and outputs (``tests/golden/f95_source.npz``).

* not gpu: ``oracle/pxf_oracle.c`` reproduces every vector bit for bit (this also runs on the GPU box); where the reference tree
  is present the translator is re-run on a sample of the cases and must reproduce the fixture; the translator's own arithmetic
  rules have known-answer tests.
* gpu: libpxf's per-routine entry points against the same vectors -- bit for bit for the routines without transcendentals in
  their loop, 1e-12 otherwise (the tolerance north_star states)."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from oracle import f2py as of, f95run, refload  # noqa: E402
from util import ROWS, assert_bit_equal, assert_close  # noqa: E402
import make_golden_reference_calls as rc  # noqa: E402
from make_golden_reference_calls import assert_pinned  # noqa: E402

HIDDEN = {"num", "arrsize", "arrsize1", "arrsize2", "cnum", "nc", "np"}
# Fortran dummy-argument order of every routine (from the .f95 headers; the fixture does not need the reference tree)
ARGS = {
    "reflect": "l m n ux uy uz num", "refract": "l m n ux uy uz num n1 n2",
    "transform": "x y z l m n ux uy uz num tx ty tz rx ry rz", "itransform": "x y z l m n ux uy uz num tx ty tz rx ry rz",
    "radgrat": "x y l m n wave num dpermm order", "radgratw": "x y l m n wave num dpermm order", "grat": "x y l m n num d order wave",
    "flat": "x y z l m n ux uy uz num", "flatopd": "x y z l m n ux uy uz opd num nr",
    "tracesphere": "x y z l m n ux uy uz num rad", "tracesphereopd": "opd x y z l m n ux uy uz num rad nr",
    "tracecyl": "x y z l m n ux uy uz num rad", "tracecylopd": "opd x y z l m n ux uy uz num rad nr",
    "cylconic": "x y z l m n ux uy uz num rad k", "conic": "x y z l m n ux uy uz num r k",
    "conicopd": "opd x y z l m n ux uy uz num r k nr", "paraxial": "x y z l m n ux uy uz num f", "paraxialy": "x y z l m n ux uy uz num f",
    "torus": "x y z l m n ux uy uz num rin rout", "conicplus": "x y z l m n ux uy uz num r k p np",
    "conicplusopd": "opd x y z l m n ux uy uz num r k p np nr",
    "legsurf": "x y z l m n ux uy uz xwidth ywidth order coeff xo yo nc num",
    "wolterprimary": "x y z l m n ux uy uz num r0 z0 psi", "wolterprimaryopd": "opd x y z l m n ux uy uz num r0 z0 psi nr",
    "woltersecondary": "x y z l m n ux uy uz num r0 z0 psi", "woltersine": "x y z l m n ux uy uz num r0 z0 amp freq",
    "wolterprimll": "x y z l m n ux uy uz num r0 z0 zmax zmin dphi coeff axial az cnum",
    "woltersecll": "x y z l m n ux uy uz num r0 z0 psi zmax zmin dphi coeff axial az cnum",
    "wsprimary": "x y z l m n ux uy uz num alpha z0 psi", "wssecondary": "x y z l m n ux uy uz num alpha z0 psi",
    "spocone": "x y z l m n ux uy uz num r0 tg",
    "ellipsoidwoltll": "x y z l m n ux uy uz num r0 z0 psi s zmax zmin dphi coeff axial az cnum",
    "wsprimaryback": "x y z l m n ux uy uz num alpha z0 psi thick", "wssecondaryback": "x y z l m n ux uy uz num alpha z0 psi thick",
    "tracezern": "x y z l m n ux uy uz num coeff rorder aorder arrsize rad",
    "tracezernopd": "opd x y z l m n ux uy uz num coeff rorder aorder arrsize rad nr",
    "zernphase": "opd x y z l m n ux uy uz num coeff rorder aorder arrsize rad wave",
    "tracezernrot": "x y z l m n ux uy uz num coeff1 rorder1 aorder1 arrsize1 coeff2 rorder2 aorder2 arrsize2 rad rot",
}
# routines whose device arithmetic is the reference's operation sequence bit for bit (DESIGN.md section 3)
BIT_EXACT = {"reflect", "transform", "itransform", "flat", "flatopd", "wolterprimary", "wolterprimaryopd", "woltersecondary", "conic",
             "conicopd", "spocone", "tracesphere", "tracesphereopd", "tracecyl", "tracecylopd", "cylconic", "paraxial", "paraxialy"}


@pytest.fixture(scope="module")
def fixture():
    return np.load(os.path.join(HERE, "golden", "f95_source.npz"))


def ray_cases(fx):
    tags = sorted({k.split("__")[0] for k in fx.files if k.startswith("c")})
    for tag in tags:
        _, module, name = tag.split("_", 2)
        extra = {k.split("__arg_")[1]: fx[k] for k in fx.files if k.startswith(tag + "__arg_")}
        extra = {k: (v if v.ndim else v.item()) for k, v in extra.items()}
        yield tag, module, name, [np.array(r) for r in fx[tag + "__in"]], [np.array(r) for r in fx[tag + "__out"]], extra


def f2py_args(name, rows, extra):
    return [extra[a] if a in extra else rows[ROWS.index(a)] for a in ARGS[name].split() if a not in HIDDEN]


def test_c_oracle_reproduces_the_fortran_source(fixture):
    n = 0
    for tag, module, name, rin, rout, extra in ray_cases(fixture):
        rows = [r.copy() for r in rin]
        getattr(getattr(of, module), name)(*f2py_args(name, rows, extra))
        assert_bit_equal(rows, rout, what=tag)
        n += 1
    assert n >= 53
    for tag in ("r00_reconstruct", "r01_reconstruct"):
        a, b, p = (np.asfortranarray(fixture[tag + "__" + k]) for k in ("xang", "yang", "phase"))
        pc = of.reconstruct.reconstruct(a, b, 1e-12, .5, p, int(fixture[tag + "__maxiter"]))
        assert np.array_equal(pc, fixture[tag + "__phasec_out"]) and np.array_equal(p, fixture[tag + "__phase_out"]), tag
    for tag, (xd, yd) in (("s00_southwellbin", (10, 8)), ("s01_southwellbin", (9, 7))):
        o = of.reconstruct.southwellbin(*(fixture[tag + "__" + k] for k in "xylm"), 1., xd, yd)
        for got, k in zip(o, ("xang_out", "yang_out", "phase_out")):
            assert np.array_equal(got, fixture[tag + "__" + k], equal_nan=True), tag


def test_c_oracle_special_functions_against_the_fortran_source(fixture):
    """specialFunctions.f95 called directly: legendre / legendrep (:337-388), radialpoly (:17-40), zernset (:142-234)."""
    fx = fixture
    for n in range(9):
        for i, x in enumerate(fx["sf_x"]):
            assert of.specialfunctions.legendre(x, n) == fx["sf_legendre"][n, i, 0]
            assert of.specialfunctions.legendrep(x, n) == fx["sf_legendre"][n, i, 1]
    for k, (n, m) in enumerate(fx["sf_nm"]):
        for i, rho in enumerate(fx["sf_rho"]):
            assert of.specialfunctions.radialpoly(rho, int(n), int(m)) == fx["sf_radialpoly"][k, i]
    for (rho, th), want in zip(fx["sf_zernset_args"], fx["sf_zernset"]):
        got = of.specialfunctions.zernset(rho, th, fx["sf_rorder"], fx["sf_aorder"])
        for u, v in zip(got, want):
            assert np.array_equal(u, v)


@pytest.mark.skipif(not refload.available(), reason="reference tree not present (GPU box)")
def test_translated_fortran_reproduces_the_fixture(fixture):
    """Re-run the translator on a third of the cases (the whole set takes a few minutes in Python)."""
    import make_f95_golden as mk
    files = {}
    for k, (tag, module, name, rin, rout, extra) in enumerate(ray_cases(fixture)):
        if k % 3 != 0:
            continue
        if module not in files:
            files[module] = f95run.load(os.path.join(mk.REF, module + ".f95"))
        units = f95run._parse_units(f95run._logical_lines(os.path.join(mk.REF, module + ".f95")))
        assert " ".join(units[name].args) == ARGS[name], name
        args, rows = mk.run_fortran(files[module], units[name].args, rin, extra)
        files[module][name](*args)
        assert_bit_equal([rows[r] for r in ROWS], rout, what=tag + " (translator)")


def test_translator_arithmetic_rules():
    """Known answers for the rules that make the translation gfortran's: literal kinds, promotion, integer division,
    powers by repeated multiplication, by-reference arguments, implicit typing, 1-based arrays."""
    import tempfile
    src = '''
subroutine kinds(a, b, c, d, e, n)
  real*8, intent(inout) :: a, b, c, d, e
  integer, intent(inout) :: n
  pi = 3.1415926535897931
  a = pi
  b = 1.e-10
  c = 7/2 + (-7)/2
  d = a**3
  e = 2.**0.5
  n = 2.9
end subroutine kinds

subroutine bump(v, k)
  real*8, intent(inout) :: v(3)
  integer, intent(in) :: k
  v(k) = v(k) + 1
end subroutine bump

subroutine caller(v, s)
  real*8, intent(inout) :: v(3), s
  integer :: i
  do i = 1, 3, 2
    call bump(v, i)
  end do
  call twice(s)
  call twice(v(2))
end subroutine caller

subroutine twice(t)
  real*8, intent(inout) :: t
  t = 2*t
end subroutine twice
'''
    with tempfile.NamedTemporaryFile("w", suffix=".f95", delete=False) as f:
        f.write(src)
    try:
        U = f95run.load(f.name)
    finally:
        os.unlink(f.name)
    a, b, c, d, e, n = U["kinds"](0., 0., 0., 0., 0., 0)
    pi32 = np.float64(np.float32(3.1415926535897931))
    assert a == pi32 and a != np.pi                                 # the literal is REAL*4, like the implicit variable
    assert b == np.float64(np.float32(1e-10))
    assert c == 0. and n == 2                                       # 7/2 = 3, (-7)/2 = -3; real -> integer truncates
    assert d == (pi32 * pi32) * pi32
    assert e == np.float64(np.float32(2.) ** np.float32(.5))        # REAL*4 ** REAL*4 is powf
    v = np.array([1., 2., 3.])
    v2, s = U["caller"](v, 5.)
    assert v.tolist() == [2., 4., 4.] and s == 10.                  # element and scalar arguments are written back
    assert f95run._powi(np.float64(1.1), 5) == (np.float64(1.1) * (np.float64(1.1) ** 2) ** 2)
    assert f95run._div(-7, 2) == -3 and f95run._div(np.float64(1.), 3) == np.float64(1.) / np.float64(3.)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_libpxf_reproduces_the_fortran_source(fixture):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyxfocus_b200 as pxf
    n = 0
    for tag, module, name, rin, rout, extra in ray_cases(fixture):
        dev = [torch.from_numpy(np.ascontiguousarray(r)).cuda() for r in rin]
        ex = {k: (torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).cuda()
                  if isinstance(v, np.ndarray) and v.dtype == np.float64 and v.shape == rin[1].shape else v) for k, v in extra.items()}
        getattr(getattr(pxf, module), name)(*f2py_args(name, dev, ex))
        got = [r.cpu().numpy() for r in dev]
        if name in BIT_EXACT:
            assert_bit_equal(got, rout, what=tag)
        else:
            scale = max(1., float(max(np.nanmax(np.abs(rout[k])) for k in (1, 2, 3))))
            assert_close(got, rout, pos_scale=scale, tol=1e-12, what=tag)
        n += 1
    assert n >= 53


def test_whole_reference_runs_here_and_equals_the_oracle_driven_reference():
    """All five BASELINE configurations at small sizes: the restatement (``oracle.refapi``) against the bits the
    reference ITSELF gave for them -- its unmodified Python layer over its unmodified Fortran text executed by
    oracle/f95run.py (``oracle.f95mods`` in the f2py slots) -- stored in tests/golden/reference_f95.npz: every ray
    row, surviving-index set and merit figure bit for bit.  Where the reference tree is present, the reference over its
    own Fortran and over the C oracle (how every golden fixture under tests/golden/ was produced) are run live and
    compared with the fixture as well."""
    from oracle import refapi
    from pyxfocus_b200 import examples as ex
    gold = np.load(os.path.join(HERE, "golden", "reference_f95.npz"))
    assert_pinned(rc.f95_runs(ex.make_api(refapi.load(), ex.NumpyXP, "refapi")), gold, what="refapi")
    if refload.available():
        from oracle import f95mods
        assert_pinned(rc.f95_runs(ex.make_api(refload.load(f2py_modules=f95mods.modules()), ex.NumpyXP,
                                              "reference over its own Fortran")), gold, what="reference over its Fortran")
        assert_pinned(rc.f95_runs(ex.make_api(refload.load(), ex.NumpyXP, "reference over the C oracle")), gold,
                      what="reference over the C oracle")


def test_translator_control_flow_and_precedence():
    """More rules of the translator: ** is right associative and binds tighter than unary minus, logical operators,
    zero-trip and negative-step do loops, do while / exit / cycle, recursive functions with a result variable, integer
    mod / sign, 2-D arrays in (row, column) order, ';'-separated statements and '&' continuations."""
    import tempfile
    src = '''
subroutine rules(out)
  implicit none
  real*8, intent(inout) :: out(12)
  integer :: i, k, grid(2,3)
  real*8 :: acc
  real*8 :: fact
  out(1) = 2**3**2
  out(2) = -2**2
  out(3) = 2*3 + 4*5 - &
           6/4
  k = 0
  do i = 5, 1
    k = k + 1
  end do
  out(4) = k
  k = 0
  do i = 10, 1, -3
    k = k + i
  end do
  out(5) = k
  k = 0 ; i = 0
  do while (.true.)
    i = i + 1
    if (i > 10) exit
    if (mod(i,2) == 0) cycle
    k = k + i
  end do
  out(6) = k
  out(7) = fact(5)
  out(8) = sign(3, -2) + mod(-7, 3)
  if (.not. (1 > 2) .and. (3 >= 3 .or. 1 == 2)) then
    out(9) = 1
  else
    out(9) = 0
  end if
  grid(2,3) = 7 ; grid(1,1) = 1
  out(10) = grid(2,3) - grid(1,1)
  acc = 1.d0/3
  out(11) = acc
  out(12) = 1./3
end subroutine rules

recursive function fact(n) result(f)
  implicit none
  integer, intent(in) :: n
  real*8 :: f
  real*8 :: fact
  if (n <= 1) then
    f = 1
    return
  end if
  f = n*fact(n-1)
end function fact
'''
    with tempfile.NamedTemporaryFile("w", suffix=".f95", delete=False) as f:
        f.write(src)
    try:
        U = f95run.load(f.name)
    finally:
        os.unlink(f.name)
    out = np.zeros(12)
    U["rules"](out)
    assert out[:10].tolist() == [512., -4., 25., 0., 22., 25., 120., -4., 1., 6.]
    assert out[10] == 1. / 3. and out[11] == np.float64(np.float32(1.) / np.float32(3.))
