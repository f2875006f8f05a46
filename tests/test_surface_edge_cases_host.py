"""The edge bundles of tests/surface_edge_cases.py on the C oracle (no GPU needed): every class a bundle claims is
really there in the oracle's output -- ties between the roots, zero discriminants, misses (zeroed, NaN normal), zero
outputs of both signs, Inf and NaN, Legendre arguments at exactly +-1, Newton iterations that stop at the
1000-iteration cap (a numpy replay counts them) -- and the entry points refuse tables they cannot hold before they
look for a device."""
import ctypes

import numpy as np
import pytest

import surface_edge_cases as E
from pyxfocus_b200 import _lib

INVALID = 1


def run(name):
    case = E.CASES[name]
    rows, classes = E.bundle(name)
    out = [np.array(r, copy=True) for r in rows]
    E.oracle(case, out)
    return case, rows, out, classes


def sel(rows, idx):
    return [r[idx] for r in rows]


def is_miss(out, idx, nan_rows=(7, 8, 9)):
    o = sel(out, idx)
    zeroed = np.all([o[k] == 0. for k in range(1, 7)], axis=0)
    return zeroed & np.all([np.isnan(o[k]) for k in nan_rows], axis=0)


def all_classes_of(name, classes, want):
    assert set(want) <= set(classes), (name, sorted(classes))
    for c in want:
        assert classes[c].size > 0, (name, c)


def test_every_case_has_n_rays_and_an_edge_ray_in_the_tail():
    for name in E.CASES:
        rows, classes = E.bundle(name)
        assert len(rows) == 10 and all(r.shape == (E.N,) and r.flags.c_contiguous for r in rows), name
        if classes:
            assert any((E.N - 1) in v for v in classes.values()), name
    # every routine, both signs of the radius, opd variants, special-value variants
    routines = {c.routine for c in E.CASES.values()}
    assert routines == {"tracesphere", "tracesphereopd", "tracecyl", "tracecylopd", "cylconic", "paraxial", "paraxialy",
                        "torus", "conicplus", "conicplusopd", "legsurf", "wsprimaryback", "wssecondaryback"}
    assert {c.routine for c in E.CASES.values() if c.special} == routines - {"wsprimaryback", "wssecondaryback"}


@pytest.mark.parametrize("name", ["tracesphere_Rp", "tracesphere_Rm", "tracesphereopd_Rp", "tracesphereopd_Rm"])
def test_sphere_classes(name):
    case, inp, out, cl = run(name)
    all_classes_of(name, cl, ["dotol0", "det0", "grazing_miss", "centre", "origin", "origin_nodir", "inside"])
    opd, x, y, z, l, m, n = inp[:7]
    R = case.args[0]
    dotol = l * x + m * y + n * z
    mago = x * x + y * y + z * z
    det = dotol * dotol - mago + R * R
    # equal-magnitude roots: the tie keeps d1 = +sqrt(det), the ray moves forward along its direction
    i = cl["dotol0"]
    assert np.all(dotol[i] == 0.) and np.all(det[i] > 0.)
    d1 = np.sqrt(det[i])
    assert np.array_equal(out[1][i], x[i] + d1 * l[i]) and np.array_equal(out[3][i], z[i] + d1 * n[i])
    assert np.all(det[cl["det0"]] == 0.) and not is_miss(out, cl["det0"]).any()
    assert np.all(det[cl["grazing_miss"]] < 0.) and np.all(det[cl["grazing_miss"]] > -1e-10)
    assert is_miss(out, cl["grazing_miss"]).all()
    assert np.all(mago[cl["inside"]] < R * R)
    assert not is_miss(out, cl["centre"]).any()
    # at the origin with no direction the ray stays there: the normal is 0/0
    i = cl["origin_nodir"]
    assert np.all(out[1][i] == 0.) and np.all(np.isnan(out[7][i]))
    # ordinary rays miss too, and the zeros of the misses carry both signs of the input's -0 nowhere
    assert 0 < int(np.isnan(out[7]).sum()) < E.N
    if case.opd:
        i = cl["dotol0"]
        assert np.array_equal(out[0][i], opd[i] + d1 * case.args[1])


@pytest.mark.parametrize("name", ["tracecyl_Rp", "tracecyl_Rm", "tracecylopd_Rp", "tracecylopd_Rm"])
def test_cylinder_classes(name):
    case, inp, out, cl = run(name)
    all_classes_of(name, cl, ["b0", "det0", "grazing_miss", "axial", "on_axis", "inside"])
    x, y, z, l, m, n = inp[1:7]
    R = case.args[0]
    a = l * l + n * n
    b = 2 * (x * l + z * n)
    c = x * x + z * z - R * R
    det = b * b - 4 * a * c
    assert np.all(b[cl["b0"]] == 0.) and np.all(det[cl["b0"]] > 0.)
    assert np.all(det[cl["det0"]] == 0.)
    # a miss: zeroed, the normal 0/0 in x and z (uy is set to 0)
    assert np.all(det[cl["grazing_miss"]] < 0.) and is_miss(out, cl["grazing_miss"], (7, 9)).all()
    assert np.all(out[8][cl["grazing_miss"]] == 0.)
    # parallel to the axis: a = 0, det = 0, the distance is 0/0
    i = cl["axial"]
    assert np.all(a[i] == 0.) and np.all(np.isnan(out[1][i])) and np.all(np.isnan(out[3][i]))
    assert np.all(x[cl["on_axis"]] == 0.) and np.all(z[cl["on_axis"]] == 0.)
    # the tangent rays along y (a = 0 on the circle) are NaN, the others hit
    assert np.isnan(out[1][cl["det0"]]).any() and np.isfinite(out[1][cl["det0"]]).any()
    assert np.all(c[cl["inside"]] < 0.)


@pytest.mark.parametrize("name", ["cylconic_Km1", "cylconic_Km3", "cylconic_K0", "cylconic_K2"])
def test_cylconic_classes_and_cap(name):
    case, inp, out, cl = run(name)
    rad, K = case.args
    assert cl["fp0"].size
    i = cl["fp0"]
    assert np.all(inp[1][i] == 0.) and np.all(inp[5][i] == 0.) and np.all(inp[2][i] != 0.)
    assert not np.isfinite(out[1][i]).any()               # delt = -F/0
    if K > -1:
        i = cl["root_nan"]
        assert np.all(1 - (1 + K) * rad * rad * inp[1][i] ** 2 < 0.) and np.all(np.isnan(out[1][i]))
    else:
        its = E.replay(case, inp)
        assert np.all(its[cl["cap"]] == E.NEWTON_CAP), np.bincount(its[cl["cap"]])[-5:]
        assert np.all(np.isfinite(out[1][cl["cap"]]))
        # the ordinary rays converge well before the cap
        ordinary = np.setdiff1d(np.arange(E.N), np.concatenate(list(cl.values())))
        assert np.median(its[ordinary]) < 10


@pytest.mark.parametrize("name", ["torus_in_lt_out", "torus_in_gt_out"])
def test_torus_classes_and_cap(name):
    case, inp, out, cl = run(name)
    rin, rout = case.args
    i = cl["on_axis"]
    assert np.all(inp[1][i] == 0.) and np.all(inp[2][i] == 0.)
    assert np.all(np.isnan(out[7][i]))                 # Fx = Fy = 0: the normal's length is 0
    its = E.replay(case, inp)
    assert np.all(its[cl["cap"]] == E.NEWTON_CAP), np.bincount(its[cl["cap"]])[-5:]
    assert np.all(np.abs(inp[1][cl["cap"]]) > rin)
    ordinary = np.setdiff1d(np.arange(E.N), np.concatenate(list(cl.values())))
    assert np.median(its[ordinary]) < 10 and np.isfinite(out[1][ordinary]).all()


@pytest.mark.parametrize("name", ["conicplus_0_Rm_Km1", "conicplusopd_0_Rm_Km1", "conicplus_1", "conicplusopd_1",
                                  "conicplus_3_rootnan", "conicplusopd_3_rootnan", "conicplus_16_Km1",
                                  "conicplusopd_16_Km1"])
def test_conicplus_classes_and_cap(name):
    case, inp, out, cl = run(name)
    R, K, p = case.args[:3]
    assert len(p) in (0, 1, 3, 16)
    i = cl["on_axis"]
    assert np.all(np.isnan(out[1][i])) and np.all(np.isnan(out[7][i]))      # rad = 0: Fx = Fr * 0 / 0
    if "root_nan" in cl:
        i = cl["root_nan"]
        r2 = inp[1][i] ** 2 + inp[2][i] ** 2
        assert np.all(1 - (K + 1) / R ** 2 * r2 < 0.) and np.all(np.isnan(out[1][i]))
    if "cap" in cl:
        its = E.replay(case, inp)
        assert np.all(its[cl["cap"]] == E.NEWTON_CAP), np.bincount(its[cl["cap"]])[-5:]
        assert np.all(np.isfinite(out[1][cl["cap"]]))
        if case.opd:
            assert np.all(np.isfinite(out[0][cl["cap"]])) and np.all(out[0][cl["cap"]] != inp[0][cl["cap"]])
    ordinary = np.setdiff1d(np.arange(E.N), np.concatenate(list(cl.values())))
    assert np.isfinite(out[3][ordinary]).mean() > .99


def test_conicplus_covers_the_term_counts():
    counts = {len(c.args[2]) for c in E.CASES.values() if c.routine.startswith("conicplus")}
    assert counts == {0, 1, 3, 16}
    assert any(c.args[0] < 0 and c.args[1] == -1. for c in E.CASES.values() if c.routine == "conicplus")


@pytest.mark.parametrize("name", ["legsurf_0", "legsurf_5", "legsurf_48"])
def test_legsurf_classes(name):
    case, inp, out, cl = run(name)
    xw, yw, order, coeff, xo, yo = case.args
    xx, yy = inp[1] / xw, inp[2] / yw
    i = cl["width_edge"]
    for v in (xx[i], yy[i]):
        assert np.any(v == 1.) and np.any(v == -1.)
        assert np.any((v == 0.) & ~np.signbit(v)) and np.any((v == 0.) & np.signbit(v))
        assert np.any((np.abs(v) < 1.) & (np.abs(v) > 1. - 1e-15))
        assert np.any((np.abs(v) > 1.) & (np.abs(v) < 1. + 1e-15))
    # n = +-0: n / |n| is 0/0
    assert np.all(np.isnan(out[6][cl["n_zero"]]))
    if len(coeff):
        # orders: every one of 0..15 on both axes for the 48-term table
        if len(coeff) == 48:
            assert set(xo) == set(yo) == set(range(16))
        # the kick pushes part of the steep rays beyond l**2 + m**2 = 1
        i = cl["steep"]
        before = inp[4][i] ** 2 + inp[5][i] ** 2
        after = out[4][i] ** 2 + out[5][i] ** 2
        assert np.all(before <= 1.) and np.any(after > 1.) and np.all(np.isnan(out[6][i][after > 1.]))
        # the x == 0 / even order guard of legendrep decides finite outputs at x = +-0
        x0 = cl["width_edge"][xx[cl["width_edge"]] == 0.]
        assert x0.size and np.all(np.isfinite(out[4][x0]))
    else:
        assert np.array_equal(out[4], inp[4]) and np.array_equal(out[5], inp[5])


# rows each routine writes
WRITTEN = {"paraxial": [4, 5], "paraxialy": [5], "legsurf": [4, 5, 6]}


@pytest.mark.parametrize("name", sorted(n for n in E.CASES if E.CASES[n].special))
def test_special_value_variants(name):
    """the specials reach the rows the routine writes: zeros of both signs, Inf and NaN (conicplus turns every
    non-finite input into NaN: rad = sqrt(Inf) feeds Inf - Inf; legsurf's n = n/|n|*sqrt(..) only gives -0 from a -0
    square root, which no salted ray produces)"""
    case, inp, out, cl = run(name)
    rows = WRITTEN.get(case.routine, [1, 2, 3, 7, 8, 9]) + ([0] if case.opd else [])
    allw = np.concatenate([out[k] for k in rows])
    assert np.any((allw == 0.) & ~np.signbit(allw))
    assert np.any((allw == 0.) & np.signbit(allw)) or case.routine == "legsurf"
    assert np.any(np.isnan(allw))
    assert np.any(np.isinf(allw)) or (case.routine == "conicplus")
    assert np.isfinite(allw).mean() > .3


@pytest.mark.parametrize("name", [n for n in E.CASES if n.startswith("paraxial")])
def test_paraxial_zero_and_huge_focal_lengths(name):
    case, inp, out, cl = run(name)
    F = case.args[0]
    k = 5
    if case.routine == "paraxial":
        assert np.array_equal(out[4], inp[4] - inp[1] / F, equal_nan=True)
    assert np.array_equal(out[k], inp[k] - inp[2] / F, equal_nan=True)
    if F == 0.:
        i = cl["zero_xy"]
        assert np.all(np.isnan(out[k][i])) and np.all(np.isinf(out[k][np.abs(inp[2]) > 0.]))


@pytest.mark.parametrize("arcmin", [0., 5., 10., 15.])
def test_ws_bundles_are_inside_the_graze_angle(arcmin):
    for r in ("wsprimaryback", "wssecondaryback"):
        case, inp, out, _ = run("%s_%d" % (r, arcmin))
        assert case.args[3] == E.WS_THICK
        moved = (out[1] != inp[1]) | (out[3] != inp[3])
        assert moved.mean() > .9, (r, arcmin, moved.mean())
        assert np.isfinite(out[7][moved]).all()


def test_segment_and_host_sources():
    rows, cl = E.seg_bundle("sphere")
    assert rows[1].shape[0] == sum(E.LAYOUT)
    start = np.concatenate([[0], np.cumsum(E.LAYOUT)])
    E.seg_oracle("sphere", rows)
    for k in range(len(E.LAYOUT)):
        a, b = start[k], start[k + 1]
        miss = np.isnan(rows[7][a:b])
        if E.seg_sphere_scalars(k)[0] == 1e-3 and b > a:
            assert miss.all(), k                       # a segment in which every ray misses
    rows, cl = E.seg_bundle("torus")
    assert cl["cap"].size > 100
    its = E.replay(E.CASES["torus_in_lt_out"], rows)
    assert np.all(its[cl["cap"]] == E.NEWTON_CAP)
    assert any(np.signbit(E.seg_paraxial_scalars(k)[0]) and E.seg_paraxial_scalars(k)[0] == 0.
               for k in range(len(E.LAYOUT)))


# ------------------------------------------------------------------ refusals that need no device
NULL9 = [None] * 9


def test_conicplus_refuses_more_than_16_terms():
    L = _lib.lib()
    for fn, extra in (("pxf_conicplus", []), ("pxf_conicplusopd", [1.1])):
        for np_, ok in ((17, False), (64, False), (-1, False)):
            p = np.zeros(max(np_, 1))
            args = ([None] * (10 if "opd" in fn else 9)) + [0, 800., -1., p.ctypes.data, np_]
            rc = getattr(L, fn)(*args, *extra, None, None)
            assert rc == INVALID, (fn, np_, rc)
            assert b"polynomial terms" in L.pxf_last_error()


@pytest.mark.parametrize("nc,xo,yo", [(49, 0, 0), (3, 16, 0), (3, 0, 16), (3, -1, 0), (3, 0, -1), (-1, 0, 0)])
def test_legsurf_refuses_bad_tables(nc, xo, yo):
    L = _lib.lib()
    n = max(nc, 1)
    coeff = np.ones(n)
    a = np.zeros(n, np.int32)
    b = np.zeros(n, np.int32)
    a[-1], b[-1] = xo, yo
    rc = L.pxf_legsurf(*NULL9, 0, 2., 30., 2., coeff.ctypes.data, a.ctypes.data, b.ctypes.data, nc, None, None)
    assert rc == INVALID
    assert b"legsurf" in L.pxf_last_error()


def test_legsurf_and_conicplus_accept_the_limits():
    """48 terms of order 15 and 16 polynomial terms pass the checks (and then need a device)"""
    L = _lib.lib()
    coeff = np.ones(48)
    o = np.full(48, 15, np.int32)
    rc = L.pxf_legsurf(*NULL9, 0, 2., 30., 2., coeff.ctypes.data, o.ctypes.data, o.ctypes.data, 48, None, None)
    assert rc != INVALID, L.pxf_last_error()
    p = np.zeros(16)
    rc = L.pxf_conicplus(*NULL9, 0, 800., -1., p.ctypes.data, 16, None, None)
    assert rc != INVALID, L.pxf_last_error()


def test_library_cap_matches_the_oracle():
    assert _lib.lib().pxf_newton_cap() == E.NEWTON_CAP
    assert ctypes.sizeof(ctypes.c_double) == 8
