"""Host-side code of conicplus, legsurf, zernphase and the rotated Zernike surface as fused-program ops (no GPU needed):
build_program accepts conicplus / legsurf alone and next to each of ops 27..36 and refuses every forbidden mix in both
orders, the row masks equal the stand-alone kernels' LOAD / STORE, the table fills refuse what the stand-alone routines
refuse, the rotated Zernike fill at rot = 0 is the plain fill of both sets, the codes Program records and its
refusals, the recorders' choice between recording and flushing, and the NVRTC compilation of programs holding every new
op."""
import ctypes
import struct

import numpy as np
import pytest

import pyxfocus_b200 as pxf
from pyxfocus_b200 import _lib
from pyxfocus_b200 import examples as ex
from pyxfocus_b200 import program as prg
from pyxfocus_b200 import surfaces as surf

OK, INVALID, UNSUPPORTED = 0, 1, 4
OP = pxf.program.OP
ALPHA = float(pxf.conicsolve.woltparam(220., 1.e4)[0])
ADDR = struct.unpack("d", struct.pack("Q", 4096))[0]          # a non-null device address (nothing is launched)

CONICPLUS = (OP["CONICPLUS"], [ADDR])
CONICPLUSOPD = (OP["CONICPLUSOPD"], [ADDR])
LEGSURF = (OP["LEGSURF"], [ADDR])
ZERNPHASE = (OP["ZERNPHASE"], [ADDR, 1e-6, 7.])
TAB_SURF = {"conicplus": CONICPLUS, "conicplusopd": CONICPLUSOPD, "legsurf": LEGSURF}
# ops 27..36, scalars as their stand-alone entry points take them
OLD_SURF = {
    "tracesphere": (OP["TRACESPHERE"], [250.]), "tracesphereopd": (OP["TRACESPHEREOPD"], [-500., 1.5]),
    "tracecyl": (OP["TRACECYL"], [100.]), "tracecylopd": (OP["TRACECYLOPD"], [100., 1.2]),
    "cylconic": (OP["CYLCONIC"], [1. / 400., -.7]), "paraxial": (OP["PARAXIAL"], [350.]),
    "paraxialy": (OP["PARAXIALY"], [-120.]), "torus": (OP["TORUS"], [150., 900.]),
    "wsprimaryback": (OP["WSPRIMARYBACK"], [ALPHA, 1.e4, 1., .4]),
    "wssecondaryback": (OP["WSSECONDARYBACK"], [ALPHA, 1.e4, 1., .4]),
}
ZERN = (OP["ZERNSURF"], [ADDR, 0., 7.])
LL = (OP["LLSURF"], [ADDR, 5.])
FAN = (OP["GRATFAN"], [1e-4, 1e4, 95., .01, -1., 1.])
ROTX = (OP["ROTX_REMAINING"], [1e-4, 3.])
TABLE_AUX = {"zern": ZERN, "ll": LL, "fan": FAN, "rotx": ROTX, "zernphase": ZERNPHASE}

R = {name: 1 << k for k, name in enumerate(["opd", "x", "y", "z", "l", "m", "n", "ux", "uy", "uz"])}
POS, DIR, NRM = R["x"] | R["y"] | R["z"], R["l"] | R["m"] | R["n"], R["ux"] | R["uy"] | R["uz"]
# (load, store) of each op alone: the LOAD / STORE of its stand-alone kernel (pxf_ops.cu)
MASKS = {
    OP["CONICPLUS"]: (POS | DIR, POS | NRM),
    OP["CONICPLUSOPD"]: (POS | DIR | R["opd"], POS | NRM | R["opd"]),
    OP["LEGSURF"]: (R["x"] | R["y"] | DIR, DIR),
    OP["ZERNPHASE"]: (R["x"] | R["y"] | DIR | R["opd"], DIR | R["opd"]),
}


def L():
    return _lib.lib()


def ops_of(seg_ops):
    nops = len(seg_ops[0])
    arr = (_lib.pxf_op * (len(seg_ops) * nops))()
    for s, ops in enumerate(seg_ops):
        for k, (code, p) in enumerate(ops):
            o = arr[s * nops + k]
            o.code = code
            for j, v in enumerate(p):
                o.p[j] = v
    return arr, nops


def trace_rc(ops):
    """build_program's verdict: pxf_trace_program validates the op list before it needs a device."""
    arr, nops = ops_of([ops])
    return L().pxf_trace_program((ctypes.c_void_p * 10)(), 0, arr, nops, None, None)


def zern_tables(nseg):
    ro, ao = (np.ascontiguousarray(v, dtype=np.int32) for v in ex.zernike_orders(7))
    per = int(L().pxf_zern_table_bytes())
    tabs = np.zeros(per * nseg, dtype=np.uint8)
    for s in range(nseg):
        c = ex.zernike_coeff(len(ro), rng_seed=s)
        assert L().pxf_zern_table_fill(c.ctypes.data, ro.ctypes.data, ao.ctypes.data, len(c), 60., 0, 0.,
                                       tabs[s * per:].ctypes.data) == 7
    return tabs


def seg_fill(seg_ops, zern=False):
    arr, nops = ops_of(seg_ops)
    nseg = len(seg_ops)
    start = np.zeros(nseg + 1, dtype=np.int64)
    start[1:] = np.cumsum([10] * nseg)
    if not zern:
        out = np.zeros(int(L().pxf_segmented_table_bytes(nops, nseg)), dtype=np.uint8)
        return L().pxf_segmented_table_fill(arr, nops, nseg, start.ctypes.data, out.ctypes.data), out
    out = np.zeros(int(L().pxf_segmented_table_bytes_zern(nops, nseg)), dtype=np.uint8)
    tabs = zern_tables(nseg)
    return L().pxf_segmented_table_fill_zern(arr, nops, nseg, start.ctypes.data, tabs.ctypes.data,
                                             out.ctypes.data), out


def header(out):
    load, store = out[:8].view(np.uint32)
    return int(load), int(store)


def chain(op):
    return [(OP["TRANSFORM"], [0., 0., 10., 0., 0., 0.]), op, (OP["REFRACT"], [1., 1.5]), (OP["FLATOPD"], [1.])]


# ---- build_program ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(TAB_SURF) + ["zernphase"])
def test_build_accepts_each_new_op(name):
    op = TAB_SURF.get(name, ZERNPHASE)
    for ops in ([op], chain(op), [(OP["FLAT"], [])] + [op]):
        assert trace_rc(ops) not in (INVALID, UNSUPPORTED), L().pxf_last_error()


@pytest.mark.parametrize("old", sorted(OLD_SURF))
@pytest.mark.parametrize("name", sorted(TAB_SURF))
def test_build_accepts_table_surface_next_to_each_scalar_surface(name, old):
    op, o = TAB_SURF[name], OLD_SURF[old]
    assert trace_rc([op, o]) not in (INVALID, UNSUPPORTED), L().pxf_last_error()
    assert trace_rc([o, op]) not in (INVALID, UNSUPPORTED), L().pxf_last_error()


def test_build_accepts_the_aspheric_singlet():
    singlet = [(OP["TRANSFORM"], [0., 0., 5., 0., 0., 0.]), (OP["TRACESPHERE"], [50.]), (OP["REFRACT"], [1., 1.5]),
               (OP["TRANSFORM"], [0., 0., 4., 0., 0., 0.]), CONICPLUS, (OP["REFRACT"], [1.5, 1.]),
               (OP["TRANSFORM"], [0., 0., 30., 0., 0., 0.]), (OP["FLAT"], [])]
    assert trace_rc(singlet) not in (INVALID, UNSUPPORTED), L().pxf_last_error()


@pytest.mark.parametrize("other", sorted(TABLE_AUX))
@pytest.mark.parametrize("name", sorted(TAB_SURF))
def test_build_refuses_table_surface_next_to_table_or_aux_ops(name, other):
    op, o = TAB_SURF[name], TABLE_AUX[other]
    assert trace_rc([op, o]) == UNSUPPORTED
    assert trace_rc([o, op]) == UNSUPPORTED
    assert trace_rc(chain(op)[:2] + [o] + chain(op)[2:]) == UNSUPPORTED


@pytest.mark.parametrize("other", sorted(set(TABLE_AUX) | set(TAB_SURF) | set(OLD_SURF)))
def test_build_refuses_zernphase_next_to_another_table_a_fan_or_a_surface(other):
    o = dict(TABLE_AUX, **TAB_SURF, **OLD_SURF)[other]
    assert trace_rc([ZERNPHASE, o]) == UNSUPPORTED
    assert trace_rc([o, ZERNPHASE]) == UNSUPPORTED
    assert trace_rc(chain(ZERNPHASE)[:2] + [o] + chain(ZERNPHASE)[2:]) == UNSUPPORTED


def test_build_refuses_zernphase_above_order_7_and_null_tables():
    assert trace_rc([(OP["ZERNPHASE"], [ADDR, 1e-6, 8.])]) == UNSUPPORTED
    for code in (OP["ZERNPHASE"], OP["CONICPLUS"], OP["CONICPLUSOPD"], OP["LEGSURF"]):
        assert trace_rc([(code, [0., 1e-6, 7.])]) == INVALID


# ---- liveness -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("code", sorted(MASKS))
def test_row_masks_are_the_stand_alone_load_store(code):
    op = (code, [ADDR, 1e-6, 7.])
    rc, out = seg_fill([[op], [op]], zern=code == OP["ZERNPHASE"])
    assert rc == OK, L().pxf_last_error()
    assert header(out) == MASKS[code]


# ---- table fills --------------------------------------------------------------------------------------------------
def conicplus_fill(p, opd=0, nr=0.):
    p = np.ascontiguousarray(p, dtype=np.float64)
    out = np.zeros(int(L().pxf_conicplus_table_bytes()), dtype=np.uint8)
    return L().pxf_conicplus_table_fill(40., -1.2, p.ctypes.data, len(p), opd, nr, out.ctypes.data), out


def legsurf_fill(coeff, xo, yo):
    c = np.ascontiguousarray(coeff, dtype=np.float64)
    a, b = np.ascontiguousarray(xo, dtype=np.int32), np.ascontiguousarray(yo, dtype=np.int32)
    out = np.zeros(int(L().pxf_legsurf_table_bytes()), dtype=np.uint8)
    return L().pxf_legsurf_table_fill(10., 12., 1e-3, c.ctypes.data, a.ctypes.data, b.ctypes.data, len(c),
                                      out.ctypes.data), out


def test_conicplus_fill_takes_0_to_16_terms():
    nb = int(L().pxf_conicplus_table_bytes())
    assert nb == 192
    for n in (0, 1, 8, 16):
        rc, out = conicplus_fill(np.linspace(1e-6, 1e-9, n))
        assert rc == nb
    assert conicplus_fill(np.ones(17))[0] == -1
    assert b"polynomial terms" in L().pxf_last_error()
    # the folded block: c = 1/R, ..., nr, tol, np, opd, p[]
    rc, out = conicplus_fill([1e-6, 2e-9], opd=1, nr=1.5)
    d = out.view(np.float64)
    assert d[0] == 1. / 40. and d[5] == 1.5 and list(out[56:64].view(np.int32)) == [2, 1]
    assert d[8] == 1e-6 and d[9] == 2e-9 and not d[10:].any()


def test_legsurf_fill_takes_0_to_48_terms_of_orders_0_to_15():
    nb = int(L().pxf_legsurf_table_bytes())
    for n in (0, 1, 48):
        assert legsurf_fill(np.ones(n), np.arange(n) % 16, (np.arange(n) * 7) % 16)[0] == nb
    assert legsurf_fill(np.ones(49), np.zeros(49), np.zeros(49))[0] == -1
    assert legsurf_fill([1.], [16], [0])[0] == -1
    assert legsurf_fill([1.], [0], [16])[0] == -1
    assert legsurf_fill([1.], [-1], [0])[0] == -1


def zern_fill(c, r, a, rad=60.):
    c, r, a = (np.ascontiguousarray(v, dtype=t) for v, t in ((c, np.float64), (r, np.int32), (a, np.int32)))
    out = np.zeros(int(L().pxf_zern_table_bytes()), dtype=np.uint8)
    return L().pxf_zern_table_fill(c.ctypes.data, r.ctypes.data, a.ctypes.data, len(c), rad, 0, 0., out.ctypes.data), out


def zern_fill_rot(t1, t2, rot, rad=60.):
    (c1, r1, a1), (c2, r2, a2) = ((np.ascontiguousarray(v, dtype=t) for v, t in zip(s, (np.float64, np.int32, np.int32)))
                                  for s in (t1, t2))
    out = np.zeros(int(L().pxf_zern_table_bytes()), dtype=np.uint8)
    return L().pxf_zern_table_fill_rot(c1.ctypes.data, r1.ctypes.data, a1.ctypes.data, len(c1), c2.ctypes.data,
                                       r2.ctypes.data, a2.ctypes.data, len(c2), rad, rot, out.ctypes.data), out


def test_rotated_fill_at_rot_0_is_the_plain_fill_of_both_sets():
    ro, ao = ex.zernike_orders(7)
    n = len(ro)
    c1, c2 = ex.zernike_coeff(n, rng_seed=1), ex.zernike_coeff(n, rng_seed=2)
    # both fills accept these sets: each set alone sizes the reference's tables for order 7
    h = n // 2
    for (s1, s2) in (((c1, ro, ao), (c2, ro, ao)), ((c1, ro, ao), (c2[:h + 8], ro[:h + 8], ao[:h + 8]))):
        rc_rot, rot0 = zern_fill_rot(s1, s2, 0.)
        rc, cat = zern_fill(*(np.concatenate([x, y]) for x, y in zip(s1, s2)))
        assert rc_rot == rc == 7
        assert np.array_equal(rot0, cat)
    rc, rot = zern_fill_rot((c1, ro, ao), (c2, ro, ao), .3)
    assert rc == 7 and not np.array_equal(rot, zern_fill_rot((c1, ro, ao), (c2, ro, ao), 0.)[1])
    assert zern_fill_rot((c1, ro, ao), ([1.], [3], [2]), .3)[0] == -1           # n - |m| odd


# ---- segmented fills ----------------------------------------------------------------------------------------------
def seg_ops_table(out, nops, nseg):
    off = 48 + (-(-(nseg + 1) * 8 // 16)) * 16
    raw = out[off:off + nseg * nops * 312]
    rec = np.frombuffer(raw.tobytes(), dtype=np.dtype([("code", "<i4"), ("row", "<i4"), ("q", "<f8", 38)]))
    return rec.reshape(nseg, nops)


def test_plain_fill_carries_each_segments_table_address():
    addrs = [4096 * (s + 1) for s in range(3)]
    seg_ops = [[(OP["TRACESPHERE"], [50.]), (OP["CONICPLUSOPD"], [struct.unpack("d", struct.pack("Q", a))[0]]),
                (OP["LEGSURF"], [struct.unpack("d", struct.pack("Q", 2 * a))[0]])] for a in addrs]
    rc, out = seg_fill(seg_ops)
    assert rc == OK, L().pxf_last_error()
    t = seg_ops_table(out, 3, 3)
    for s, a in enumerate(addrs):
        assert int(t[s, 1]["q"][:1].view(np.uint64)[0]) == a and int(t[s, 2]["q"][:1].view(np.uint64)[0]) == 2 * a


@pytest.mark.parametrize("name", sorted(TAB_SURF))
def test_zern_fill_refuses_table_surfaces(name):
    rc, _ = seg_fill([chain(TAB_SURF[name])] * 2, zern=True)
    assert rc == UNSUPPORTED


def test_zern_fill_takes_zernphase_with_its_own_wave_and_refuses_mixed_kinds():
    rc, out = seg_fill([chain((OP["ZERNPHASE"], [ADDR, w, 7.])) for w in (1e-6, 2e-6)], zern=True)
    assert rc == OK, L().pxf_last_error()
    t = seg_ops_table(out, 4, 2)
    assert t[0, 1]["q"][0] == 1e-6 and t[1, 1]["q"][0] == 2e-6
    rc, _ = seg_fill([chain(ZERNPHASE), chain(ZERN)], zern=True)
    assert rc == INVALID
    rc, _ = seg_fill([chain(ZERNPHASE)] * 2)             # the plain fill has no Zernike tables
    assert rc == UNSUPPORTED


# ---- Program ------------------------------------------------------------------------------------------------------
def zern_terms():
    ro, ao = ex.zernike_orders(7)
    return ex.zernike_coeff(len(ro)), ro, ao


def test_program_methods_record_the_codes():
    c, ro, ao = zern_terms()
    p = (pxf.Program().tracesphere(50.).conicplus(40., -1.2, [1e-6] * 8).conicplusopd(40., -1.2, [], 1.5)
         .legsurf(10., 12., 1e-3, [1., 2.], [1, 2], [0, 3]))
    assert [code for code, _ in p.ops] == [OP["TRACESPHERE"], OP["CONICPLUS"], OP["CONICPLUSOPD"], OP["LEGSURF"]]
    assert sorted(p._tables) == [1, 2, 3] and p.can_hold_surface()
    z = pxf.Program().flat().zernphase(c, ro, ao, 60., 1e-6)
    assert z.ops[-1] == (OP["ZERNPHASE"], [0., 1e-6, 7.]) and 1 in z._tables
    r = pxf.Program().tracezernrot(c, ro, ao, c[:10], ro[:10], ao[:10], 60., .3)
    assert r.ops[-1] == (OP["ZERNSURF"], [0., 0., 7.])
    tab = r._tables[0].numpy()
    assert np.array_equal(tab, zern_fill_rot((c, ro, ao), (c[:10], ro[:10], ao[:10]), .3)[1])


def test_program_refusals():
    c, ro, ao = zern_terms()
    ax, az = ex.ll_orders(3)
    lc = ex.ll_coeff(16)
    P = pxf.Program
    holders = [lambda p: p.zernsurf(c, ro, ao, 62.5), lambda p: p.zernphase(c, ro, ao, 62.5, 1e-6),
               lambda p: p.wolterprimll(220., 8400., 8500., 8400., .25, lc, ax, az),
               lambda p: p.gratfan(1e-4, 1e4, 95., .01, -1., 1.), lambda p: p.rotx_remaining(1e-4, 3)]
    tables = [lambda p: p.conicplus(40., -1.2, [1e-6]), lambda p: p.conicplusopd(40., -1.2, [1e-6], 1.5),
              lambda p: p.legsurf(10., 12., 1e-3, [1.], [1], [0])]
    for hold in holders:
        for add in tables:
            with pytest.raises(NotImplementedError):
                add(hold(P()))
            with pytest.raises(NotImplementedError):
                hold(add(P()))
    for hold in holders:
        with pytest.raises(NotImplementedError):
            hold(P().zernphase(c, ro, ao, 62.5, 1e-6))
        with pytest.raises(NotImplementedError):
            hold(P()).zernphase(c, ro, ao, 62.5, 1e-6)
    for old in ("tracesphere", "torus"):
        with pytest.raises(NotImplementedError):
            getattr(P(), old)(*OLD_SURF[old][1]).zernphase(c, ro, ao, 62.5, 1e-6)
        with pytest.raises(NotImplementedError):
            getattr(P().zernphase(c, ro, ao, 62.5, 1e-6), old)(*OLD_SURF[old][1])
    ro8, ao8 = ex.zernike_orders(8)
    with pytest.raises(NotImplementedError):
        P().zernphase(ex.zernike_coeff(len(ro8)), ro8, ao8, 62.5, 1e-6)
    with pytest.raises(NotImplementedError):
        P().tracezernrot(c, ro, ao, ex.zernike_coeff(len(ro8)), ro8, ao8, 62.5, .1)
    with pytest.raises(ValueError):
        P().conicplus(40., -1.2, np.ones(17))
    with pytest.raises(ValueError):
        P().legsurf(10., 12., 1e-3, np.ones(49), np.zeros(49), np.zeros(49))


# ---- recorders ----------------------------------------------------------------------------------------------------
class FakeRays(list):
    """Ten placeholder rows: the recorders never touch them while they record."""


@pytest.fixture
def recording(monkeypatch):
    """A recording program for a fake bundle; flushes are counted instead of run."""
    rays = FakeRays([None] * 10)
    prog = pxf.Program()
    monkeypatch.setitem(prg._active, id(rays), (rays, prog))
    flushed = []

    def fake_flush(r):
        flushed.append(True)
        raise _Flushed()
    monkeypatch.setattr(surf, "flush", fake_flush)
    return rays, prog, flushed


class _Flushed(Exception):
    pass


def test_recorders_record_into_a_program_that_can_hold_them(recording):
    rays, prog, flushed = recording
    c, ro, ao = zern_terms()
    surf.sphere(rays, 50.)
    surf.conicplus(rays, 40., -1.2, [1e-6] * 8)
    surf.conicplus(rays, 40., -1.2, [1e-6] * 8, nr=1.5)
    surf.legSurf(rays, 10., 12., 1e-3, [1., 2.], [1, 2], [0, 3])
    assert [code for code, _ in prog.ops] == [OP["TRACESPHERE"], OP["CONICPLUS"], OP["CONICPLUSOPD"], OP["LEGSURF"]]
    prog.ops, prog._tables = [], {}
    surf.zernphase(rays, c, 60., 1e-6, ro, ao)
    assert [code for code, _ in prog.ops] == [OP["ZERNPHASE"]]
    prog.ops, prog._tables = [], {}
    surf.zernsurfrot(rays, c, c, 60., .3, ro, ao, ro, ao)
    assert [code for code, _ in prog.ops] == [OP["ZERNSURF"]]
    assert not flushed


def test_recorders_flush_where_they_must(recording):
    rays, prog, flushed = recording
    c, ro, ao = zern_terms()
    ro8, ao8 = ex.zernike_orders(8)
    c8 = ex.zernike_coeff(len(ro8))
    cases = [
        ([], lambda: surf.zernphase(rays, c8, 60., 1e-6, ro8, ao8)),                    # radial order above 7
        ([], lambda: surf.zernsurfrot(rays, c, c8, 60., .3, ro, ao, ro8, ao8)),
        ([], lambda: surf.conicplus(rays, 40., -1.2, np.ones(17))),                     # the routine's own refusal
        ([], lambda: surf.legSurf(rays, 10., 12., 1e-3, np.ones(49), np.zeros(49), np.zeros(49))),
        ([ZERN], lambda: surf.conicplus(rays, 40., -1.2, [1e-6])),                      # forbidden mixes
        ([ZERNPHASE], lambda: surf.legSurf(rays, 10., 12., 1e-3, [1.], [1], [0])),
        ([LL], lambda: surf.zernphase(rays, c, 60., 1e-6, ro, ao)),
        ([ZERN], lambda: surf.zernphase(rays, c, 60., 1e-6, ro, ao)),
        ([OLD_SURF["torus"]], lambda: surf.zernphase(rays, c, 60., 1e-6, ro, ao)),
        ([CONICPLUS], lambda: surf.zernphase(rays, c, 60., 1e-6, ro, ao)),
        ([ZERNPHASE], lambda: surf.zernsurfrot(rays, c, c, 60., .3, ro, ao, ro, ao)),
        ([CONICPLUS], lambda: surf.zernsurfrot(rays, c, c, 60., .3, ro, ao, ro, ao)),
        ([ZERNPHASE], lambda: surf.zernsurf(rays, c, 60., ro, ao)),
        ([LEGSURF], lambda: surf.zernsurf(rays, c, 60., ro, ao)),
        ([ZERNPHASE], lambda: surf.primaryLL(rays, 220., 8400., 8500., 8400., .25, ex.ll_coeff(16),
                                             *ex.ll_orders(3))),
        ([CONICPLUSOPD], lambda: surf.primaryLL(rays, 220., 8400., 8500., 8400., .25, ex.ll_coeff(16),
                                                *ex.ll_orders(3))),
    ]
    for held, call in cases:
        prog.ops = [(code, list(p)) for code, p in held]
        n = len(flushed)
        with pytest.raises(_Flushed):
            call()
        assert len(flushed) == n + 1 and len(prog.ops) == len(held)


# ---- NVRTC --------------------------------------------------------------------------------------------------------
def test_programs_with_every_new_op_compile_for_both_forms():
    """The specialised kernels of programs holding every new op, single and segmented, compile (NVRTC; no device
    needed).  ZERNPHASE shares no program with the others, so it has a program of its own."""
    c, ro, ao = zern_terms()
    surfaces = (pxf.Program().transform(0, 0, 5, 0, 0, 0).tracesphere(50.).refract(1., 1.5)
                .conicplus(40., -1.2, [1e-6] * 8).refract(1.5, 1.).conicplusopd(40., -1.2, [1e-6], 1.5).flat()
                .legsurf(10., 12., 1e-3, [1., 2.], [1, 2], [0, 3]))
    phase = pxf.Program().flat().zernphase(c, ro, ao, 60., 1e-6).transform(0, 0, 5, 0, 0, 0).flatopd(1.)
    rot = (pxf.Program().transform(0, 0, 5, 0, 0, 0).tracezernrot(c, ro, ao, c, ro, ao, 60., .3).reflect()
           .flat())
    if surfaces.precompile() == 0:
        pytest.skip("NVRTC unavailable: " + L().pxf_jit_status().decode())
    for p in (surfaces, phase, rot):
        assert p.precompile() > 0, L().pxf_jit_status()
        assert p.precompile(segmented=True) > 0, L().pxf_jit_status()
