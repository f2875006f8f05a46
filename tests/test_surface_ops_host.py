"""Host-side code of the remaining scalar surfaces as fused-program ops (no GPU needed): build_program accepts each new
opcode and refuses it next to a Zernike surface, an LL shell or a grating fan in either order, the segmented fills
(plain: accepted, with each segment's own folded scalars and the stand-alone routines' row masks; _zern / _ll:
refused), the codes and scalars Program records and its refusals, and the NVRTC compilation of a program holding all
ten ops."""
import ctypes
import struct

import numpy as np
import pytest

import pyxfocus_b200 as pxf
from pyxfocus_b200 import _lib
from pyxfocus_b200 import examples as ex

OK, INVALID, UNSUPPORTED = 0, 1, 4
OP = pxf.program.OP
ALPHA = float(pxf.conicsolve.woltparam(220., 1.e4)[0])

# (code, scalars) of each new op, scalars as the stand-alone entry point takes them
NEW = [
    (OP["TRACESPHERE"], [250.]),
    (OP["TRACESPHEREOPD"], [-500., 1.5]),
    (OP["TRACECYL"], [100.]),
    (OP["TRACECYLOPD"], [100., 1.2]),
    (OP["CYLCONIC"], [1. / 400., -.7]),
    (OP["PARAXIAL"], [350.]),
    (OP["PARAXIALY"], [-120.]),
    (OP["TORUS"], [150., 900.]),
    (OP["WSPRIMARYBACK"], [ALPHA, 1.e4, 1., .4]),
    (OP["WSSECONDARYBACK"], [ALPHA, 1.e4, 1., .4]),
]
NAMES = ["tracesphere", "tracesphereopd", "tracecyl", "tracecylopd", "cylconic", "paraxial", "paraxialy", "torus",
         "wsprimaryback", "wssecondaryback"]
ZERN = (OP["ZERNSURF"], [0., 0., 7.])
LL = (OP["LLSURF"], [0., 5.])
FAN = (OP["GRATFAN"], [1e-4, 1e4, 95., .01, -1., 1.])
ROTX = (OP["ROTX_REMAINING"], [1e-4, 3.])
OTHERS = {"zern": ZERN, "ll": LL, "fan": FAN, "rotx": ROTX}

# bundle rows: opd, x, y, z, l, m, n, ux, uy, uz
R = {name: 1 << k for k, name in enumerate(["opd", "x", "y", "z", "l", "m", "n", "ux", "uy", "uz"])}
POS, DIR, NRM = R["x"] | R["y"] | R["z"], R["l"] | R["m"] | R["n"], R["ux"] | R["uy"] | R["uz"]
# (load, store) of each op alone: the LOAD / STORE of its stand-alone kernel (pxf_ops.cu), except that paraxialy
# neither reads x nor touches l
MASKS = {
    OP["TRACESPHERE"]: (POS | DIR, POS | DIR | NRM),
    OP["TRACESPHEREOPD"]: (POS | DIR | R["opd"], POS | DIR | NRM | R["opd"]),
    OP["TRACECYL"]: (POS | DIR, POS | DIR | NRM),
    OP["TRACECYLOPD"]: (POS | DIR | R["opd"], POS | DIR | NRM | R["opd"]),
    OP["CYLCONIC"]: (POS | DIR, POS | NRM),
    OP["PARAXIAL"]: (R["x"] | R["y"] | R["l"] | R["m"], R["l"] | R["m"]),
    OP["PARAXIALY"]: (R["y"] | R["m"], R["m"]),
    OP["TORUS"]: (POS | DIR, POS | NRM),
    OP["WSPRIMARYBACK"]: (POS | DIR | NRM, POS | NRM),
    OP["WSSECONDARYBACK"]: (POS | DIR | NRM, POS | NRM),
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
            if code in (OP["LLSURF"], OP["ZERNSURF"]):
                o.p[0] = struct.unpack("d", struct.pack("Q", 4096))[0]     # a non-null address (the fills ignore it)
    return arr, nops


def trace_rc(ops):
    """build_program's verdict: pxf_trace_program validates the op list before it needs a device."""
    arr, nops = ops_of([ops])
    return L().pxf_trace_program((ctypes.c_void_p * 10)(), 0, arr, nops, None, None)


def seg_fill(seg_ops, fn="pxf_segmented_table_fill", bytes_fn="pxf_segmented_table_bytes"):
    arr, nops = ops_of(seg_ops)
    nseg = len(seg_ops)
    start = np.zeros(nseg + 1, dtype=np.int64)
    start[1:] = np.cumsum([10] * nseg)
    out = np.zeros(int(getattr(L(), bytes_fn)(nops, nseg)), dtype=np.uint8)
    if fn == "pxf_segmented_table_fill":
        return getattr(L(), fn)(arr, nops, nseg, start.ctypes.data, out.ctypes.data), out
    # a table per segment of the size the fill expects (zeroed: the refusal comes before they are read)
    per = int(L().pxf_zern_table_bytes() if "zern" in fn else 2 * L().pxf_ll_table_bytes())
    tabs = np.zeros(per * nseg, dtype=np.uint8)
    return getattr(L(), fn)(arr, nops, nseg, start.ctypes.data, tabs.ctypes.data, out.ctypes.data), out


def chain(op):
    return [(OP["TRANSFORM"], [0., 0., 10., 0., 0., 0.]), op, (OP["REFRACT"], [1., 1.5]), (OP["FLATOPD"], [1.])]


@pytest.mark.parametrize("op", NEW, ids=NAMES)
def test_build_accepts_each_new_op(op):
    for ops in ([op], chain(op)):
        assert trace_rc(ops) not in (INVALID, UNSUPPORTED), L().pxf_last_error()


@pytest.mark.parametrize("other", sorted(OTHERS), ids=sorted(OTHERS))
@pytest.mark.parametrize("op", NEW, ids=NAMES)
def test_build_refuses_new_op_next_to_table_or_aux_ops(op, other):
    o = OTHERS[other]
    assert trace_rc([op, o]) == UNSUPPORTED
    assert trace_rc([o, op]) == UNSUPPORTED
    assert trace_rc(chain(op)[:2] + [o] + chain(op)[2:]) == UNSUPPORTED
    assert trace_rc([o]) != UNSUPPORTED and trace_rc([op]) != UNSUPPORTED     # each alone is fine


def header(out):
    load, store = out[:8].view(np.uint32)
    return int(load), int(store)


def seg_ops_table(out, nops, nseg):
    """the folded FusedOp table of a segmented table: (code, row, q[38]) per op, segment-major"""
    off = 48 + (-(-(nseg + 1) * 8 // 16)) * 16
    raw = out[off:off + nseg * nops * 312]
    rec = np.frombuffer(raw.tobytes(), dtype=np.dtype([("code", "<i4"), ("row", "<i4"), ("q", "<f8", 38)]))
    return rec.reshape(nseg, nops)


@pytest.mark.parametrize("op", NEW, ids=NAMES)
def test_plain_fill_accepts_with_the_stand_alone_row_masks(op):
    rc, out = seg_fill([[op], [op]])
    assert rc == OK, L().pxf_last_error()
    assert header(out) == MASKS[op[0]]


def test_plain_fill_folds_each_segments_own_scalars():
    rads, Fs, thick = [250., -400., 1.e3], [350., -80., 12.], [.4, .5, 1.]
    seg_ops = [[(OP["TRACESPHEREOPD"], [rads[s], 1.5]), (OP["PARAXIALY"], [Fs[s]]), (OP["PARAXIAL"], [Fs[s]]),
                (OP["CYLCONIC"], [1. / rads[s], -.7]), (OP["TORUS"], [150., rads[s]]),
                (OP["WSSECONDARYBACK"], [ALPHA, 1.e4, 1., thick[s]])] for s in range(3)]
    rc, out = seg_fill(seg_ops)
    assert rc == OK, L().pxf_last_error()
    t = seg_ops_table(out, 6, 3)
    for s in range(3):
        q = [t[s, k]["q"] for k in range(6)]
        assert [int(t[s, k]["code"]) for k in range(6)] == [c for c, _ in seg_ops[s]]
        # SphereP {rad2, nr, opd}, ParaxialP {F, yonly}, CylConicP {A, rad, tworad}, TorusP {rin, rout, rin2, rout2, ..}
        assert q[0][0] == rads[s] * rads[s] and q[0][1] == 1.5 and q[0][2:3].view(np.int32)[0] == 1
        assert q[1][0] == Fs[s] and q[1][1:2].view(np.int32)[0] == 1
        assert q[2][0] == Fs[s] and q[2][1:2].view(np.int32)[0] == 0
        c = 1. / rads[s]
        assert q[3][0] == (1 + -.7) * (c * c) and q[3][1] == c and q[3][2] == 2 * c
        assert q[4][1] == rads[s] and q[4][3] == rads[s] * rads[s] and q[4][4] == 4 * (rads[s] * rads[s])
        # WSP: thick is its 27th double
        assert q[5][26] == thick[s]


@pytest.mark.parametrize("fn,bytes_fn", [("pxf_segmented_table_fill_zern", "pxf_segmented_table_bytes_zern"),
                                         ("pxf_segmented_table_fill_ll", "pxf_segmented_table_bytes_ll")])
@pytest.mark.parametrize("op", NEW, ids=NAMES)
def test_zern_and_ll_fills_refuse_new_ops(op, fn, bytes_fn):
    rc, _ = seg_fill([chain(op), chain(op)], fn=fn, bytes_fn=bytes_fn)
    assert rc == UNSUPPORTED
    assert b"pxf_segmented_table_fill" in L().pxf_last_error()
    table = ZERN if "zern" in fn else LL
    rc, _ = seg_fill([chain(op) + [table], chain(op) + [table]], fn=fn, bytes_fn=bytes_fn)
    assert rc == UNSUPPORTED


def test_plain_fill_refuses_mixed_segments():
    # segments must agree on the opcode sequence, as for every other op
    rc, _ = seg_fill([chain(NEW[0]), chain(NEW[2])])
    assert rc == INVALID
    rc, _ = seg_fill([chain(NEW[0]) + [ZERN], chain(NEW[0]) + [ZERN]])
    assert rc == UNSUPPORTED


@pytest.mark.parametrize("name,op", list(zip(NAMES, NEW)), ids=NAMES)
def test_program_methods_record_code_and_scalars(name, op):
    prog = getattr(pxf.Program().transform(0, 0, 1, 0, 0, 0), name)(*op[1])
    assert prog.ops[-1] == (op[0], op[1])
    assert prog.can_hold_surface()


def test_program_refuses_mixing_in_either_order():
    P = pxf.Program
    ro, ao = ex.zernike_orders(7)
    zc = ex.zernike_coeff(len(ro))
    ax, az = ex.ll_orders(3)
    c = ex.ll_coeff(16)
    holders = [lambda p: p.zernsurf(zc, ro, ao, 62.5),
               lambda p: p.wolterprimll(220., 8400., 8500., 8400., .25, c, ax, az),
               lambda p: p.gratfan(1e-4, 1e4, 95., .01, -1., 1.),
               lambda p: p.rotx_remaining(1e-4, 3)]
    for hold in holders:
        with pytest.raises(NotImplementedError):
            hold(P()).tracesphere(250.)
        with pytest.raises(NotImplementedError):
            hold(P().torus(150., 900.))
        assert not hold(P()).can_hold_surface()


def test_segmented_program_refuses_a_mixed_program():
    # Program refuses the mix; ops added by hand reach the C fills, which refuse it as well
    P = pxf.Program
    ax, az = ex.ll_orders(3)
    c = ex.ll_coeff(16)
    ll = P().transform(0, 0, 1, 0, 0, 0).wolterprimll(220., 8400., 8500., 8400., .25, c, ax, az).reflect()
    ll.add(OP["TRACESPHERE"], 250.)
    with pytest.raises(_lib.PxfError):
        pxf.SegmentedProgram([ll, ll], [3, 4])
    ro, ao = ex.zernike_orders(7)
    zp = P().transform(0, 0, 1, 0, 0, 0).zernsurf(ex.zernike_coeff(len(ro)), ro, ao, 62.5).reflect()
    zp.add(OP["PARAXIAL"], 100.)
    with pytest.raises(_lib.PxfError):
        pxf.SegmentedProgram([zp], [3])


def all_ten_program():
    p = pxf.Program().transform(0, 0, 10, 0, 0, 0)
    for name, (_, args) in zip(NAMES, NEW):
        getattr(p, name)(*args)
        p.refract(1., 1.5)
    return p.flatopd(1.)


def test_all_ten_ops_compile_for_both_forms():
    """The specialised kernels of a program holding every new op, single and segmented, compile (NVRTC; no device
    needed)."""
    prog = all_ten_program()
    assert len(prog) == 22
    if prog.precompile() == 0:
        pytest.skip("NVRTC unavailable: " + L().pxf_jit_status().decode())
    assert prog.precompile(segmented=True) > 0, L().pxf_jit_status()
