"""Host-side code of radgratW and grat as fused-program ops (no GPU needed): the opcodes and how Program encodes them,
the broadcast of scalars, the refusal of arrays of the wrong length, dtype or device and of null addresses, the
combinations build_program accepts and refuses, the row masks, segmented fills with the ops at the same and at
different positions, the refusal of the host-buffer path, and the NVRTC compilation of chains holding each op."""
import ctypes
import struct

import numpy as np
import pytest
import torch

import pyxfocus_b200 as pxf
from pyxfocus_b200 import _lib

OK, INVALID, UNSUPPORTED = 0, 1, 4
OP = pxf.program.OP
ADDR = struct.unpack("d", struct.pack("Q", 4096))[0]          # a non-null device address (nothing is launched)
RADGRATW = (OP["RADGRATW"], [ADDR, .2, -3.])
GRAT = (OP["GRAT"], [160., ADDR, ADDR])
R = {name: 1 << k for k, name in enumerate(["opd", "x", "y", "z", "l", "m", "n", "ux", "uy", "uz"])}
DIR = R["l"] | R["m"] | R["n"]
# the ops the side-array interpreter does not hold
REFUSED = {"zernsurf": (OP["ZERNSURF"], [ADDR, 0., 7.]), "zernphase": (OP["ZERNPHASE"], [ADDR, 1e-6, 7.]),
           "llsurf": (OP["LLSURF"], [ADDR, 5.]), "tracesphere": (OP["TRACESPHERE"], [250.]),
           "torus": (OP["TORUS"], [150., 900.]), "conicplus": (OP["CONICPLUS"], [ADDR]),
           "legsurf": (OP["LEGSURF"], [ADDR])}
ACCEPTED = {"radgrat": (OP["RADGRAT"], [5., .2, -3.]), "gratfan": (OP["GRATFAN"], [1e-4, 1e4, 95., .01, -1., 1.]),
            "vignette": (OP["VIGNETTE_MAG"], []), "kickn": (OP["KICKN"], [1e-3, 0.])}


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
    arr, nops = ops_of([ops])
    return L().pxf_trace_program((ctypes.c_void_p * 10)(), 0, arr, nops, None, None)


def seg_fill(seg_ops):
    arr, nops = ops_of(seg_ops)
    nseg = len(seg_ops)
    start = np.zeros(nseg + 1, dtype=np.int64)
    start[1:] = np.cumsum([10] * nseg)
    out = np.zeros(int(L().pxf_segmented_table_bytes(nops, nseg)), dtype=np.uint8)
    return L().pxf_segmented_table_fill(arr, nops, nseg, start.ctypes.data, out.ctypes.data), out


def chain(op):
    return [(OP["TRANSFORM"], [0., 0., 10., .01, 0., 0.]), (OP["FLAT"], []), op,
            (OP["TRANSFORM"], [1., 0., 5., 0., 0., 0.]), (OP["FLAT"], [])]


def test_opcodes_and_encoding():
    assert (OP["RADGRATW"], OP["GRAT"]) == (41, 42)
    w = np.linspace(3.6, 7.2, 5)
    p = pxf.Program().radgratw(w, .2, -3.).grat(160., -1, w).grat(150., w, 5.5)
    assert [op for op in p.ops] == [(41, [0., .2, -3.]), (42, [160., 0., 0.]), (42, [150., 0., 0.])]
    assert p._arrays[0][0] is w                      # kept by reference, uploaded once per device
    # scalars of grat are kept as floats and broadcast when the program runs
    assert p._arrays[1][0] == -1. and isinstance(p._arrays[1][0], float) and p._arrays[2][1] == 5.5
    # the ops carry the arrays' addresses at p[0] (radgratw) and p[1], p[2] (grat)
    t = [torch.zeros(5, dtype=torch.float64) for _ in range(5)]
    arr = p.c_ops(None, {0: [t[0]], 1: [t[1], t[2]], 2: [t[3], t[4]]})
    addr = lambda v: struct.unpack("Q", struct.pack("d", v))[0]          # noqa: E731
    assert addr(arr[0].p[0]) == t[0].data_ptr() and arr[0].p[1] == .2 and arr[0].p[2] == -3.
    assert arr[1].p[0] == 160. and addr(arr[1].p[1]) == t[1].data_ptr() and addr(arr[1].p[2]) == t[2].data_ptr()
    with pytest.raises(ValueError):
        p.c_ops(None)


def test_arrays_of_the_wrong_kind_are_refused():
    P = pxf.Program
    for bad in (np.ones(4, dtype=np.float32), np.ones(4, dtype=np.int64), np.ones((2, 2)),
                torch.ones(4, dtype=torch.float64), [1., 2.]):
        with pytest.raises(ValueError):
            P().radgratw(bad, .2, -3.)
        with pytest.raises(ValueError):
            P().grat(160., bad, 5.)
    with pytest.raises(ValueError):
        P().radgratw(5., .2, -3.)                    # radgratw has no scalar wave: that is radgrat
    # the length is checked against the bundle before anything is uploaded
    p = P().radgratw(np.ones(4), .2, -3.)
    with pytest.raises(ValueError):
        p.device_arrays(5, "cuda:0")
    g = P().grat(160., -1., np.ones(4))
    with pytest.raises(ValueError):
        g.device_arrays(3, "cuda:0")
    with pytest.raises(ValueError):
        pxf.SegmentedProgram([P().radgratw(np.ones(9), .2, -3.)] * 2, [5, 5], device="cuda:0")


def test_null_addresses_are_invalid():
    assert trace_rc([(OP["RADGRATW"], [0., .2, -3.])]) == INVALID
    assert trace_rc([(OP["GRAT"], [160., 0., ADDR])]) == INVALID
    assert trace_rc([(OP["GRAT"], [160., ADDR, 0.])]) == INVALID


@pytest.mark.parametrize("op", [RADGRATW, GRAT], ids=["radgratw", "grat"])
def test_build_accepts_the_ops_alone_in_chains_and_next_to_the_side_array_ops(op):
    for ops in ([op], chain(op), [op, RADGRATW, GRAT]):
        assert trace_rc(ops) not in (INVALID, UNSUPPORTED), L().pxf_last_error()
    for o in ACCEPTED.values():
        assert trace_rc([op, o]) not in (INVALID, UNSUPPORTED), L().pxf_last_error()
        assert trace_rc([o, op]) not in (INVALID, UNSUPPORTED), L().pxf_last_error()


@pytest.mark.parametrize("other", sorted(REFUSED))
@pytest.mark.parametrize("op", [RADGRATW, GRAT], ids=["radgratw", "grat"])
def test_build_refuses_the_ops_next_to_table_and_surface_ops(op, other):
    o = REFUSED[other]
    assert trace_rc([op, o]) == UNSUPPORTED
    assert trace_rc([o, op]) == UNSUPPORTED
    assert trace_rc(chain(op)[:2] + [o] + chain(op)[2:]) == UNSUPPORTED


def test_program_refuses_the_same_mixes():
    P = pxf.Program
    w = np.ones(3)
    holders = [lambda p: p.tracesphere(50.), lambda p: p.conicplus(40., -1.2, [1e-6]),
               lambda p: p.zernsurf([1.], [0], [0], 60.), lambda p: p.zernphase([1.], [0], [0], 60., 1e-6),
               lambda p: p.wolterprimll(220., 8400., 8500., 8400., .25, [1e-4], [1], [0])]
    for hold in holders:
        for add in (lambda p: p.radgratw(w, .2, -3.), lambda p: p.grat(160., -1., w)):
            with pytest.raises(NotImplementedError):
                add(hold(P()))
            with pytest.raises(NotImplementedError):
                hold(add(P()))
    assert P().gratfan(1e-4, 1e4, 95., .01, -1, 1.).radgrat(5., .2, -1).radgratw(w, .2, -3.).can_hold_arrays()


def test_row_masks():
    for op, masks in ((RADGRATW, (R["x"] | R["y"] | DIR, DIR)), (GRAT, (DIR, DIR))):
        rc, out = seg_fill([[op], [op]])
        assert rc == OK, L().pxf_last_error()
        assert tuple(int(v) for v in out[:8].view(np.uint32)) == masks
    # behind a flat the ops still read x, y and the direction: nothing the flat does not write is dropped
    rc, out = seg_fill([chain(RADGRATW)] * 2)
    assert rc == OK, L().pxf_last_error()


def test_segmented_fill_takes_the_ops_at_the_same_positions_only():
    a = struct.unpack("d", struct.pack("Q", 8192))[0]
    rc, _ = seg_fill([chain(RADGRATW), chain((OP["RADGRATW"], [a, .3, -2.]))])
    assert rc == OK, L().pxf_last_error()
    rc, _ = seg_fill([chain(GRAT) + [RADGRATW], chain((OP["GRAT"], [150., a, a])) + [RADGRATW]])
    assert rc == OK, L().pxf_last_error()
    rc, _ = seg_fill([[RADGRATW, GRAT], [GRAT, RADGRATW]])
    assert rc == INVALID
    rc, _ = seg_fill([[RADGRATW, (OP["FLAT"], [])], [(OP["FLAT"], []), RADGRATW]])
    assert rc == INVALID
    rc, _ = seg_fill([[RADGRATW], [(OP["RADGRAT"], [5., .2, -3.])]])
    assert rc == INVALID


@pytest.mark.parametrize("op", [RADGRATW, GRAT], ids=["radgratw", "grat"])
def test_host_buffer_path_refuses_the_ops(op):
    arr, nops = ops_of([chain(op)])
    rows = [np.zeros(4) for _ in range(10)]
    ptrs = (ctypes.c_void_p * 10)(*[r.ctypes.data for r in rows])
    rc = L().pxf_host_trace_program(ptrs, 4, arr, nops, 1, None, None, None, None, None)
    assert rc == UNSUPPORTED
    assert b"RADGRATW" in L().pxf_last_error()


def test_chains_with_each_op_compile_plain_and_segmented():
    w = np.ones(3)
    progs = [pxf.Program().transform(0, 0, 10, 0, 0, 0).flat().radgratw(w, .2, -3.).transform(0, 0, 5, 0, 0, 0).flat(),
             pxf.Program().transform(0, 0, 10, 0, 0, 0).flat().grat(160., w, -1.).transform(0, 0, 5, 0, 0, 0).flat()]
    if progs[0].precompile() == 0:
        pytest.skip("NVRTC unavailable: " + L().pxf_jit_status().decode())
    for p in progs:
        assert p.precompile() > 0, L().pxf_jit_status()
        assert p.precompile(segmented=True) > 0, L().pxf_jit_status()
