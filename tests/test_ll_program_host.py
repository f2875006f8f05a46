"""Host-side code of the Legendre-Legendre shells as fused-program ops (no GPU needed): the table layout and fold of
pxf_ll_table_fill, the validation of build_program and pxf_segmented_table_fill_ll, the unchanged refusal of the
other segmented fills, and the ValueError / NotImplementedError paths of Program and SegmentedProgram."""
import ctypes
import struct

import numpy as np
import pytest

import pyxfocus_b200 as pxf
from pyxfocus_b200 import _lib
from pyxfocus_b200 import examples as ex

OK, INVALID, UNSUPPORTED = 0, 1, 4
OP = pxf.program.OP
HEAD = 4 * 4 + 14 * 8          # kind, nz, nt, stride; 14 folded scalars
GEOM = dict(r0=220., z0=8400., psi=1., S=0., zmax=8500., zmin=8400., dphi=.25)


def L():
    return _lib.lib()


def fill(axial, az, coeff=None, kind=0, S=0., psi=1.):
    ax, a = np.ascontiguousarray(axial, dtype=np.int32), np.ascontiguousarray(az, dtype=np.int32)
    c = np.ascontiguousarray(np.random.default_rng(len(ax)).normal(0, 1e-4, len(ax)) if coeff is None else coeff,
                             dtype=np.float64)
    tab = np.zeros(int(L().pxf_ll_table_bytes()), dtype=np.uint8)
    top = L().pxf_ll_table_fill(kind, 220., 8400., psi, S, 8500., 8400., .25, c.ctypes.data, ax.ctypes.data,
                                a.ctypes.data, len(c), tab.ctypes.data)
    return top, tab


def parse(tab):
    ints = tab[:16].view(np.int32)
    return dict(kind=ints[0], nz=ints[1], nt=ints[2], stride=ints[3], C=tab[HEAD:].view(np.float64).reshape(8, 8))


def test_table_sizes():
    tb = int(L().pxf_ll_table_bytes())
    assert tb == HEAD + 64 * 8
    for nops, nseg in [(1, 1), (6, 7), (24, 25000)]:
        plain = int(L().pxf_segmented_table_bytes(nops, nseg))
        assert int(L().pxf_segmented_table_bytes_ll(nops, nseg)) >= plain + nseg * 2 * tb
    assert int(L().pxf_segmented_table_bytes_ll(0, 3)) == 0 and int(L().pxf_segmented_table_bytes_ll(3, 0)) == 0


@pytest.mark.parametrize("nmax", [0, 2, 3, 5, 7])
def test_fill_matrix_is_the_power_basis_fold(nmax):
    rng = np.random.default_rng(nmax)
    axial = np.concatenate([rng.integers(0, nmax + 1, 20), [nmax, 0]])
    az = np.concatenate([rng.integers(0, nmax + 1, 20), [0, nmax]])
    coeff = rng.normal(0., 3e-4, len(axial))
    top, tab = fill(axial, az, coeff)
    assert top == nmax
    t = parse(tab)
    # power-basis coefficients of each Legendre polynomial as exact rationals, (n+1) P_{n+1} = (2n+1) x P_n - n P_{n-1}
    # (numpy's leg2poly agrees to rounding: it is computed in floating point), the outer products summed exactly, then
    # rounded once
    from fractions import Fraction
    P = [[Fraction(1)], [Fraction(0), Fraction(1)]]
    for m in range(1, 7):
        nxt = [Fraction(0)] * (m + 2)
        for k in range(m + 2):
            nxt[k] = ((2 * m + 1) * (P[m][k - 1] if k else 0) - m * (P[m - 1][k] if k < m else 0)) / (m + 1)
        P.append(nxt)
    for m in range(8):
        ref = np.polynomial.legendre.leg2poly(np.eye(8)[m])
        assert np.allclose([float(v) for v in P[m]], ref, rtol=1e-14, atol=0)
    exact = [[Fraction(0)] * 8 for _ in range(8)]
    mag = np.zeros((8, 8))
    for c, i, j in zip(coeff, axial, az):
        for a in range(len(P[i])):
            for b in range(len(P[j])):
                term = Fraction(c) * P[i][a] * P[j][b]
                exact[a][b] += term
                mag[a, b] += abs(float(term))
    want = np.array([[float(v) for v in row] for row in exact])
    got = t["C"]
    # 1 ulp, plus the long-double rounding of the fold's running sums where terms cancel (2**-63 per term, generously)
    tol = np.spacing(np.abs(want)) + 2. ** -58 * mag
    assert np.all(np.abs(got - want) <= tol), np.max(np.abs(got - want) - tol)
    # zero beyond the orders present, and no -0 anywhere (the zero padding must be +0)
    assert np.all(got[nmax + 1:, :] == 0) and np.all(got[:, nmax + 1:] == 0)
    assert not np.any(np.signbit(got[got == 0]))


@pytest.mark.parametrize("nz,nt", [(0, 0), (3, 1), (2, 4), (5, 5), (6, 0), (1, 7)])
def test_orders_in_the_table_follow_the_rounding_of_the_fold(nz, nt):
    top, tab = fill([nz, 0], [0, nt])
    t = parse(tab)
    assert (t["nz"], t["nt"]) == (nz, nt) and top == max(nz, nt)
    m = max(nz, nt)
    assert t["stride"] - 1 == (3 if m <= 3 else 5 if m <= 5 else 7)


def test_fill_rejects_orders_above_7_and_bad_arguments():
    assert fill([8], [0])[0] == -1
    assert fill([0], [9])[0] == -1
    assert fill([-1], [0])[0] == -1
    assert fill([1], [1], kind=3)[0] == -1


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


def pair(order=5.):
    return [(OP["TRANSFORM"], [0., 0., 8400., 0., 0., 0.]), (OP["LLSURF"], [0., order]), (OP["REFLECT"], []),
            (OP["LLSURF"], [0., order]), (OP["REFLECT"], []), (OP["FLAT"], [])]


def fill_ll(seg_ops, tables, sizes=None, fn="pxf_segmented_table_fill_ll", bytes_fn="pxf_segmented_table_bytes_ll"):
    arr, nops = ops_of(seg_ops)
    nseg = len(seg_ops)
    start = np.zeros(nseg + 1, dtype=np.int64)
    start[1:] = np.cumsum(sizes if sizes is not None else [10] * nseg)
    out = np.zeros(int(getattr(L(), bytes_fn)(nops, nseg)), dtype=np.uint8)
    lt = None if tables is None else np.concatenate(tables)
    if fn == "pxf_segmented_table_fill":
        return getattr(L(), fn)(arr, nops, nseg, start.ctypes.data, out.ctypes.data), out
    return getattr(L(), fn)(arr, nops, nseg, start.ctypes.data, None if lt is None else lt.ctypes.data,
                            out.ctypes.data), out


def tables(orders):
    return [fill([o, 1], [1, o], kind=k % 2)[1] for k, o in enumerate(orders)]


def trace_rc(ops):
    """build_program's verdict: pxf_trace_program validates the op list before it needs a device."""
    arr, nops = ops_of([ops])
    return L().pxf_trace_program((ctypes.c_void_p * 10)(), 0, arr, nops, None, None)


def test_fill_copies_every_segment_table():
    tabs = tables([3, 5, 7, 2, 0, 6])      # 3 segments x 2 LL ops, orders differ between segments
    rc, out = fill_ll([pair(), pair(), pair()], tabs, sizes=[0, 4097, 3])
    assert rc == OK, L().pxf_last_error()
    nb = int(L().pxf_ll_table_bytes())
    off = int(L().pxf_segmented_table_bytes(6, 3))
    off += -off % 16
    assert np.array_equal(out[off:off + 6 * nb], np.concatenate(tabs))


def test_fill_without_ll_op_accepts_no_tables():
    rc, _ = fill_ll([[(OP["REFLECT"], [])], [(OP["REFLECT"], [])]], None)
    assert rc == OK


def test_build_rejects_order_8():
    assert trace_rc(pair(7.)[:2]) != UNSUPPORTED          # valid up to here (fails later: no device / null rows)
    assert trace_rc(pair(8.)[:2]) == UNSUPPORTED
    top, t8 = fill([7], [7])
    t8 = t8.copy()
    t8[4:8] = np.array([8], dtype=np.int32).view(np.uint8)     # a forged table of order 8
    rc, _ = fill_ll([pair()[:2], pair()[:2]], [tables([3])[0], t8])
    assert rc == UNSUPPORTED


def test_rejects_a_third_ll_op():
    three = pair() + [(OP["LLSURF"], [0., 3.])]
    assert trace_rc(three) == UNSUPPORTED
    rc, _ = fill_ll([three], tables([3, 3, 3]))
    assert rc == UNSUPPORTED


def test_rejects_ll_with_zernike_or_grating_fan():
    zern = [(OP["ZERNSURF"], [0., 0., 7.])]
    assert trace_rc(pair() + zern) == UNSUPPORTED
    assert trace_rc(zern + pair()[:2]) == UNSUPPORTED
    fan = [(OP["GRATFAN"], [1e-4, 1e4, 95., .01, -1., 1.])]
    assert trace_rc(pair() + fan) == UNSUPPORTED
    rc, _ = fill_ll([pair() + zern], tables([3, 3]))
    assert rc == UNSUPPORTED


def test_rejects_null_tables():
    rc, _ = fill_ll([pair(), pair()], None)
    assert rc == INVALID
    arr, nops = ops_of([[(OP["LLSURF"], [0., 3.])]])
    arr[0].p[0] = 0.
    assert L().pxf_trace_program((ctypes.c_void_p * 10)(), 0, arr, nops, None, None) == INVALID


def test_rejects_ll_ops_at_different_positions():
    moved = [pair()[0], pair()[2], pair()[1], pair()[3], pair()[4], pair()[5]]
    rc, _ = fill_ll([pair(), moved], tables([3, 3, 3, 3]))
    assert rc == INVALID


@pytest.mark.parametrize("fn,bytes_fn", [("pxf_segmented_table_fill", "pxf_segmented_table_bytes"),
                                         ("pxf_segmented_table_fill_zern", "pxf_segmented_table_bytes_zern")])
def test_old_fills_refuse_ll(fn, bytes_fn):
    rc, _ = fill_ll([pair(), pair()], None, fn=fn, bytes_fn=bytes_fn)
    assert rc == UNSUPPORTED
    assert b"pxf_segmented_table_fill_ll" in L().pxf_last_error()


def test_program_value_and_not_implemented_errors():
    P = pxf.Program
    ax, az = ex.ll_orders(5)
    c = ex.ll_coeff(36)
    g = (220., 8400., 8500., 8400., .25)
    with pytest.raises(ValueError):
        P().wolterprimll(*g, c[:-1], ax, az)                 # lengths differ
    with pytest.raises(ValueError):
        P().wolterprimll(*g, [], [], [])
    with pytest.raises(ValueError):
        P().wolterprimll(*g, [1e-4], [-1], [0])
    with pytest.raises(ValueError):
        P().wolterprimll(*g, [1e-4], [1.5], [0])
    with pytest.raises(NotImplementedError):
        P().wolterprimll(*g, [1e-4], [8], [0])
    two = P().wolterprimll(*g, c, ax, az).woltersecll(220., 8400., 1., 8400., 8300., .25, c, ax, az)
    with pytest.raises(NotImplementedError):
        two.ellipsoidwoltll(220., 8400., 1., 2.5e5, 8500., 8400., .25, c, ax, az)
    ro, ao = ex.zernike_orders(7)
    with pytest.raises(NotImplementedError):
        P().wolterprimll(*g, c, ax, az).zernsurf(ex.zernike_coeff(len(ro)), ro, ao, 62.5)
    with pytest.raises(NotImplementedError):
        P().zernsurf(ex.zernike_coeff(len(ro)), ro, ao, 62.5).wolterprimll(*g, c, ax, az)
    assert [code for code, _ in two.ops] == [OP["LLSURF"]] * 2 and two.ops[0][1] == [0., 5.]


def test_segmented_program_rejects_missing_tables_and_misaligned_ll_ops():
    P = pxf.Program
    ax, az = ex.ll_orders(3)
    c = ex.ll_coeff(16)
    a = P().transform(0, 0, 1, 0, 0, 0).wolterprimll(220., 8400., 8500., 8400., .25, c, ax, az).reflect()
    b = P().transform(0, 0, 1, 0, 0, 0).reflect().wolterprimll(220., 8400., 8500., 8400., .25, c, ax, az)
    with pytest.raises(ValueError):
        pxf.SegmentedProgram([a, b], [3, 4])
    bare = P().transform(0, 0, 1, 0, 0, 0).add(OP["LLSURF"], 0., 3.).reflect()     # no recorded table
    with pytest.raises(ValueError):
        pxf.SegmentedProgram([a, bare], [3, 4])


def test_ll_pair_program_compiles_for_both_forms():
    """The specialised kernels of the LL pair, single and segmented, compile (NVRTC; no device needed)."""
    prog = ex.llpair_program(ex.ll_coeff(36), ex.ll_coeff(36, 1), *ex.ll_orders(5))
    if prog.precompile() == 0:
        pytest.skip("NVRTC unavailable: " + L().pxf_jit_status().decode())
    assert prog.precompile(segmented=True) > 0, L().pxf_jit_status()
