"""Host-side table code of segmented programs with one Zernike surface per segment (no GPU needed): sizes, the
validation of pxf_segmented_table_fill_zern, the unchanged refusal of pxf_segmented_table_fill, and the ValueErrors
of SegmentedProgram."""
import struct

import numpy as np
import pytest

import pyxfocus_b200 as pxf
from pyxfocus_b200 import _lib
from pyxfocus_b200 import examples as ex

OK, INVALID, UNSUPPORTED = 0, 1, 4
OP = pxf.program.OP


def L():
    return _lib.lib()


def zern_table(nmax=7, seed=0, opd=False):
    ro, ao = (o.astype(np.int32) for o in ex.zernike_orders(nmax))
    c = ex.zernike_coeff(len(ro), seed)
    tab = np.empty(int(L().pxf_zern_table_bytes()), dtype=np.uint8)
    got = L().pxf_zern_table_fill(c.ctypes.data, ro.ctypes.data, ao.ctypes.data, len(ro), 62.5, 1 if opd else 0,
                                  1. if opd else 0., tab.ctypes.data)
    assert got == nmax
    return tab


def ops_of(seg_ops):
    """[[(code, [p...]), ...] per segment] -> pxf_op array; a ZERNSURF gets a non-null address in p[0] (the old
    entry point wants one; the new one ignores it)."""
    nops = len(seg_ops[0])
    arr = (_lib.pxf_op * (len(seg_ops) * nops))()
    for s, ops in enumerate(seg_ops):
        for k, (code, p) in enumerate(ops):
            o = arr[s * nops + k]
            o.code = code
            for j, v in enumerate(p):
                o.p[j] = v
            if code == OP["ZERNSURF"]:
                o.p[0] = struct.unpack("d", struct.pack("Q", 4096))[0]
    return arr, nops


def tzr(opd=0., nmax=7.):
    return [(OP["TRANSFORM"], [1., 0., 100., 0., 0., 0.]), (OP["ZERNSURF"], [0., opd, nmax]), (OP["REFLECT"], [])]


def fill_zern(seg_ops, tables, sizes=None):
    arr, nops = ops_of(seg_ops)
    nseg = len(seg_ops)
    start = np.zeros(nseg + 1, dtype=np.int64)
    start[1:] = np.cumsum(sizes if sizes is not None else [10] * nseg)
    out = np.zeros(int(L().pxf_segmented_table_bytes_zern(nops, nseg)), dtype=np.uint8)
    zt = None if tables is None else np.concatenate(tables)
    rc = L().pxf_segmented_table_fill_zern(arr, nops, nseg, start.ctypes.data,
                                           None if zt is None else zt.ctypes.data, out.ctypes.data)
    return rc, out


@pytest.mark.parametrize("nops,nseg", [(1, 1), (3, 7), (14, 1000), (24, 25000)])
def test_table_sizes(nops, nseg):
    plain = int(L().pxf_segmented_table_bytes(nops, nseg))
    zern = int(L().pxf_segmented_table_bytes_zern(nops, nseg))
    assert plain > 0 and zern >= plain + nseg * int(L().pxf_zern_table_bytes())
    assert int(L().pxf_segmented_table_bytes_zern(0, nseg)) == 0 and int(L().pxf_segmented_table_bytes_zern(nops, 0)) == 0


def test_old_fill_still_refuses_zernike():
    arr, nops = ops_of([tzr(), tzr()])
    start = np.array([0, 5, 9], dtype=np.int64)
    out = np.zeros(int(L().pxf_segmented_table_bytes(nops, 2)), dtype=np.uint8)
    assert L().pxf_segmented_table_fill(arr, nops, 2, start.ctypes.data, out.ctypes.data) == UNSUPPORTED
    assert b"pxf_segmented_table_fill_zern" in L().pxf_last_error()


def test_fill_copies_every_segment_table():
    tabs = [zern_table(7, 1), zern_table(3, 2), zern_table(5, 3)]
    rc, out = fill_zern([tzr(), tzr(nmax=3.), tzr(nmax=5.)], tabs, sizes=[0, 4097, 3])
    assert rc == OK
    nb = int(L().pxf_zern_table_bytes())
    assert np.array_equal(out[-3 * nb:], np.concatenate(tabs))      # behind the rest, back to back


def test_fill_without_zernike_op_accepts_no_tables():
    rc, _ = fill_zern([[(OP["REFLECT"], [])], [(OP["REFLECT"], [])]], None)
    assert rc == OK


def test_rejects_radial_order_8():
    rc, _ = fill_zern([tzr(), tzr()], [zern_table(7), zern_table(8)])
    assert rc == UNSUPPORTED


def test_rejects_mixed_opd_flags():
    rc, _ = fill_zern([tzr(opd=0.), tzr(opd=1.)], [zern_table(7), zern_table(7, opd=True)])
    assert rc == INVALID


def test_rejects_zernike_op_at_different_positions():
    moved = [tzr()[0], tzr()[2], tzr()[1]]
    rc, _ = fill_zern([tzr(), moved], [zern_table(7), zern_table(7)])
    assert rc == INVALID


def test_rejects_null_tables():
    rc, _ = fill_zern([tzr(), tzr()], None)
    assert rc == INVALID


def test_rejects_grating_fan():
    fan = [(OP["GRATFAN"], [1e-4, 1e4, 95., .01, -1., 1.])]
    rc, _ = fill_zern([fan, fan], None)
    assert rc == UNSUPPORTED
    rc, _ = fill_zern([tzr() + fan, tzr() + fan], [zern_table(7), zern_table(7)])
    assert rc == UNSUPPORTED


def test_segmented_program_rejects_misaligned_zernike_ops():
    ro, ao = ex.zernike_orders(7)
    c = ex.zernike_coeff(len(ro))
    P = pxf.Program
    a = P().transform(0, 0, 1, 0, 0, 0).zernsurf(c, ro, ao, 62.5).reflect()
    b = P().transform(0, 0, 1, 0, 0, 0).reflect().zernsurf(c, ro, ao, 62.5)
    with pytest.raises(ValueError):
        pxf.SegmentedProgram([a, b], [3, 4])
    with_nr = P().transform(0, 0, 1, 0, 0, 0).zernsurf(c, ro, ao, 62.5, 1.).reflect()
    with pytest.raises(ValueError):
        pxf.SegmentedProgram([a, with_nr], [3, 4])
    bare = P().transform(0, 0, 1, 0, 0, 0).add(OP["ZERNSURF"], 0., 0., 7.).reflect()     # no recorded table
    with pytest.raises(ValueError):
        pxf.SegmentedProgram([a, bare], [3, 4])
