"""radgratW and grat as fused-program ops against the stand-alone entry points, on whichever path this process runs:
the interpreter with PXF_JIT=0, the run-time specialised kernels with PXF_JIT_MIN_RAYS=0.  Every comparison is of
64-bit patterns.  Prints the kernel names it saw and exits non-zero on the first mismatch.

    python tests/run_grating_ops.py interp|jit
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import pyxfocus_b200 as pxf                              # noqa: E402
from pyxfocus_b200 import surfacesf, transformationsf    # noqa: E402
from pyxfocus_b200._call import bundle_alloc, bundle_split    # noqa: E402

DEV = torch.device("cuda", 0)
T1 = (0., 0., 10., .01, .02, 0.)           # the Fortran's arguments (transformations.transform negates them)
T2 = (1., -2., 5., 0., -.01, .03)
SEEN = set()


def bits(t):
    return t.detach().cpu().numpy().view(np.int64)


def same(a, b, what):
    """Every value by its bits, NaN for NaN: the sign of a NaN follows the operand order the compiler picked (a
    negation flips it), so two builds of the same arithmetic may give NaNs of either sign."""
    for k in range(10):
        x, y = a[k].detach().cpu().numpy(), b[k].detach().cpu().numpy()
        nx, ny = np.isnan(x), np.isnan(y)
        bad = np.flatnonzero((nx != ny) | ((x.view(np.int64) != y.view(np.int64)) & ~(nx & ny)))
        if bad.size:
            raise AssertionError("%s: row %d differs at %d rays (first %d)" % (what, k, bad.size, bad[0]))


def source(num, seed, edges=False):
    """A bundle heading down -z at small angles; ``edges``: rays with y = 0, x = y = 0, and steep directions."""
    r = np.random.default_rng(seed)
    rows = [np.zeros(num) for _ in range(10)]
    rows[1], rows[2] = r.uniform(-50., 50., num), r.uniform(-50., 50., num)
    rows[3] = r.uniform(-1., 1., num)
    rows[4], rows[5] = r.uniform(-.05, .05, num), r.uniform(-.05, .05, num)
    rows[6] = -np.sqrt(1. - rows[4] ** 2 - rows[5] ** 2)
    rows[0] = r.uniform(0., 1., num)
    rows[9] = np.ones(num)
    if edges and num >= 8:
        rows[2][0:2] = [0., -0.]
        rows[1][2], rows[2][2] = 0., 0.
        rows[1][3], rows[2][3] = -0., -0.
        rows[4][4:6], rows[5][4:6] = [.9, -.8], [.3, .5]
        rows[6][4:6] = [np.sqrt(1 - .81 - .09), -np.sqrt(1 - .64 - .25)]
    out = bundle_alloc(num, DEV)
    for o, v in zip(out, rows):
        o.copy_(torch.from_numpy(v))
    return out


def arrays(num, seed, edges=False):
    r = np.random.default_rng(seed + 100)
    wave = r.uniform(3.6, 7.2, num)
    order = r.integers(-3, 4, num).astype(np.float64)
    if edges and num >= 8:
        wave[:4] = [np.nan, 0., -0., 1e3]          # NaN, +-0, and a kick that leaves l^2+m^2 > 1 in grat
        order[4:8] = [np.nan, -0., 0., 400.]
    return torch.from_numpy(wave).to(DEV), torch.from_numpy(order).to(DEV)


def clone(rays):
    out = bundle_alloc(rays[1].shape[0], DEV)
    for o, r in zip(out, rays):
        o.copy_(r)
    return out


def standalone(rays, op, chain):
    x, y, z, l, m, n, ux, uy, uz = rays[1:]
    if chain:
        transformationsf.transform(*rays[1:], *T1)
        surfacesf.flat(x, y, z, l, m, n, ux, uy, uz)
    kind, p = op
    if kind == "radgratw":
        transformationsf.radgratw(x, y, l, m, n, p["wave"], p["dpermm"], p["order"])
    else:
        transformationsf.grat(x, y, l, m, n, p["d"], p["order"], p["wave"])
    if chain:
        transformationsf.transform(*rays[1:], *T2)
        surfacesf.flat(x, y, z, l, m, n, ux, uy, uz)


def program(op, chain):
    prog = pxf.Program()
    if chain:
        prog.transform(*T1).flat()
    kind, p = op
    if kind == "radgratw":
        prog.radgratw(p["wave"], p["dpermm"], p["order"])
    else:
        prog.grat(p["d"], p["order"], p["wave"])
    if chain:
        prog.transform(*T2).flat()
    return prog


def ops_for(num, seed, edges):
    wave, order = arrays(num, seed, edges)
    return [("radgratw", dict(wave=wave, dpermm=2., order=-3.)),
            ("grat", dict(d=160., order=order, wave=wave)),
            ("grat", dict(d=160., order=-2., wave=wave)),                   # a scalar order, broadcast
            ("grat", dict(d=160., order=order, wave=wave.cpu().numpy()))]   # a host array, uploaded


def check_alone_and_chained():
    for num in (0, 1, 2, 3, 1001, 4099):
        for edges in (False, True):
            for op in ops_for(num, num, edges):
                for chain in (False, True):
                    src = source(num, num, edges)
                    want = clone(src)
                    p = dict(op[1])
                    if op[0] == "grat":
                        p = dict(p, order=torch.as_tensor(p["order"], dtype=torch.float64, device=DEV).expand(num)
                                 .contiguous(), wave=torch.as_tensor(p["wave"], device=DEV))
                    standalone(want, (op[0], p), chain)
                    prog = program(op, chain)
                    inplace = clone(src)
                    prog.run(inplace)
                    if num:
                        SEEN.add(pxf.last_trace_kernel())
                    same(inplace, want, "%s n=%d edges=%s chain=%s in place" % (op[0], num, edges, chain))
                    out = clone(src)
                    prog.run(src, out=out)
                    same(out, want, "%s n=%d edges=%s chain=%s out of place" % (op[0], num, edges, chain))
                    same(src, source(num, num, edges), "input of the out-of-place run")
    print("alone and chained: ok")


def check_segmented():
    sizes = [1000, 3000, 1, 0, 2500, 4097]
    num = sum(sizes)
    start = np.concatenate([[0], np.cumsum(sizes)])
    wave, order = arrays(num, 7, True)
    wave2 = wave.flip(0).contiguous()
    progs, singles = [], []
    for k in range(len(sizes)):
        w = wave if k % 2 else wave2
        mk = lambda: (pxf.Program().transform(*T1).flat().radgratw(w, 2. + .1 * k, -3. + k)      # noqa: E731
                      .grat(150. + k, float(k - 2) if k % 3 else order, w).transform(*T2).flat())
        progs.append(mk())
        lo, hi = int(start[k]), int(start[k + 1])
        singles.append(pxf.Program().transform(*T1).flat().radgratw(w[lo:hi], 2. + .1 * k, -3. + k)
                       .grat(150. + k, float(k - 2) if k % 3 else order[lo:hi], w[lo:hi]).transform(*T2).flat())
    seg = pxf.SegmentedProgram(progs, sizes, device=DEV)
    for oop in (False, True):
        src = source(num, 11, True)
        got = clone(src) if not oop else bundle_alloc(num, DEV)
        if oop:
            for o, r in zip(got, src):
                o.copy_(r)
            seg.run(src, out=got)
        else:
            seg.run(got)
        SEEN.add(pxf.last_trace_kernel())
        want = clone(src)
        for k, part in enumerate(bundle_split(want, sizes)):
            if sizes[k]:
                singles[k].run(part)
        same(got, want, "segmented, out of place=%s" % oop)
    print("segmented: ok")


if __name__ == "__main__":
    mode = sys.argv[1]
    check_alone_and_chained()
    check_segmented()
    print("kernels:", sorted(SEEN))
    if mode == "interp":
        assert all("k_program" in k for k in SEEN), SEEN
        assert "k_program<aux> (interpreter)" in SEEN and "k_program_seg<grat> (interpreter)" in SEEN, SEEN
    else:
        assert any("CRadgratW" in k for k in SEEN) and any("CGrat" in k for k in SEEN), SEEN
        assert any(k.startswith("pxf_jit_chain_seg") for k in SEEN), SEEN
    print("ok")
