"""The remaining scalar surfaces as fused-program ops: a program gives the bits of the stand-alone calls it replaces
(each op, with and without a vignette predicate, in place and out of place, sphere and cylinder misses included),
``fused`` records the surfaces2.npz flows into one launch, segmented programs give the bits of per-segment
``Program.run`` (interpreter and run-time specialised kernel alike) in one launch, the host-buffer path gives the bits
of the device program, and mixing with a Zernike surface or an LL shell flushes and keeps the stand-alone bits."""
import os
import subprocess
import sys

import numpy as np
import pytest

from ll_cases import source as ll_source
from surface_cases import LAYOUT, SEG, SINGLE, single_name, single_program, single_routines, source, vig_cut
from util import assert_bit_equal, assert_close, rows_of, to_dev, to_host

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pxf():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyxfocus_b200 as p
    return p


def bits(t):
    import torch
    return t.contiguous().view(torch.int64).cpu().numpy()


def assert_same_bits(got, want, what):
    for row in range(10):
        assert np.array_equal(bits(got[row]), bits(want[row])), (what, row)


@pytest.mark.parametrize("oop", [False, True], ids=["inplace", "oop"])
@pytest.mark.parametrize("vig", [False, True], ids=["novig", "vig"])
@pytest.mark.parametrize("name", sorted(SINGLE))
def test_program_equals_stand_alone_calls(pxf, name, vig, oop):
    import torch
    h = source(SINGLE[name][2], 20_001, seed=3)
    mid = to_dev(h)
    single_routines(pxf, mid, name, upto_op=True)
    prog = single_program(pxf, name, vig_rows=to_host(mid) if vig else None)
    rays = to_dev(h)
    out = [torch.full_like(r, float("nan")) for r in rays] if oop else None      # a missing store shows
    alive = prog.run(rays, out=out)
    got = out if oop else rays
    ref = to_dev(h)
    single_routines(pxf, ref, name)
    if vig:
        row, lo, hi = vig_cut(to_host(mid))
        want_alive = (mid[row] > lo) & (mid[row] < hi)
        assert torch.equal(alive, want_alive.to(torch.uint8))
        assert 0 < int(alive.sum()) < alive.shape[0]
        # a stopped ray is stored in the state it had at the predicate
        ref = [torch.where(want_alive, a, b) for a, b in zip(ref, mid)]
    else:
        assert alive is None
    assert_same_bits(got, ref, (name, pxf.last_trace_kernel()))
    if name in ("tracesphere", "tracecyl"):
        assert 0 < int(torch.isnan(mid[7]).sum()) < mid[7].shape[0]         # misses are part of the bundle
    if oop:
        assert_same_bits(rays, to_dev(h), "input left alone")


def test_fused_golden_flows_are_one_launch_each(pxf, golden):
    import torch
    g = golden("surfaces2")
    T, S = pxf.transformations, pxf.surfaces

    def parax(r):
        S.paraxial(r, 350.)
        S.paraxialY(r, -120.)

    def ws(r):
        S.wsPrimaryB(r, 220., 1.e4, 1., .4)
        T.reflect(r)
        S.wsSecondaryB(r, 220., 1.e4, 1., .4)
    flows = [("sphere_in", "sphere_out", lambda r: S.sphere(r, 250.)),
             ("tansphere_in", "tansphere_out", lambda r: S.tanSphere(r, -500., nr=1.5)),
             ("cyl_in", "cyl_out", lambda r: S.cyl(r, 100., nr=1.2)),
             ("cylconic_in", "cylconic_out", lambda r: S.cylconic(r, 1. / 400., -.7)),
             ("torus_in", "torus_out", lambda r: S.torus(r, 150., 900.)),
             ("paraxial_in", "paraxial_out", parax),
             ("wsback_in", "wsback_secondary", ws)]
    for key_in, key_out, flow in flows:
        plain = to_dev(rows_of(g[key_in]))
        flow(plain)
        dev = to_dev(rows_of(g[key_in]))
        torch.cuda.synchronize()
        before = pxf.launch_count()
        with pxf.fused(dev):
            flow(dev)
        assert pxf.launch_count() - before == 1, (key_in, pxf.last_trace_kernel())
        assert_same_bits(dev, plain, key_in)
        if key_in == "wsback_in":
            assert_close(to_host(dev), rows_of(g[key_out]), pos_scale=1.e4, tol=1e-11, what="wsPrimaryB/wsSecondaryB")
        else:
            assert_bit_equal(to_host(dev), rows_of(g[key_out]), what=key_in)
    # the W-S primary alone against its own fixture (1e-12)
    dev = to_dev(rows_of(g["wsback_in"]))
    with pxf.fused(dev):
        S.wsPrimaryB(dev, 220., 1.e4, 1., .4)
    assert_close(to_host(dev), rows_of(g["wsback_primary"]), pos_scale=1.e4, what="wsPrimaryB")


def test_check_true_still_flushes(pxf, golden):
    g = golden("surfaces2")
    S = pxf.surfaces
    dev = to_dev(rows_of(g["wsback_in"]))
    plain = to_dev(rows_of(g["wsback_in"]))
    S.wsPrimaryB(plain, 220., 1.e4, 1., .4)
    with pxf.fused(dev):
        same = S.wsPrimaryB(dev, 220., 1.e4, 1., .4, check=True)
        assert same is not None and same.shape[0] == dev[1].shape[0]
    assert_same_bits(dev, plain, "check=True")


@pytest.mark.parametrize("oop", [False, True], ids=["inplace", "oop"])
@pytest.mark.parametrize("family", sorted(SEG))
def test_segments_equal_per_segment_programs(pxf, family, oop):
    import torch
    make, key = SEG[family]
    progs = [make(pxf, k) for k in range(len(LAYOUT))]
    h = source(key, int(np.sum(LAYOUT)), seed=1)
    rays = to_dev(h)
    out = [torch.full_like(r, float("nan")) for r in rays] if oop else None
    seg = pxf.SegmentedProgram(progs, LAYOUT)
    torch.cuda.synchronize()
    before = pxf.launch_count()
    assert seg.run(rays, out=out) is None
    assert pxf.launch_count() - before == 1
    assert "surf" in pxf.last_trace_kernel() or "jit_chain_seg" in pxf.last_trace_kernel(), pxf.last_trace_kernel()
    got = out if oop else rays
    start = seg.seg_start
    for k, prog in enumerate(progs):
        a, b = int(start[k]), int(start[k + 1])
        if a == b:
            continue
        one = to_dev([r[a:b] for r in h])
        one_out = [torch.full_like(r, float("nan")) for r in one] if oop else None
        prog.run(one, out=one_out)
        want = one_out if oop else one
        for row in range(10):
            assert np.array_equal(bits(got[row][a:b]), bits(want[row])), (family, k, row)
    if oop:
        assert_same_bits(rays, to_dev(h), "input left alone")


@pytest.mark.parametrize("K", [1, 31, 1000])
def test_one_launch(pxf, K):
    import torch
    n = 200
    make, key = SEG["lens"]
    seg = pxf.SegmentedProgram([make(pxf, k) for k in range(K)], [n] * K)
    rays = to_dev(source(key, n * K, seed=3))
    seg.run([r.clone() for r in rays])                 # warm (module load, specialised kernel)
    torch.cuda.synchronize()
    before = pxf.launch_count()
    seg.run(rays)
    assert pxf.launch_count() - before == 1


def test_interpreter_and_specialised_kernel_give_the_same_bits():
    def run(env_extra):
        env = dict(os.environ)
        for k in ("PXF_JIT", "PXF_JIT_MIN_RAYS", "PXF_NO_SPECIALIZE"):
            env.pop(k, None)
        env.update(env_extra)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_surface_compare.py")], env=env,
                           capture_output=True, text=True, timeout=1500)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
        out = {}
        for line in p.stdout.splitlines():
            f = line.split()
            if len(f) == 3:
                out[f[0]] = (f[1], f[2])
        return out

    interp = run({"PXF_JIT": "0"})
    jit = run({"PXF_JIT_MIN_RAYS": "0", "PXF_JIT_VERBOSE": "1"})
    names = {"seg_%s_oop%d" % (f, o) for f in SEG for o in (0, 1)} | \
            {single_name(n, v) for n in SINGLE for v in (False, True)}
    assert set(interp) == set(jit) == names
    for name in names:
        assert interp[name][0] == jit[name][0], "%s: specialised kernel and interpreter differ" % name
        seg = name.startswith("seg")
        assert interp[name][1] == ("k_program_seg<surf>_(interpreter)" if seg else "k_program<surf>_(interpreter)"), \
            (name, interp[name][1])
        assert jit[name][1].startswith("pxf_jit_chain_seg<" if seg else "pxf_jit_chain<"), (name, jit[name][1])


@pytest.mark.parametrize("name", ["tracesphere", "paraxialy", "wssecondaryback"])
def test_host_trace_equals_device_program(pxf, name):
    h = source(SINGLE[name][2], 30_001, seed=5)
    prog = single_program(pxf, name)
    dev = to_dev(h)
    prog.run(dev)
    host = [np.array(r, copy=True) for r in h]
    pxf.host.trace(host, prog)
    assert_bit_equal(host, to_host(dev), what="host.trace " + name)
    # a closing flat leaves z and the normal constant: filled on the host, same bits
    p2 = pxf.Program().transform(-0., -0., .5, -0., -0., -0.).paraxial(350.).paraxialy(-120.).flat()
    h2 = source("paraxial_in", 10_001, seed=6)
    d2 = to_dev(h2)
    p2.run(d2)
    host2 = [np.array(r, copy=True) for r in h2]
    pxf.host.trace(host2, p2)
    assert_bit_equal(host2, to_host(d2), what="host.trace paraxial + flat")


def test_mixing_with_zernike_or_ll_flushes(pxf, golden):
    import torch
    T, S = pxf.transformations, pxf.surfaces
    ex = pxf.examples
    ro, ao = ex.zernike_orders(5)
    zc = ex.zernike_coeff(len(ro), 2) * 1e-3
    ax, az = ex.ll_orders(3)
    lc = ex.ll_coeff(len(ax), 7)
    h = source("sphere_in", 10_001, seed=8)
    h_ll = ll_source(10_001, seed=8)

    flows = {
        "sphere_then_zern": lambda r: (T.transform(r, 0, 0, 5., 0, 0, 0), S.sphere(r, 30.), T.refract(r, 1., 1.5),
                                       S.zernsurf(r, zc, 40., rorder=ro, aorder=ao), T.reflect(r), S.flat(r)),
        "zern_then_cyl": lambda r: (T.transform(r, 0, 0, 5., 0, 0, 0), S.zernsurf(r, zc, 40., rorder=ro, aorder=ao),
                                    T.reflect(r), S.cyl(r, 30., nr=1.2), S.flat(r, nr=1.)),
        "ll_then_paraxial": lambda r: (T.transform(r, 0, 0, -8400., 0, 0, 0),
                                       S.primaryLL(r, 220., 8400., 8500., 8400., .25, lc, ax, az), T.reflect(r),
                                       S.paraxial(r, 500.), S.flat(r)),
        "paraxial_then_ll": lambda r: (S.paraxial(r, 500.), T.transform(r, 0, 0, -8400., 0, 0, 0),
                                       S.primaryLL(r, 220., 8400., 8500., 8400., .25, lc, ax, az), T.reflect(r),
                                       S.flat(r)),
    }
    for name, flow in flows.items():
        hh = h_ll if "ll" in name else h
        plain = to_dev(hh)
        flow(plain)
        dev = to_dev(hh)
        torch.cuda.synchronize()
        before = pxf.launch_count()
        with pxf.fused(dev):
            flow(dev)
        assert pxf.launch_count() - before >= 2, name          # the program was split where the kinds meet
        # NaN rays (sphere misses) may differ in the NaN's sign: the existing ops behind the split (flat) do not pin it
        assert_bit_equal(to_host(dev), to_host(plain), what=name)
