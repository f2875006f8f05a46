"""Legendre-Legendre shells as fused-program ops: a program gives the bits of the per-routine calls it replaces (every
kind and order <= 7, with and without a vignette predicate, in place and out of place), ``fused`` records the reference
flow into one launch, segmented programs with differing orders and kinds give the bits of per-segment
``Program.run`` (interpreter and run-time specialised kernel alike) and agree with the C oracle, the whole bundle is
one launch, and ``examples.ll_tolerance_fast`` reproduces the loop of ``llpair_fast``."""
import os
import subprocess
import sys

import numpy as np
import pytest

from ll_cases import (LAYOUT, SINGLE, T_IN, ZCUT, routine, seg_program, seg_segment_routines, single_name,
                      single_program, source)
from util import assert_close, of, rows_of, to_dev, to_host

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
@pytest.mark.parametrize("kind,order,vig", SINGLE, ids=[single_name(*c) for c in SINGLE])
def test_program_equals_per_routine_calls(pxf, kind, order, vig, oop):
    import torch
    h = source(30_001, seed=3)
    prog = single_program(pxf, kind, order, vig)
    rays = to_dev(h)
    out = [torch.zeros_like(r) for r in rays] if oop else None
    alive = prog.run(rays, out=out)
    got = out if oop else rays
    ref = to_dev(h)
    tf = pxf.transformationsf
    tf.transform(*ref[1:], *T_IN)
    if kind == 1:
        pxf.woltsurf.wolterprimary(*ref[1:], 220., 8400., 1.)
        tf.reflect(*ref[4:])
    routine(pxf, ref[1:], kind, order, 10 * kind + order)
    tf.reflect(*ref[4:])
    # rows the program never touches are not written out of place (opd here); compare the nine it does
    for row in range(1, 10):
        assert np.array_equal(bits(got[row]), bits(ref[row])), (row, pxf.last_trace_kernel())
    if vig:
        lo, hi = ZCUT[kind]
        z = ref[3]
        want = ((z > lo) & (z < hi)).to(torch.uint8)
        assert torch.equal(alive, want)
        assert 0 < int(alive.sum()) < alive.shape[0]
    else:
        assert alive is None
    if oop:
        assert np.array_equal(bits(rays[3]), bits(to_dev(h)[3]))       # the input is left alone


def golden_flow(pxf, g, dev):
    T, S = pxf.transformations, pxf.surfaces
    coeff, axial, az = g["coeff"], g["axial"], g["az"]
    T.transform(dev, 0, 0, -8400., 0, 0, 0)
    S.primaryLL(dev, 220., 8400., 8500., 8400., .25, coeff, axial, az)
    T.reflect(dev)
    S.secondaryLL(dev, 220., 8400., 1., 8400., 8300., .25, coeff * .5, axial, az)
    T.reflect(dev)
    S.flat(dev)


def test_fused_golden_flow_is_one_launch_with_the_same_bits(pxf, golden):
    import torch
    g = golden("legendre")
    plain = to_dev(rows_of(g["rays_in"]))
    golden_flow(pxf, g, plain)
    dev = to_dev(rows_of(g["rays_in"]))
    torch.cuda.synchronize()
    before = pxf.launch_count()
    with pxf.fused(dev):
        golden_flow(pxf, g, dev)
    assert pxf.launch_count() - before == 1, pxf.last_trace_kernel()
    assert_same_bits(dev, plain, "fused vs per-routine")
    assert_close(to_host(dev), rows_of(g["rays_out"]), pos_scale=8.5e3, tol=1e-11, what="LL rays_out")
    assert pxf.analyses.hpd(dev) == pytest.approx(float(g["hpd"]), rel=1e-9)


def test_fused_ellipsoid_flow_matches_the_golden(pxf, golden):
    g = golden("legendre")
    T, S = pxf.transformations, pxf.surfaces
    coeff, axial, az = g["coeff"], g["axial"], g["az"]
    Sd = float(g["S"])

    def flow(dev):
        S.ellipsoidPrimaryLL(dev, 220., 8400., Sd, 1., 8500., 8400., .25, coeff, axial, az)
        T.reflect(dev)
        S.ellipsoidSecondaryLL(dev, 220., 8400., Sd, 1., 8400., 8300., .25, coeff * .5, axial, az)
        T.reflect(dev)
        S.flat(dev)
    plain = to_dev(rows_of(g["rays_in2"]))
    flow(plain)
    dev = to_dev(rows_of(g["rays_in2"]))
    before = pxf.launch_count()
    with pxf.fused(dev):
        flow(dev)
    assert pxf.launch_count() - before == 1
    assert_same_bits(dev, plain, "fused ellipsoid pair")
    assert_close(to_host(dev), rows_of(g["rays_out2"]), pos_scale=8.5e3, tol=1e-11, what="ellipsoid LL rays_out")


def test_fused_order_11_keeps_the_stand_alone_routine(pxf):
    T, S = pxf.transformations, pxf.surfaces
    axial = np.array([0, 1, 9, 11, 3])
    az = np.array([0, 2, 1, 4, 10])
    coeff = np.random.default_rng(5).normal(0, 1e-4, axial.size)
    h = source(10_000, seed=6)

    def flow(dev):
        T.transform(dev, 0, 0, -8400., 0, 0, 0)
        S.primaryLL(dev, 220., 8400., 8500., 8400., .25, coeff, axial, az)
        T.reflect(dev)
        S.flat(dev)
    plain = to_dev(h)
    flow(plain)
    dev = to_dev(h)
    with pxf.fused(dev):
        flow(dev)
    assert_same_bits(dev, plain, "order 11 inside fused")


@pytest.mark.parametrize("oop", [False, True], ids=["inplace", "oop"])
def test_segments_equal_per_segment_programs(pxf, oop):
    import torch
    progs = [seg_program(pxf, k) for k in range(len(LAYOUT))]
    h = source(int(np.sum(LAYOUT)), seed=1)
    rays = to_dev(h)
    out = [torch.zeros_like(r) for r in rays] if oop else None
    seg = pxf.SegmentedProgram(progs, LAYOUT)
    assert seg.run(rays, out=out) is None
    got = out if oop else rays
    start = seg.seg_start
    for k, prog in enumerate(progs):
        a, b = int(start[k]), int(start[k + 1])
        if a == b:
            continue
        one = to_dev([r[a:b] for r in h])
        one_out = [torch.zeros_like(r) for r in one] if oop else None
        prog.run(one, out=one_out)
        want = one_out if oop else one
        for row in range(10):
            assert np.array_equal(bits(got[row][a:b]), bits(want[row])), (k, row, pxf.last_trace_kernel())
    if oop:
        assert np.array_equal(bits(rays[1]), bits(to_dev(h)[1]))


def test_interpreter_and_specialised_kernel_give_the_same_bits():
    def run(env_extra):
        env = dict(os.environ)
        for k in ("PXF_JIT", "PXF_JIT_MIN_RAYS", "PXF_NO_SPECIALIZE"):
            env.pop(k, None)
        env.update(env_extra)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_ll_compare.py")], env=env,
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
    names = {"seg_oop0", "seg_oop1"} | {single_name(*c) for c in SINGLE}
    assert set(interp) == set(jit) == names
    for name in names:
        assert interp[name][0] == jit[name][0], "%s: specialised kernel and interpreter differ" % name
        seg = name.startswith("seg")
        assert interp[name][1] == ("k_program_seg<ll>_(interpreter)" if seg else "k_program<ll>_(interpreter)"), \
            (name, interp[name][1])
        assert jit[name][1].startswith("pxf_jit_chain_seg<" if seg else "pxf_jit_chain<"), (name, jit[name][1])


def test_ll_segments_match_the_oracle(pxf):
    sizes = [3000, 0, 2049, 5000, 4097, 1000]
    progs = [seg_program(pxf, k) for k in range(len(sizes))]
    h = source(int(np.sum(sizes)), seed=2)
    d = to_dev(h)
    seg = pxf.SegmentedProgram(progs, sizes)
    seg.run(d)
    start = seg.seg_start
    for k in range(len(sizes)):
        a, b = int(start[k]), int(start[k + 1])
        if a == b:
            continue
        cpu = [np.ascontiguousarray(r[a:b]) for r in h]
        seg_segment_routines(of, cpu, k)
        # segments with the ellipsoid primary (odd k) meet it with a plane wave, not the point source it is designed
        # for; through the pair and 8.4 m to the plane they agree to 1e-11, as the stand-alone routines do in
        # test_golden_legendre_shells
        tol = 1e-11 if k % 2 else 1e-12
        assert_close([r[a:b].cpu().numpy() for r in d], cpu, pos_scale=8.5e3, tol=tol, what="segment %d" % k)


@pytest.mark.parametrize("K", [1, 31, 1000])
def test_one_launch(pxf, K):
    import torch
    n = 200
    progs = [seg_program(pxf, k) for k in range(K)]
    seg = pxf.SegmentedProgram(progs, [n] * K)
    rays = to_dev(source(n * K, seed=3))
    seg.run([r.clone() for r in rays])                 # warm (module load, specialised kernel)
    torch.cuda.synchronize()
    before = pxf.launch_count()
    seg.run(rays)
    assert pxf.launch_count() - before == 1


def test_tolerance_example_matches_the_loop(pxf):
    ex = pxf.examples
    n, K = 20_000, 12
    axial, az = ex.ll_orders(5)
    real = [(ex.ll_coeff(36, 1000 + k), ex.ll_coeff(36, 2000 + k)) for k in range(K)]
    joint = ex.ll_tolerance_fast(n, real, axial, az, rng_seed=4)
    assert len(joint) == K
    for k, (cp, cs) in enumerate(real):
        one = ex.llpair_fast(n, cp, cs, axial, az, rng_seed=4)
        assert joint[k]["rays"][1].shape[0] == one["rays"][1].shape[0] == n, k
        for row in range(10):
            assert np.array_equal(bits(joint[k]["rays"][row]), bits(one["rays"][row])), (k, row)
        for key in ("hpd", "rms"):
            assert abs(joint[k][key] - one[key]) <= 1e-9 * abs(one[key]), (k, key, joint[k][key], one[key])
    assert len({round(r["hpd"], 12) for r in joint}) > 1
