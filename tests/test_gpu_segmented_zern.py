"""Segmented programs with one Zernike surface per segment: every segment gives the bits ``Program.run`` gives on its
slice (interpreter and run-time specialised kernel alike), the Zernike routines agree with the C oracle, the whole
bundle is one launch, and ``examples.config3_tolerance_fast`` reproduces the loop of ``config3_fast(coeff=...)``."""
import os
import subprocess
import sys

import numpy as np
import pytest

from seg_zern_cases import CASES, LAYOUT, case_name, program, source, zern_nr, zern_table
from util import assert_close, of, to_dev

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


@pytest.mark.parametrize("chain,with_nr,oop", CASES, ids=[case_name(*c) for c in CASES])
def test_segments_equal_per_segment_programs(pxf, chain, with_nr, oop):
    import torch
    progs = [program(pxf, chain, k, with_nr) for k in range(len(LAYOUT))]
    h = source(chain, int(np.sum(LAYOUT)), seed=1)
    rays = to_dev(h)
    out = [torch.zeros_like(r) for r in rays] if oop else None
    seg = pxf.SegmentedProgram(progs, LAYOUT)
    alive = seg.run(rays, out=out)
    got = out if oop else rays
    start = seg.seg_start
    for k, prog in enumerate(progs):
        a, b = int(start[k]), int(start[k + 1])
        if a == b:
            continue
        one = to_dev([r[a:b] for r in h])
        one_out = [torch.zeros_like(r) for r in one] if oop else None
        one_alive = prog.run(one, out=one_out)
        want = one_out if oop else one
        for row in range(10):
            assert np.array_equal(bits(got[row][a:b]), bits(want[row])), (k, row, pxf.last_trace_kernel())
        if chain == "c3":
            assert torch.equal(alive[a:b], one_alive), k
            assert 0 < int(one_alive.sum()) < b - a or b - a < 10, k     # the predicates cut some rays
        else:
            assert alive is None and one_alive is None
    if oop:
        assert np.array_equal(bits(rays[1]), bits(to_dev(h)[1]))      # the input is left alone


def test_interpreter_and_specialised_kernel_give_the_same_bits():
    def run(env_extra):
        env = dict(os.environ)
        for k in ("PXF_JIT", "PXF_JIT_MIN_RAYS", "PXF_NO_SPECIALIZE"):
            env.pop(k, None)
        env.update(env_extra)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_seg_zern_compare.py")], env=env,
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
    assert set(interp) == set(jit) == {case_name(*c) for c in CASES}
    for name in interp:
        assert interp[name][0] == jit[name][0], "%s: specialised kernel and interpreter differ" % name
        assert interp[name][1] == "k_program_seg<zernike>_(interpreter)", (name, interp[name][1])
        assert jit[name][1].startswith("pxf_jit_chain_seg<"), (name, jit[name][1])


@pytest.mark.parametrize("with_nr", [False, True])
def test_zernike_segments_match_the_oracle(pxf, with_nr):
    sizes = [3000, 0, 2049, 5000, 4097]
    progs = [program(pxf, "tzr", k, with_nr) for k in range(len(sizes))]
    h = source("tzr", int(np.sum(sizes)), seed=2)
    d = to_dev(h)
    seg = pxf.SegmentedProgram(progs, sizes)
    seg.run(d)
    start = seg.seg_start
    for k, prog in enumerate(progs):
        a, b = int(start[k]), int(start[k + 1])
        if a == b:
            continue
        cpu = [np.ascontiguousarray(r[a:b]) for r in h]
        c, ro, ao, rad = zern_table(k)
        tp = prog.ops[0][1]
        of.transformationsf.transform(*cpu[1:], *tp)
        if with_nr:
            of.zernsurf.tracezernopd(*cpu, c, ro, ao, rad, zern_nr(k))
        else:
            of.zernsurf.tracezern(*cpu[1:], c, ro, ao, rad)
        of.transformationsf.reflect(*cpu[4:])
        assert_close([r[a:b].cpu().numpy() for r in d], cpu, pos_scale=100., tol=1e-12, what="segment %d" % k)


@pytest.mark.parametrize("K", [1, 31, 1000])
def test_one_launch(pxf, K):
    import torch
    n = 200
    progs = [program(pxf, "c3", k, True) for k in range(K)]
    seg = pxf.SegmentedProgram(progs, [n] * K)
    rays = to_dev(source("c3", n * K, seed=3))
    seg.run([r.clone() for r in rays])                 # warm (module load, specialised kernel)
    torch.cuda.synchronize()
    before = pxf.launch_count()
    seg.run(rays)
    assert pxf.launch_count() - before == 1


def test_tolerance_example_matches_the_loop(pxf):
    ex = pxf.examples
    n, K = 20_000, 12
    coeffs = [ex.zernike_coeff(36, 1000 + k) for k in range(K)]
    joint = ex.config3_tolerance_fast(n, coeffs, rng_seed=4)
    assert len(joint) == K
    for k, c in enumerate(coeffs):
        one = ex.config3_fast(n, rng_seed=4, coeff=c)
        assert joint[k]["rays"][1].shape[0] == one["rays"][1].shape[0], k
        assert np.array_equal(joint[k]["idx"].cpu().numpy(), one["idx"].cpu().numpy()), k
        for row in range(10):
            assert np.array_equal(bits(joint[k]["rays"][row]), bits(one["rays"][row])), (k, row)
        for key in ("hpd", "rms"):
            assert abs(joint[k][key] - one[key]) <= 1e-9 * abs(one[key]), (k, key, joint[k][key], one[key])
    # the realisations differ from one another
    assert len({round(r["hpd"], 12) for r in joint}) > 1


def test_config3_fast_default_coeff_is_unchanged(pxf):
    ex = pxf.examples
    a = ex.config3_fast(5000, rng_seed=5)
    b = ex.config3_fast(5000, rng_seed=5, coeff=ex.zernike_coeff(36, 5))
    for row in range(10):
        assert np.array_equal(bits(a["rays"][row]), bits(b["rays"][row])), row
    assert a["hpd"] == b["hpd"] and a["rms"] == b["rms"]
