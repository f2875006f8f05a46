"""The remaining scalar surfaces at their edges, on every path that runs them, each against the C oracle (never against
another GPU path): the stand-alone kernels through the f2py-shaped modules (aligned double2 rows, unaligned rows,
mask= / index predicates, 0..3 rays), every fused-program op alone and followed by ``flat`` (in place and out of
place), the interpreter and the run-time specialised kernel in separate processes, segmented programs with
per-segment scalars at the edges, and the host-buffer path behind a closing ``flat``.  Bundles: tests/surface_edge_cases.py.

Algebraic routines agree bit for bit: 64-bit patterns including the sign of zero, NaN at the same rays (payloads not
compared).  The W-S back surfaces call libm per ray: 1e-12, positions relative to 1e4, unit vectors absolutely; NaN
patterns and the set of rays the 26-iteration cap restores are identical.  PXF_OPT_WS_LIBM = 1 evaluates the
reference's literal libm sequence correctly rounded and is compared with the oracle built the same way, at every field
angle.  The default (transcendental-free) evaluation is compared with the glibc oracle; at 15' the secondary is inside
the chaotic band below the graze angle (DESIGN.md section 3), where a 1-ulp change of one input row moves 211-2277 of the
oracle's own rays by more than 1e-12 and flips restored rays: there the default mode's rays beyond 1e-12 and its restored
set are bounded (measured on one B200: 238 of 50001 rays, 4 restored rays), not required to be identical."""
import os
import subprocess
import sys

import numpy as np
import pytest

import surface_edge_cases as E
from oracle import f2py as of
from util import ROWS, to_dev, to_host

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# rows each op stores (pxf_fused.cu op_masks); `flat` adds the position and the normal
R = {name: 1 << k for k, name in enumerate(ROWS)}
POS, DIR, NRM = R["x"] | R["y"] | R["z"], R["l"] | R["m"] | R["n"], R["ux"] | R["uy"] | R["uz"]
STORE = {"tracesphere": POS | DIR | NRM, "tracesphereopd": POS | DIR | NRM | R["opd"], "tracecyl": POS | DIR | NRM,
         "tracecylopd": POS | DIR | NRM | R["opd"], "cylconic": POS | NRM, "torus": POS | NRM,
         "paraxial": R["l"] | R["m"], "paraxialy": R["m"], "wsprimaryback": POS | NRM, "wssecondaryback": POS | NRM}


@pytest.fixture(scope="module")
def pxf():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyxfocus_b200 as p
    return p


def assert_same_bits(got, want, rows=range(10), what=""):
    for k in rows:
        a, b = np.asarray(got[k]), np.asarray(want[k])
        assert a.shape == b.shape, (what, ROWS[k])
        na, nb = np.isnan(a), np.isnan(b)
        if not np.array_equal(na, nb):
            i = int(np.flatnonzero(na != nb)[0])
            raise AssertionError("%s row %s: NaN pattern differs at %d rays, first %d: %r vs %r"
                                 % (what, ROWS[k], int((na != nb).sum()), i, a[i], b[i]))
        bad = np.flatnonzero((a.view(np.uint64) != b.view(np.uint64)) & ~na)
        if bad.size:
            i = int(bad[0])
            raise AssertionError("%s row %s: %d bit patterns differ, first at %d: %r vs %r"
                                 % (what, ROWS[k], bad.size, i, a[i], b[i]))


def restored(inp, out):
    return (inp[1] == out[1]) & (inp[2] == out[2]) & (inp[3] == out[3])


# default W-S evaluation in the chaotic band: (share of rays allowed beyond 1e-12, restored rays allowed to differ)
CHAOTIC = {"wssecondaryback_15": (.01, 8)}


def compare(case, got, want, inp, rows=range(10), what="", mode=0):
    """mode: the PXF_OPT_WS_LIBM mode the W-S rows were traced in (the oracle ``want`` must match it: oracle_out)"""
    if case.exact:
        assert_same_bits(got, want, rows, what)
        return
    share, nrest = CHAOTIC.get(case.name, (0., 0)) if mode == 0 else (0., 0)
    off = np.zeros(got[1].shape[0], bool)
    for k in rows:
        a, b = np.asarray(got[k]), np.asarray(want[k])
        na, nb = np.isnan(a), np.isnan(b)
        assert np.array_equal(na, nb), "%s row %s: NaN pattern differs (%d vs %d)" % (what, ROWS[k], na.sum(), nb.sum())
        off |= ~na & ~(np.abs(a - b) <= 1e-12 * (1.e4 if k < 4 else 1.))
    assert off.sum() <= share * off.size, "%s: %d of %d rays off by more than 1e-12" % (what, off.sum(), off.size)
    ndiff = int((restored(inp, got) != restored(inp, want)).sum())
    assert ndiff <= nrest, "%s: %d restored rays differ" % (what, ndiff)


def oracle_out(case, inp, mode=0):
    """the oracle's output; mode 1: the W-S oracle with correctly rounded libm (what PXF_OPT_WS_LIBM = 1 reproduces)"""
    want = [np.array(r, copy=True) for r in inp]
    if mode == 1:
        with of.libm("cr"):
            E.oracle(case, want)
    else:
        E.oracle(case, want)
    return want


def call_dev(pxf, case, rows, **kw):
    getattr(getattr(pxf, case.mod), case.routine)(*E.call_args(case, rows), **kw)


def ws_modes(case):
    """the W-S back surfaces in both evaluation modes, the algebraic routines once"""
    return (0, 1) if not case.exact else (None,)


class _ws_mode:
    def __init__(self, pxf, mode):
        self.pxf, self.mode = pxf, mode

    def __enter__(self):
        if self.mode is not None:
            self.pxf.set_option(self.pxf.OPT_WS_LIBM, self.mode)

    def __exit__(self, *a):
        if self.mode is not None:
            self.pxf.set_option(self.pxf.OPT_WS_LIBM, 0)


# ------------------------------------------------------------------ stand-alone kernels
@pytest.mark.parametrize("name", sorted(E.CASES))
def test_stand_alone_aligned(pxf, name):
    case = E.CASES[name]
    inp, _ = E.bundle(name)
    for mode in ws_modes(case):
        dev = to_dev(inp)
        assert dev[1].data_ptr() % 16 == 0
        with _ws_mode(pxf, mode):
            call_dev(pxf, case, dev)
        compare(case, to_host(dev), oracle_out(case, inp, mode or 0), inp, what="%s libm=%s" % (name, mode),
                mode=mode or 0)


@pytest.mark.parametrize("name", sorted(E.CASES))
def test_stand_alone_unaligned(pxf, name):
    import torch
    case = E.CASES[name]
    inp, _ = E.bundle(name)
    for mode in ws_modes(case):
        big = torch.zeros(10, E.N + 3, dtype=torch.float64, device="cuda")
        dev = [big[i, 1:E.N + 1] for i in range(10)]          # 8-byte offset: the one-ray-per-thread path
        for i in range(10):
            dev[i].copy_(torch.from_numpy(inp[i]))
        assert dev[1].data_ptr() % 16 == 8
        with _ws_mode(pxf, mode):
            call_dev(pxf, case, dev)
        compare(case, [d.cpu().numpy() for d in dev], oracle_out(case, inp, mode or 0), inp,
                what="%s unaligned libm=%s" % (name, mode), mode=mode or 0)
        assert float(big[:, 0].abs().sum()) == 0. and float(big[:, E.N + 1:].abs().sum()) == 0.


@pytest.mark.parametrize("name", sorted(E.CASES))
def test_stand_alone_masked(pxf, name):
    case = E.CASES[name]
    inp, _ = E.bundle(name)
    rng = np.random.default_rng(len(name))
    mask = rng.random(E.N) < .6
    mask[-1] = True
    for mode in ws_modes(case):
        # the oracle: gather, routine, scatter (the reference's ind= idiom)
        want = [np.array(r, copy=True) for r in inp]
        sub = oracle_out(case, [np.ascontiguousarray(r[mask]) for r in want], mode or 0)
        for r, s in zip(want, sub):
            r[mask] = s
        for kind, m in (("bool", mask), ("index", np.flatnonzero(mask))):
            dev = to_dev(inp)
            with _ws_mode(pxf, mode):
                call_dev(pxf, case, dev, mask=m)
            compare(case, to_host(dev), want, inp, what="%s mask=%s libm=%s" % (name, kind, mode), mode=mode or 0)


@pytest.mark.parametrize("name", sorted(E.CASES))
def test_stand_alone_tiny_bundles(pxf, name):
    case = E.CASES[name]
    inp, classes = E.bundle(name)
    # edge rays first: one of each class, then ordinary rays
    first = [int(v[0]) for v in classes.values()] + [0, 1, 2]
    for n in (0, 1, 2, 3):
        idx = np.array(first[:n], dtype=np.int64)
        small = [np.ascontiguousarray(r[idx]) for r in inp]
        want = oracle_out(case, small) if n else small
        dev = to_dev(small)
        call_dev(pxf, case, dev)
        compare(case, to_host(dev), want, small, what="%s n=%d" % (name, n))


# ------------------------------------------------------------------ program ops, alone and followed by flat
def op_program(pxf, case, flat):
    p = getattr(pxf.Program(), case.routine)(*case.args)
    return p.flat() if flat else p


def program_want(case, inp, flat):
    want = oracle_out(case, inp)
    if flat:
        E.oracle_flat(want)
    return want


@pytest.mark.parametrize("oop", [False, True], ids=["inplace", "oop"])
@pytest.mark.parametrize("flat", [False, True], ids=["alone", "flat"])
@pytest.mark.parametrize("name", E.PROGRAM)
def test_program_op_vs_oracle(pxf, name, flat, oop):
    """each op with no neighbour to load or overwrite a row for it: a row missing from the op's load mask or its store
    mask shows here; behind `flat` the position and normal are overwritten, the direction of a miss is not"""
    import torch
    case = E.CASES[name]
    inp, _ = E.bundle(name)
    want = program_want(case, inp, flat)
    rays = to_dev(inp)
    out = [torch.full_like(r, float("nan")) for r in rays] if oop else None       # a missing store shows
    assert op_program(pxf, case, flat).run(rays, out=out) is None
    got = to_host(out if oop else rays)
    stored = STORE[case.routine] | (POS | NRM if flat else 0)
    rows = [k for k in range(10) if stored >> k & 1] if oop else range(10)
    compare(case, got, want, inp, rows=rows, what="%s flat=%d oop=%d %s" % (name, flat, oop, pxf.last_trace_kernel()))
    if oop:
        assert_same_bits(to_host(rays), inp, what="input left alone")


# ------------------------------------------------------------------ interpreter and specialised kernel
def test_interpreter_and_specialised_kernel_vs_oracle(tmp_path):
    def run(tag, env_extra):
        env = dict(os.environ)
        for k in ("PXF_JIT", "PXF_JIT_MIN_RAYS", "PXF_NO_SPECIALIZE"):
            env.pop(k, None)
        env.update(env_extra)
        path = str(tmp_path / (tag + ".npz"))
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_surface_edges.py"), path], env=env,
                           capture_output=True, text=True, timeout=2400)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
        return np.load(path)

    results = {"interp": run("interp", {"PXF_JIT": "0"}), "jit": run("jit", {"PXF_JIT_MIN_RAYS": "0"})}
    for tag, res in results.items():
        for name in E.PROGRAM:
            case = E.CASES[name]
            for flat in (False, True):
                if flat and case.special:
                    continue
                key = "%s_flat%d" % (name, int(flat))
                kernel = str(res[key + "_kernel"])
                assert kernel.startswith("k_program<surf>" if tag == "interp" else "pxf_jit_chain<"), (key, kernel)
                inp, _ = E.bundle(name)
                got = [res["%s_row%d" % (key, k)] for k in range(10)]
                compare(case, got, program_want(case, inp, flat), inp, what="%s %s %s" % (tag, key, kernel))
        for family in sorted(E.SEG):
            key = "seg_" + family
            kernel = str(res[key + "_kernel"])
            assert kernel.startswith("k_program_seg<surf>" if tag == "interp" else "pxf_jit_chain_seg<"), (key, kernel)
            inp, _ = E.seg_bundle(family)
            want = [np.array(r, copy=True) for r in inp]
            E.seg_oracle(family, want)
            assert_same_bits([res["%s_row%d" % (key, k)] for k in range(10)], want, what="%s %s" % (tag, key))


# ------------------------------------------------------------------ segmented programs
@pytest.mark.parametrize("oop", [False, True], ids=["inplace", "oop"])
@pytest.mark.parametrize("family", sorted(E.SEG))
def test_segmented_edges_vs_oracle(pxf, family, oop):
    """per-segment scalars at the edges (radii at which a whole segment misses, F = -0, +-1e308, torus rays at the
    Newton cap) on the layout [0, 1, 2, 3, 2047, 2048, 2049, 0, 5001]: segment k against the oracle on its slice"""
    import torch
    inp, classes = E.seg_bundle(family)
    want = [np.array(r, copy=True) for r in inp]
    E.seg_oracle(family, want)
    progs = [E.SEG[family][1](pxf.Program, k) for k in range(len(E.LAYOUT))]
    seg = pxf.SegmentedProgram(progs, E.LAYOUT)
    rays = to_dev(inp)
    out = [torch.full_like(r, float("nan")) for r in rays] if oop else None
    assert seg.run(rays, out=out) is None
    got = to_host(out if oop else rays)
    store = {"sphere": STORE["tracesphereopd"], "paraxial": STORE["paraxial"], "torus": STORE["torus"]}[family]
    rows = [k for k in range(10) if store >> k & 1] if oop else range(10)
    start = np.concatenate([[0], np.cumsum(E.LAYOUT)])
    for k in range(len(E.LAYOUT)):
        a, b = int(start[k]), int(start[k + 1])
        assert_same_bits([g[a:b] for g in got], [w[a:b] for w in want], rows, what="%s segment %d" % (family, k))
    if family == "sphere":
        assert np.isnan(want[7][start[4]:start[5]]).all()          # a segment in which every ray misses
    if family == "torus":
        assert classes["cap"].size > 100


# ------------------------------------------------------------------ host-buffer path
@pytest.mark.parametrize("name", sorted(E.HOST))
def test_host_trace_closing_flat_then_op(pxf, name):
    """a closing flat leaves z and the normal constant; paraxial keeps them so (filled on the host, never downloaded),
    tracecyl / cylconic / tracesphere overwrite them (downloaded)"""
    key, make, _ = E.HOST[name]
    inp, _ = E.bundle(key)
    want = [np.array(r, copy=True) for r in inp]
    E.host_oracle(name, want)
    host = [np.array(r, copy=True) for r in inp]
    pxf.host.trace(host, make(pxf.Program))
    assert_same_bits(host, want, what="host.trace flat, " + name)
    assert np.isfinite(want[1]).mean() > .3
    if name == "tracesphere":
        assert np.isnan(want[7]).any()                              # misses behind the flat
