"""conicplus, legsurf, zernphase and the rotated Zernike surface as fused-program ops: a program gives the bits of the
stand-alone calls it replaces (with and without a vignette predicate, in place and out of place, every row the
stand-alone kernel loads or stores written), the conicplus / legsurf edge bundles give the oracle's bits on every path
(interpreter and specialised kernel, single and segmented, each pinned by its kernel name; host-buffer path), ``fused`` records the surfaces2 flows, the aspheric singlet and a Legendre plate behind a sphere into
one launch, segmented programs with per-segment tables give the bits of per-segment ``Program.run`` in one launch, and
forbidden mixes or radial orders above 7 flush and keep the stand-alone bits."""
import os
import subprocess
import sys

import numpy as np
import pytest

import surface_edge_cases as E
from table_surface_cases import G, PROGRAMS, SEGMENTED, add_op, call_surfaces, source, vig_hi
from util import assert_close, rows_of, to_dev, to_host

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EDGE = sorted(n for n, c in E.CASES.items() if c.routine in ("conicplus", "conicplusopd", "legsurf"))
# rows each op reads or writes: the LOAD | STORE of its stand-alone kernel (pxf_ops.cu; zernrot: OpZern)
R = {name: 1 << k for k, name in enumerate(["opd", "x", "y", "z", "l", "m", "n", "ux", "uy", "uz"])}
POS, DIR, NRM = R["x"] | R["y"] | R["z"], R["l"] | R["m"] | R["n"], R["ux"] | R["uy"] | R["uz"]
LOAD_STORE = {"conicplus": POS | DIR | NRM, "conicplusopd": POS | DIR | NRM | R["opd"],
              "legsurf": R["x"] | R["y"] | DIR, "zernphase": R["x"] | R["y"] | DIR | R["opd"], "zernrot": POS | DIR | NRM}


@pytest.fixture(scope="module")
def pxf():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyxfocus_b200 as p
    return p


def bits(t):
    return np.ascontiguousarray(np.asarray(t)).view(np.int64)


def assert_same_bits(got, want, what, rows=range(10)):
    for k in rows:
        assert np.array_equal(bits(got[k]), bits(want[k])), (what, k)


def assert_oracle_bits(got, want, what):
    """the oracle's bits, NaN for NaN: the oracle's NaNs carry the host's sign and payload, the device's its own"""
    for k in range(10):
        a, b = np.asarray(got[k]), np.asarray(want[k])
        na, nb = np.isnan(a), np.isnan(b)
        assert np.array_equal(na, nb), (what, k, int((na != nb).sum()))
        assert np.array_equal(bits(a)[~na], bits(b)[~nb]), (what, k)


def stand_alone(pxf, h, name):
    rays = to_dev(h)
    call_surfaces(pxf, rays, name)
    return to_host(rays)


# ------------------------------------------------------------------ each op against the stand-alone call
@pytest.mark.parametrize("oop", [False, True], ids=["inplace", "oop"])
@pytest.mark.parametrize("vig", [False, True], ids=["novig", "vig"])
@pytest.mark.parametrize("name", sorted(PROGRAMS))
def test_program_equals_stand_alone_call(pxf, name, vig, oop):
    import torch
    h = source(name, 20_001, seed=3)
    want = stand_alone(pxf, h, name)
    rays = to_dev(h)
    out = [torch.full_like(r, float("nan")) for r in rays] if oop else None
    alive = PROGRAMS[name](pxf, vig).run(rays, out=out)
    got = to_host(out if oop else rays)
    if vig:
        keep = np.abs(h[1]) < vig_hi(name)
        assert np.array_equal(alive.cpu().numpy(), keep.astype(np.uint8))
        assert 0 < keep.sum() < keep.size
        want = [np.where(keep, w, r) for w, r in zip(want, h)]      # a stopped ray keeps its state at the predicate
    else:
        assert alive is None
    kernel = pxf.last_trace_kernel()
    rows = range(10)
    if oop:
        # out of place, every row the program reads or writes is stored (the vignette reads x)
        rows = [k for k in range(10) if (LOAD_STORE[name] | (2 if vig else 0)) >> k & 1]
        assert_same_bits(to_host(rays), h, "input left alone")
    assert_same_bits(got, want, (name, kernel), rows)
    if oop:
        assert all(np.isnan(got[k]).all() for k in range(10) if k not in rows), "rows the program never touches"


# ------------------------------------------------------------------ oracle edges on every path
def edge_want(name, flat):
    case = E.CASES[name]
    inp, _ = E.bundle(name)
    want = [np.array(r, copy=True) for r in inp]
    E.oracle(case, want)
    if flat:
        E.oracle_flat(want)
    return inp, want


@pytest.mark.parametrize("flat", [False, True], ids=["alone", "flat"])
@pytest.mark.parametrize("name", EDGE)
def test_edge_cases_host_trace_vs_oracle(pxf, name, flat):
    """the 1000-iteration cap, the NaN root and the special values through the host-buffer path"""
    case = E.CASES[name]
    inp, want = edge_want(name, flat)
    p = getattr(pxf.Program(), case.routine)(*case.args)
    host = [np.array(r, copy=True) for r in inp]
    pxf.host.trace(host, p.flat() if flat else p)
    assert_oracle_bits(host, want, "host.trace %s flat=%d" % (name, flat))


def test_edge_cases_interpreter_and_specialised_kernel_vs_oracle(tmp_path):
    """the same edges on the interpreter and on the specialised kernel, single and segmented (three segments, the
    middle one empty): each in a process of its own, since PXF_JIT / PXF_JIT_MIN_RAYS are read once"""
    def run(tag, env_extra):
        env = dict(os.environ)
        for k in ("PXF_JIT", "PXF_JIT_MIN_RAYS", "PXF_NO_SPECIALIZE"):
            env.pop(k, None)
        env.update(env_extra)
        path = str(tmp_path / (tag + ".npz"))
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_table_surface_edges.py"), path], env=env,
                           capture_output=True, text=True, timeout=2400)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
        return np.load(path)

    for tag, res in (("interp", run("interp", {"PXF_JIT": "0"})), ("jit", run("jit", {"PXF_JIT_MIN_RAYS": "0"}))):
        for name in EDGE:
            for flat in (False, True):
                _, want = edge_want(name, flat)
                for seg in (False, True):
                    key = "%s_flat%d_seg%d" % (name, int(flat), int(seg))
                    kernel = str(res[key + "_kernel"])
                    expect = {("interp", False): "k_program<tabsurf>", ("interp", True): "k_program_seg<tabsurf>",
                              ("jit", False): "pxf_jit_chain<", ("jit", True): "pxf_jit_chain_seg<"}[(tag, seg)]
                    assert kernel.startswith(expect), (key, kernel)
                    got = [res["%s_row%d" % (key, k)] for k in range(10)]
                    assert_oracle_bits(got, want, "%s %s %s" % (tag, key, kernel))


def test_interpreter_and_specialised_kernel_agree(tmp_path):
    def run(env_extra):
        env = dict(os.environ)
        for k in ("PXF_JIT", "PXF_JIT_MIN_RAYS", "PXF_NO_SPECIALIZE"):
            env.pop(k, None)
        env.update(env_extra)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_table_surface_compare.py")], env=env,
                           capture_output=True, text=True, timeout=2400)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
        return [line.split() for line in p.stdout.splitlines() if line.strip()]

    interp, jit = run({"PXF_JIT": "0"}), run({"PXF_JIT_MIN_RAYS": "0"})
    assert len(interp) == len(jit) == 2 * len(PROGRAMS) + len(SEGMENTED)
    expect = {"conicplus": "tabsurf", "conicplusopd": "tabsurf", "legsurf": "tabsurf", "zernphase": "zphase",
              "zernrot": "zernike"}
    for (name, d_i, k_i), (name_j, d_j, k_j) in zip(interp, jit):
        assert name == name_j and d_i == d_j, (name, k_i, k_j)
        base = name[4:] if name.startswith("seg_") else name.rsplit("_vig", 1)[0]
        if name.startswith("seg_"):
            assert k_i == "k_program_seg<%s>_(interpreter)" % expect[base], (name, k_i)
            assert k_j.startswith("pxf_jit_chain_seg<"), (name, k_j)
        else:
            assert k_i == "k_program<%s>_(interpreter)" % expect[base], (name, k_i)
            assert k_j.startswith("pxf_jit_chain<"), (name, k_j)


# ------------------------------------------------------------------ fused recording
def fused_once(pxf, h, fn):
    rays = to_dev(h)
    n0 = pxf.launch_count()
    with pxf.fused(rays):
        fn(rays)
    return to_host(rays), pxf.launch_count() - n0


@pytest.mark.parametrize("name", ["conicplus", "conicplusopd", "legsurf", "zernphase", "zernrot", "asphere",
                                  "leg_behind_sphere"])
def test_fused_flows_are_one_launch(pxf, name):
    key = {"conicplus": "conicplus_in", "conicplusopd": "conicplus_in", "legsurf": "legsurf_in",
           "zernphase": "zernphase_in", "zernrot": "zernrot_in"}.get(name)
    h = rows_of(G[key]) if key else source(name, 3000, seed=5)
    got, launches = fused_once(pxf, h, lambda r: call_surfaces(pxf, r, name))
    assert launches == 1, name
    assert_same_bits(got, stand_alone(pxf, h, name), name)
    if name == "legsurf":
        assert_same_bits(got, rows_of(G["legsurf_out"]), "legSurf golden")
    if name == "zernphase":
        assert_close(got, rows_of(G["zernphase_out"]), pos_scale=20., what="zernphase golden")
    if name == "zernrot":
        assert_close(got, rows_of(G["zernrot_out"]), pos_scale=20., what="zernsurfrot golden")
    if name == "asphere":
        assert np.isfinite(got[1]).mean() > .5


def test_fused_conicplus_matches_the_golden_data(pxf):
    # the fixture was made with nr = 1.1 (tests/test_gpu_parity.py)
    got, launches = fused_once(pxf, rows_of(G["conicplus_in"]), lambda r: call_surfaces(pxf, r, "conicplusopd"))
    assert launches == 1
    assert_same_bits(got, rows_of(G["conicplus_out"]), "conicplus golden")


def test_forbidden_mixes_and_high_orders_flush(pxf):
    S, T = pxf.surfaces, pxf.transformations
    ro8, ao8 = pxf.examples.zernike_orders(8)
    c8 = pxf.examples.zernike_coeff(len(ro8), sigma=1e-7)
    flows = {
        "zernsurf+conicplus": (lambda r: (S.zernsurf(r, G["z_coeff"], 20., G["z_rorder"], G["z_aorder"]),
                                          T.transform(r, 0, 0, 1., 0, 0, 0), call_surfaces(pxf, r, "conicplus")), 2),
        "conicplus+zernphase": (lambda r: (call_surfaces(pxf, r, "conicplus"), call_surfaces(pxf, r, "zernphase")), 2),
        "zernphase+zernrot": (lambda r: (call_surfaces(pxf, r, "zernphase"), call_surfaces(pxf, r, "zernrot")), 2),
        "zernphase_order8": (lambda r: (S.flat(r), S.zernphase(r, c8, 20., 5.e-4, rorder=ro8, aorder=ao8),
                                        S.flat(r)), 3),
    }
    for what, (fn, nlaunch) in flows.items():
        h = rows_of(G["zernphase_in"])
        got, launches = fused_once(pxf, h, fn)
        assert launches == nlaunch, (what, launches)
        want = to_dev(h)
        fn(want)
        assert_same_bits(got, to_host(want), what)


# ------------------------------------------------------------------ segmented programs
@pytest.mark.parametrize("nseg", [1, 31, 1000])
@pytest.mark.parametrize("name", sorted(SEGMENTED))
def test_segmented_per_segment_tables(pxf, name, nseg):
    progs, sizes, key = SEGMENTED[name](pxf, nseg)
    if sum(sizes) == 0:
        sizes = [257] * nseg
    h = source(key, sum(sizes), seed=7)
    seg = pxf.SegmentedProgram(progs, sizes)
    rays = to_dev(h)
    n0 = pxf.launch_count()
    assert seg.run(rays) is None
    assert pxf.launch_count() - n0 == 1
    got = to_host(rays)
    start = np.concatenate([[0], np.cumsum(sizes)])
    for k in range(nseg) if nseg < 100 else list(range(0, nseg, 37)) + [nseg - 1]:
        a, b = int(start[k]), int(start[k + 1])
        if a == b:
            continue
        ref = to_dev([r[a:b] for r in h])
        progs[k].run(ref)
        assert_same_bits([g[a:b] for g in got], to_host(ref), "%s segment %d of %d" % (name, k, nseg))
    if nseg > 1:
        # the tables differ per segment: so do the results
        a, b, c = int(start[1]), int(start[2]), int(start[3])
        ref = to_dev([r[a:c] for r in h])
        progs[1].run(ref)
        assert not all(np.array_equal(bits(g[b:c]), bits(r[b - a:])) for g, r in zip(got, to_host(ref)))


def test_segment_table_outlives_its_programs(pxf):
    import gc
    progs, sizes, key = SEGMENTED["conicplus"](pxf, 31)
    h = source(key, sum(sizes), seed=8)
    want = to_dev(h)
    pxf.SegmentedProgram(progs, sizes).run(want)
    seg = pxf.SegmentedProgram(progs, sizes)
    del progs
    gc.collect()
    rays = to_dev(h)
    seg.run(rays)
    assert_same_bits(to_host(rays), to_host(want), "after the programs are gone")


def test_add_op_records_per_segment_values(pxf):
    p0, p1 = add_op(pxf.Program(), "zernrot", 0), add_op(pxf.Program(), "zernrot", 1)
    assert not np.array_equal(p0._tables[0].numpy(), p1._tables[0].numpy())
