"""radgratW and grat as fused-program ops: each op alone and inside a chain gives the bits of the stand-alone entry
points on the interpreter and on the specialised kernels, in place and out of place, at 0..3 and odd ray counts, with
edge rays and NaN / +-0 array entries (tests/run_grating_ops.py, one process per path); the stand-alone results at the
edges are the oracle's; ``fused`` records a grating with per-ray arrays into one launch with the unfused bits, while
``ind=`` calls keep running the masked stand-alone kernels; segmented programs read each segment's slice of the
arrays; and the spectrum example gives the bits of its calls made one by one."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


@pytest.fixture(scope="module")
def pxf():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyxfocus_b200 as p
    return p


def bits(t):
    a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
    return np.ascontiguousarray(a).view(np.int64)


def same_rays(a, b, what, rows=range(10)):
    """Bits, NaN for NaN (run_grating_ops.same; the oracle's NaNs also carry the host's sign)."""
    for k in rows:
        x, y = (t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t) for t in (a[k], b[k]))
        nx, ny = np.isnan(x), np.isnan(y)
        assert np.array_equal(nx, ny), "%s: row %d: NaN pattern differs" % (what, k)
        assert np.array_equal(bits(x)[~nx], bits(y)[~ny]), "%s: row %d differs" % (what, k)


@pytest.mark.parametrize("mode", ["interp", "jit"])
def test_ops_give_the_stand_alone_bits_on_each_path(mode, tmp_path):
    env = dict(os.environ, PXF_JIT_CACHE=str(tmp_path))
    env.update({"PXF_JIT": "0"} if mode == "interp" else {"PXF_JIT": "1", "PXF_JIT_MIN_RAYS": "0"})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_grating_ops.py"), mode], env=env,
                       capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "ok" in r.stdout


def test_edge_bundles_match_the_oracle(pxf):
    """radgratW calls libm (atan2, sincos): 1e-12 against the oracle, as every libm routine (DESIGN.md section 3).
    grat is algebraic: the oracle's bits, NaN for NaN."""
    import torch
    from oracle.f2py import transformationsf as O
    import run_grating_ops as G
    from pyxfocus_b200 import transformationsf as T
    num = 64
    src = G.source(num, 3, True)
    wave, order = G.arrays(num, 3, True)
    w, o = wave.cpu().numpy(), order.cpu().numpy()
    host = [r.cpu().numpy().copy() for r in src]
    O.radgratw(host[1], host[2], host[4], host[5], host[6], w, 2., -3.)
    dev = G.clone(src)
    pxf.Program().radgratw(wave, 2., -3.).run(dev)
    for k in range(10):
        # NaN where the oracle has NaN, infinities (the x = y = 0 rays divide by zero) and every unchanged row by their
        # bits, the finite direction cosines within 1e-12
        x, y = dev[k].cpu().numpy(), host[k]
        nx, ny, fin = np.isnan(x), np.isnan(y), np.isfinite(y)
        assert np.array_equal(nx, ny), ("radgratw program vs oracle: NaN pattern", k)
        exact = ~fin & ~ny if k in (4, 5, 6) else ~ny
        assert np.array_equal(bits(x)[exact], bits(y)[exact]), ("radgratw program vs oracle: bits", k)
        assert np.all(np.abs(x[fin] - y[fin]) <= 1e-12), ("radgratw program vs oracle: 1e-12", k)
    host = [r.cpu().numpy().copy() for r in dev]
    O.grat(host[1], host[2], host[4], host[5], host[6], 160., o, w)
    pxf.Program().grat(160., order, wave).run(dev)
    same_rays(dev, [torch.from_numpy(h) for h in host], "grat program vs oracle")
    alone = G.clone(src)
    T.radgratw(alone[1], alone[2], alone[4], alone[5], alone[6], wave, 2., -3.)
    T.grat(alone[1], alone[2], alone[4], alone[5], alone[6], 160., order, wave)
    same_rays(alone, dev, "stand-alone vs program")
    # the zeroing branch of grat and the y = 0 / x = y = 0 rays of radgratw were exercised
    assert (np.stack([host[4], host[5], host[6]])[:, 7] == 0).all() and np.isnan(host[6][:4]).any()


def fused_calls(pxf, rays, wave, order, ind=None):
    tran, surf = pxf.transformations, pxf.surfaces
    tran.transform(rays, 0, 0, -10., .01, .02, 0)
    surf.flat(rays)
    tran.radgrat(rays, 2., -3, wave, ind=ind)
    tran.grat(rays, 160., order, wave, ind=ind)
    tran.grat(rays, 150., -1, wave.cpu().numpy(), ind=ind)        # a scalar order and a host wave array
    tran.transform(rays, 1., -2., -5., 0, .01, -.03)
    surf.flat(rays)


@pytest.mark.parametrize("num", [1, 3, 1001, 200003])
def test_fused_records_one_launch_with_the_unfused_bits(pxf, num):
    import run_grating_ops as G
    src = G.source(num, 5, num >= 8)
    wave, order = G.arrays(num, 5, num >= 8)
    want = G.clone(src)
    fused_calls(pxf, want, wave, order)
    got = G.clone(src)
    before = pxf.launch_count()
    with pxf.fused(got):
        fused_calls(pxf, got, wave, order)
    assert pxf.launch_count() - before == 1
    same_rays(got, want, "fused vs unfused")


def test_ind_calls_keep_the_masked_stand_alone_kernels(pxf):
    import torch
    import run_grating_ops as G
    num = 3001
    src = G.source(num, 9, True)
    wave, order = G.arrays(num, 9, True)
    ind = torch.from_numpy(np.random.default_rng(1).random(num) < .5).to(src[1].device)
    want = G.clone(src)
    fused_calls(pxf, want, wave, order, ind=ind)
    got = G.clone(src)
    before = pxf.launch_count()
    with pxf.fused(got):
        fused_calls(pxf, got, wave, order, ind=ind)
    assert pxf.launch_count() - before >= 4          # the three masked gratings and the program around them
    same_rays(got, want, "ind= inside fused vs outside")
    # the size-1 wave array with ind= is broadcast, as the reference passes it whole
    a, b = G.clone(src), G.clone(src)
    pxf.transformations.radgrat(a, 2., -3, np.array([5.]), ind=ind)
    with pxf.fused(b):
        pxf.transformations.radgrat(b, 2., -3, np.array([5.]), ind=ind)
    same_rays(a, b, "size-1 wave with ind=")


def test_segmented_reads_each_segments_slice(pxf):
    """Also run on both paths by run_grating_ops.py; here on the default path, with a shared array and per-segment
    scalars."""
    import run_grating_ops as G
    from pyxfocus_b200._call import bundle_split
    sizes = [5, 2049, 0, 777, 3]
    num = sum(sizes)
    wave, order = G.arrays(num, 21, True)
    start = np.concatenate([[0], np.cumsum(sizes)])
    progs = [pxf.Program().flat().grat(160. + k, order, wave).radgratw(wave, 1. + .5 * k, 1. - k).flat()
             for k in range(len(sizes))]
    src = G.source(num, 21, True)
    got = G.clone(src)
    before = pxf.launch_count()
    pxf.SegmentedProgram(progs, sizes, device=src[1].device).run(got)
    assert pxf.launch_count() - before == 1
    want = G.clone(src)
    for k, part in enumerate(bundle_split(want, sizes)):
        lo, hi = int(start[k]), int(start[k + 1])
        if hi > lo:
            pxf.Program().flat().grat(160. + k, order[lo:hi], wave[lo:hi]).radgratw(wave[lo:hi], 1. + .5 * k,
                                                                                    1. - k).flat().run(part)
    same_rays(got, want, "segmented vs per-segment runs")


def test_arrays_of_another_bundle_are_refused(pxf):
    import run_grating_ops as G
    src = G.source(100, 1)
    wave, _ = G.arrays(99, 1)
    with pytest.raises(ValueError):
        pxf.Program().radgratw(wave, 2., -3).run(src)
    with pytest.raises(ValueError):
        pxf.SegmentedProgram([pxf.Program().radgratw(wave, 2., -3)] * 2, [50, 50], device=src[1].device)


def test_spectrum_example_matches_its_calls_one_by_one(pxf):
    from pyxfocus_b200 import examples as ex
    before = pxf.launch_count()
    f = ex.config4_spectrum_fast(300, 12, rng="philox")
    s = ex.config4_spectrum_fast(300, 12, rng="philox", fuse=False)
    same_rays(f["rays"], s["rays"], "spectrum example, fused vs call by call")
    assert f["dz"] == s["dz"] and f["rmsY"] == s["rmsY"]
    assert np.isfinite(f["rmsY"]) and f["rmsY"] > 0
    # the grating stage of the fused run is one launch: the SPO shells, the stage, then focusY / rmsY of both runs
    assert pxf.launch_count() - before > 0
    for k in (4, 5, 6):
        assert np.isfinite(f["rays"][k].cpu().numpy()).all()
