"""Per-segment analyses of a segmented bundle (``segments=``) against the oracle on every segment alone, the
exactness of the segmented HPD, its launch count, ``Segments.after`` and the one-bundle config 2 sweep."""
import os
import sys

import numpy as np
import pytest

from util import UploadedSources, pyref, random_bundle, to_dev

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from make_golden_configs import SIZES  # noqa: E402

# 0/1/2/3-ray segments, odd starts, both sides of the 8192-ray direct/bracket threshold
LAYOUT = [0, 1, 2, 3, 0, 5, 8191, 8192, 8193, 7, 30001, 0, 120003, 4]


@pytest.fixture(scope="module")
def pxf():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyxfocus_b200 as p
    return p


def bundle(sizes, seed=0, tweak=None):
    rays = random_bundle(int(np.sum(sizes)), seed=seed)
    rays[6] = -np.abs(rays[6]) - .5                # n bounded away from 0 for the image-plane sums
    if tweak is not None:
        tweak(rays)
    return rays


def slices(rays, sizes):
    start = np.concatenate([[0], np.cumsum(sizes)])
    return [[r[start[k]:start[k + 1]] for r in rays] for k in range(len(sizes))]


def radii_about(pxf, x, y, cx, cy):
    import torch
    from pyxfocus_b200 import _lib
    from pyxfocus_b200._call import stream_ptr
    x, y = torch.as_tensor(x, device="cuda"), torch.as_tensor(y, device="cuda")
    out = torch.empty_like(x)
    if x.shape[0]:
        _lib.check(_lib.lib().pxf_rho(x.data_ptr(), y.data_ptr(), x.shape[0], float(cx), float(cy), out.data_ptr(),
                                      stream_ptr(x.device)))
    return out.cpu().numpy()


def rel(a, b):
    return abs(a - b) / max(abs(b), 1e-300)


@pytest.mark.parametrize("weighted", [False, True])
def test_sums_match_oracle_per_segment(pxf, weighted):
    anal = pxf.analyses
    h = bundle(LAYOUT, seed=1)
    w = np.random.default_rng(2).uniform(.1, 2., h[1].shape[0]) if weighted else None
    d = to_dev(h)
    segs = pxf.Segments(LAYOUT)
    wd = None if w is None else w.copy()
    cx, cy = anal.centroid(d, weights=wd, segments=segs)
    rms = anal.rmsCentroid(d, weights=wd, segments=segs)
    rx, ry = anal.rmsX(d, weights=wd, segments=segs), anal.rmsY(d, weights=wd, segments=segs)
    ip = anal.analyticImagePlane(d, weights=wd, segments=segs)
    px, py = anal.analyticXPlane(d, weights=wd, segments=segs), anal.analyticYPlane(d, weights=wd, segments=segs)
    start = segs.start
    for k, sl in enumerate(slices(h, LAYOUT)):
        if LAYOUT[k] == 0:
            for v in (cx, cy, rms, rx, ry, ip, px, py):
                assert np.isnan(v[k])
            continue
        ws = None if w is None else w[start[k]:start[k + 1]]
        ocx, ocy = pyref.centroid(sl, weights=ws)
        assert abs(cx[k] - ocx) <= 1e-12 * 100. and abs(cy[k] - ocy) <= 1e-12 * 100., k
        assert rel(rms[k], pyref.rmsCentroid(sl, weights=ws)) <= 1e-9, k
        assert rel(rx[k], np.sqrt(np.average((sl[1] - np.average(sl[1], weights=ws)) ** 2, weights=ws))) <= 1e-9, k
        assert rel(ry[k], np.sqrt(np.average((sl[2] - np.average(sl[2], weights=ws)) ** 2, weights=ws))) <= 1e-9, k
        if LAYOUT[k] > 2:
            assert rel(ip[k], pyref.analyticImagePlane(sl, weights=ws)) <= 1e-9, k
            single = to_dev(sl)
            assert rel(px[k], anal.analyticXPlane(single, weights=ws)) <= 1e-9, k
            assert rel(py[k], anal.analyticYPlane(single, weights=ws)) <= 1e-9, k
    # deterministic: the same bits on a second call
    a = anal.imageplane_sums(d, weights=wd, at_z0=True, segments=segs).cpu().numpy()
    b = anal.imageplane_sums(d, weights=wd, at_z0=True, segments=segs).cpu().numpy()
    assert np.array_equal(a, b, equal_nan=True)


def test_zero_weight_segment_is_nan(pxf):
    anal = pxf.analyses
    sizes = [50, 60, 70]
    h = bundle(sizes, seed=3)
    w = np.ones(180)
    w[50:110] = 0.
    d = to_dev(h)
    segs = pxf.Segments(sizes)
    for v in (anal.centroid(d, weights=w, segments=segs)[0], anal.rmsCentroid(d, weights=w, segments=segs),
              anal.analyticImagePlane(d, weights=w, segments=segs), anal.hpd(d, weights=w, segments=segs),
              anal.findimageplane(d, 20., 100, weights=w, segments=segs)):
        assert np.isnan(v[1]) and not np.isnan(v[0]) and not np.isnan(v[2])


def test_findimageplane_per_segment_matches_single_bundle(pxf):
    anal = pxf.analyses
    sizes = [1000, 3, 20001, 777]
    h = bundle(sizes, seed=4)
    h[3] = h[3] * 0.                               # on the z = 0 plane
    d = to_dev(h)
    segs = pxf.Segments(sizes)
    s9 = anal.imageplane_sums(d, at_z0=True, segments=segs)
    d2 = anal.findimageplane(d, 20., 100, sums=s9, segments=segs)
    d3 = anal.findimageplane(d, 1., 100, sums=s9, moved=d2, segments=segs)
    for k, sl in enumerate(slices(h, sizes)):
        single = to_dev(sl)
        one = anal.imageplane_sums(single, at_z0=True)
        e2 = anal.findimageplane(single, 20., 100, sums=one)
        assert d2[k] == e2 and d3[k] == anal.findimageplane(single, 1., 100, sums=one, moved=e2), k


def check_hpd_exact(pxf, h, sizes, w=None):
    anal = pxf.analyses
    d = to_dev(h)
    segs = pxf.Segments(sizes)
    got = anal.hpd(d, weights=w, segments=segs)
    cx, cy = anal.centroid(d, weights=w, segments=segs)
    start = segs.start
    for k, sl in enumerate(slices(h, sizes)):
        if sizes[k] == 0:
            assert np.isnan(got[k])
            continue
        ws = None if w is None else w[start[k]:start[k + 1]]
        want = pyref.hpd(sl, weights=ws)
        if w is None:
            r = radii_about(pxf, sl[1], sl[2], cx[k], cy[k])
            ref = 2 * np.median(r)
            assert (np.isnan(got[k]) and np.isnan(ref)) or got[k] == ref, (k, got[k], ref)
        if np.isnan(want):
            assert np.isnan(got[k]), k
        else:
            assert abs(got[k] - want) <= 1e-9 * max(abs(want), 1e-300), (k, got[k], want)
    return d, segs, got


def test_hpd_unweighted_exact_on_many_layouts(pxf):
    check_hpd_exact(pxf, bundle(LAYOUT, seed=5), LAYOUT)


def test_hpd_unweighted_ties_cauchy_nan_and_empty(pxf):
    sizes = [20000, 0, 50001, 9000, 12, 0, 1]
    rng = np.random.default_rng(6)

    def tweak(r):
        r[1][:20000] = rng.integers(0, 5, 20000).astype(np.float64)            # many exact ties
        r[2][:20000] = rng.integers(0, 3, 20000).astype(np.float64)
        r[1][20000:70001] = rng.standard_cauchy(50001) * 10.                    # heavy tails
        r[2][20000:70001] = rng.standard_cauchy(50001) * 10.
        r[1][70001 + 4321] = np.nan                                             # a NaN in one segment only
    check_hpd_exact(pxf, bundle(sizes, seed=6, tweak=tweak), sizes)


def test_hpd_unweighted_overflowing_bracket_stays_exact(pxf):
    # 60 % of the middle segment at one point: its radii tie at the median, the bracket holds far more than the
    # candidate buffer takes, the segment is resolved by the exact fallback; its neighbours are not touched
    sizes = [30000, 100000, 30001]
    rng = np.random.default_rng(7)

    def tweak(r):
        a = 30000
        r[1][a:a + 60000] = 10.
        r[2][a:a + 60000] = 0.
        r[1][a + 60000:a + 100000] = 10. + rng.normal(0., 5., 40000)
        r[2][a + 60000:a + 100000] = rng.normal(0., 5., 40000)
    h = bundle(sizes, seed=7, tweak=tweak)
    d, segs, got = check_hpd_exact(pxf, h, sizes)
    raw = pxf.analyses._hpd_seg(d[1], d[2], None, segs, raw=True)
    assert np.array_equal(raw[:, 0], got)


def test_hpd_mode1_gives_the_same_bits(pxf):
    d = to_dev(bundle(LAYOUT, seed=8))
    segs = pxf.Segments(LAYOUT)
    a = pxf.analyses._hpd_seg(d[1], d[2], None, segs, mode=0)
    b = pxf.analyses._hpd_seg(d[1], d[2], None, segs, mode=1)
    assert np.array_equal(a, b, equal_nan=True)


def test_hpd_one_large_segment(pxf):
    sizes = [6_000_000]
    check_hpd_exact(pxf, bundle(sizes, seed=9), sizes)


def test_hpd_ten_thousand_small_segments(pxf):
    sizes = list(np.random.default_rng(10).integers(80, 121, 10000))
    check_hpd_exact(pxf, bundle(sizes, seed=10), sizes)


def test_hpd_weighted_matches_oracle(pxf):
    sizes = [0, 1, 2, 300, 9000, 20001, 5]
    h = bundle(sizes, seed=11)
    w = np.random.default_rng(12).uniform(.1, 3., h[1].shape[0])
    check_hpd_exact(pxf, h, sizes, w=w)


def test_hpd_launch_count_does_not_grow_with_segments(pxf):
    import torch
    d = to_dev(bundle([4096 * 300], seed=13))
    counts = []
    for sizes in ([4096 * 300], [300] * 4096):
        segs = pxf.Segments(sizes)
        pxf.analyses.hpd(d, segments=segs)                # warm (attributes, allocator)
        torch.cuda.synchronize()
        before = pxf.launch_count()
        pxf.analyses.hpd(d, segments=segs)
        counts.append(pxf.launch_count() - before)
    assert counts[0] == counts[1], counts


def test_segments_after_compaction(pxf):
    import torch
    tran, anal = pxf.transformations, pxf.analyses
    sizes = [0, 1000, 3, 9999, 20000, 1]
    h = bundle(sizes, seed=14)
    d = to_dev(h)
    segs = pxf.Segments(sizes)
    flags = np.random.default_rng(15).integers(0, 2, h[1].shape[0]).astype(np.uint8)
    alive = torch.as_tensor(flags, device="cuda")
    after = segs.after(alive)
    start = segs.start
    assert list(after.sizes()) == [int(flags[start[k]:start[k + 1]].sum()) for k in range(len(sizes))]
    comp = tran.compact(d, alive)
    got = anal.hpd(comp, segments=after)
    rms = anal.rmsCentroid(comp, segments=after)
    for k in range(len(sizes)):
        sl = [torch.as_tensor(np.ascontiguousarray(r[start[k]:start[k + 1]]), device="cuda") for r in h]
        own = tran.compact(sl, alive[start[k]:start[k + 1]].contiguous())
        one = pxf.Segments([own[1].shape[0]])
        for a, b in ((got[k], anal.hpd(own, segments=one)[0]), (rms[k], anal.rmsCentroid(own, segments=one)[0])):
            assert (np.isnan(a) and np.isnan(b)) or abs(a - b) <= 1e-12 * abs(b), (k, a, b)


def _c2_close(got, want):
    # bench.py's config 2 parity criterion: 1e-9 relative with a 40 mm floor
    return abs(got - want) / max(abs(want), 40.) <= 1e-9


def test_config2_sweep_matches_per_point_loop(pxf):
    ex = pxf.examples
    n = SIZES["c2_n"]
    arc = np.linspace(0., 30., 31)
    ap = ex.ws_aperture(ex.product_api())
    loop = ex.config2_fast(n, arc, ap)
    sweep = ex.config2_sweep_fast(n, arc, ap)
    assert len(loop) == len(sweep) == 31
    for a, p, q in zip(arc, loop, sweep):
        assert p["d2"] == q["d2"] and p["d3"] == q["d3"], a
        for k in ("f", "hpd", "rms", "hpd_scan", "rms_scan"):
            assert _c2_close(q[k], p[k]), (a, k, q[k], p[k])


def test_config2_sweep_matches_reference_golden(pxf):
    ex = pxf.examples
    g = np.load(os.path.join(ROOT, "tests", "golden", "configs.npz"))
    arc = [0., 5., 10.]
    res = ex.config2_sweep_fast(SIZES["c2_n"], arc, tuple(g["c2_aperture"]), sources=UploadedSources())
    for a, r in zip(arc, res):
        want = g["c2_%02d_scalars" % int(a)]
        assert r["d2"] == want[1] and r["d3"] == want[2], a
        assert abs(r["f"] - want[0]) <= 1e-9 * 1e4, a
        for got, w in ((r["hpd"], want[3]), (r["rms"], want[4]), (r["hpd_scan"], want[5]), (r["rms_scan"], want[6])):
            assert _c2_close(got, w), (a, got, w)
