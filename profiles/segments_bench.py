"""Per-segment analyses (``segments=``) against the Python loop over per-item calls they replace.

    python profiles/segments_bench.py [--scale S] [--out FILE]

Workloads (same seeded inputs for both paths; every timing ends in a device synchronise):
  W1  tolerance batch: K = 1000 realisations x 1e5 rays of config 1's chain (Wolter-I pair), each with a seeded rigid
      misalignment of the secondary (a transform before it, the inverse after); unweighted hpd + rmsCentroid each.
      Loop: one fused trace + hpd + rmsCentroid per realisation.  Segmented: one SegmentedProgram launch over the
      K x 1e5 bundle, hpd(segments=) and rmsCentroid(segments=).
  W2  config 2's field sweep, 31 x 1e7 rays: examples.config2_fast against examples.config2_sweep_fast.
  W3  config 5 (260 shells, 1.25e8 rays before vignetting): the weighted hpd of every shell, a loop over the shell
      slices of the compacted bundle against hpd(weights, segments=Segments.after(alive)).
  K   kernel scaling: segmented unweighted hpd of 1.25e8 rays split into 1, 31, 1000 and 1e5 segments against the
      single-bundle hpd of the same rays; algorithmic bytes (sums pass + collect pass: 2 x 16 B/ray) over time.
Each entry reports ms, rays/s, the libpxf launch-count delta and the device-to-host read-backs of one call.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.stdout.strip() else q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


def timed(fn, reps=3):
    """Best-of-reps wall time of fn() ending in a synchronise, its result and its launch-count delta."""
    import torch
    import pyxfocus_b200 as pxf
    fn()                                           # warm: module loads, attributes, allocator
    torch.cuda.synchronize()
    best, out, launches = None, None, None
    for _ in range(reps):
        torch.cuda.synchronize()
        l0 = pxf.launch_count()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        t = time.perf_counter() - t0
        launches = pxf.launch_count() - l0
        best = t if best is None else min(best, t)
    return best, out, launches


def entry(t, rays, launches, readbacks):
    return {"ms": 1e3 * t, "rays_per_s": rays / t, "launches": int(launches), "readbacks": int(readbacks)}


def w1(pxf, K, n):
    import torch
    from pyxfocus_b200._call import bundle_alloc
    ex, anal = pxf.examples, pxf.analyses
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(1)
    mis = np.column_stack([rng.normal(0., .05, K), rng.normal(0., .05, K), np.zeros(K),
                           rng.normal(0., 1e-4, K), rng.normal(0., 1e-4, K), np.zeros(K)])
    ex.seed(0)
    src = pxf.sources.subannulus(220., 220.6, 2 * np.pi, n, zhat=-1., device=dev)

    def prog(m):
        # transformations.transform negates its arguments; Program takes them as the kernel sees them
        return (pxf.Program().transform(0, 0, 8400., 0, 0, 0).wolterprimary(220., 8400., 1.).reflect()
                .transform(*(-m)).woltersecondary(220., 8400., 1.).itransform(*(-m)).reflect().flat())
    progs = [prog(mis[k]) for k in range(K)]
    work = bundle_alloc(n, dev)

    def loop():
        h, r = np.empty(K), np.empty(K)
        for k in range(K):
            for a, b in zip(work, src):
                a.copy_(b)
            progs[k].run(work)
            h[k], r[k] = anal.hpd(work), anal.rmsCentroid(work)
        return h, r
    big = bundle_alloc(K * n, dev)
    segs = pxf.Segments([n] * K, device=dev)
    sp = pxf.SegmentedProgram(progs, segs.sizes(), device=dev)

    def seg():
        for a, b in zip(big, src):
            a.view(K, n).copy_(b.unsqueeze(0).expand(K, n))
        sp.run(big)
        return anal.hpd(big, segments=segs), anal.rmsCentroid(big, segments=segs)
    tl, (hl, rl), ll = timed(loop, reps=1)
    ts, (hs, rs), ls = timed(seg, reps=3)
    return {"K": K, "rays_per_realisation": n, "loop": entry(tl, K * n, ll, 2 * K), "segmented": entry(ts, K * n, ls, 2),
            "max_rel_diff_hpd": float(np.max(np.abs(hs - hl) / np.abs(hl))),
            "max_rel_diff_rms": float(np.max(np.abs(rs - rl) / np.abs(rl)))}


def w2(pxf, n):
    import torch
    ex = pxf.examples
    dev = torch.device("cuda", 0)
    ap = ex.ws_aperture(ex.product_api(dev))
    arc = np.linspace(0., 30., 31)
    strip = lambda res: [{k: v for k, v in p.items() if k != "rays"} for p in res]   # noqa: E731
    tl, rl, ll = timed(lambda: strip(ex.config2_fast(n, arc, ap, rng="philox", device=dev)), reps=2)
    ts, rs, ls = timed(lambda: strip(ex.config2_sweep_fast(n, arc, ap, rng="philox", device=dev)), reps=2)
    worst = max(abs(q[k] - p[k]) / max(abs(p[k]), 40.) for p, q in zip(rl, rs) for k in ("f", "hpd", "rms", "hpd_scan", "rms_scan"))
    same = all(p["d2"] == q["d2"] and p["d3"] == q["d3"] for p, q in zip(rl, rs))
    # read-backs: per point 2 image-plane sums, 2 x (hpd + rms), 2 focusI sums = 8; segmented: the same 8 in all
    return {"rays_per_field_point": n, "field_points": 31, "loop": entry(tl, 31 * n, ll, 8 * 31),
            "segmented": entry(ts, 31 * n, ls, 8), "scan_offsets_equal": bool(same), "worst_rel_err_40mm_floor": worst}


def w3(pxf, n_per_shell, nshell=260):
    import torch
    from pyxfocus_b200._call import bundle_alloc, bundle_split
    ex, anal, conic, tran = pxf.examples, pxf.analyses, pxf.conicsolve, pxf.transformations
    dev = torch.device("cuda", 0)
    g = ex.nested_geometry(nshell)
    L, nodegap, N = g.L, g.nodegap, int(n_per_shell)
    per = [N] * len(g.r)
    aper, progs, wts = [], [], []
    prev = 0.
    for r, z in zip(g.r, g.z):             # examples.config5_fast's shells
        r, z = float(r), float(z)
        a0, a1 = float(conic.primrad(z + nodegap / 2., r, z)), float(conic.primrad(z + nodegap / 2. + L, r, z))
        aper.append((a0, a1, 0., -1.))
        wts.append((a1 ** 2 - a0 ** 2) * np.pi / 100. / N)
        progs.append(pxf.Program().transform(0, 0, z, 0, 0, 0).wolterprimary(r, z, 1.).kick(0., 0., -1.)
                     .reflect().woltersecondary(r, z, 1.).reflect()
                     .vignette_box(3, z - nodegap / 2. - L, z - nodegap / 2.)
                     .transform(0, 0, -(z - nodegap / 2 - L), 0, 0, 0).flat().vignette_rhogt(prev)
                     .transform(0, 0, -(-z + nodegap / 2 + L), 0, 0, 0).flat())
        prev = float(conic.secrad(z - nodegap / 2 - L, r, z)) + .4
    rays = bundle_alloc(N * len(per), dev, zero=True)
    pxf.sources.segments("annulus", aper, per, seed=0, out=rays)
    weights = torch.repeat_interleave(torch.as_tensor(np.array(wts), device=dev), N)
    alive = pxf.SegmentedProgram(progs, per, device=dev).run(rays)
    segs = pxf.Segments(per, device=dev).after(alive)
    mrays, (mw,) = tran.compact(rays, alive, extra=[weights])
    del rays
    views = bundle_split(mrays, list(segs.sizes()))
    wv = [mw[int(segs.start[k]):int(segs.start[k + 1])] for k in range(segs.nseg)]

    def loop():
        return np.array([anal.hpd(v, weights=w) if v[1].shape[0] else np.nan for v, w in zip(views, wv)])
    tl, hl, ll = timed(loop, reps=1)
    ts, hs, ls = timed(lambda: anal.hpd(mrays, weights=mw, segments=segs), reps=2)
    ok = np.isfinite(hl)
    # where the two differ, the reference's own arithmetic (numpy argsort / cumsum / argmin) decides which is right:
    # with one weight per shell, |cdf - .75| can tie between neighbouring ranks to the last bit
    from oracle import pyref
    diff = np.nonzero(ok & (np.abs(hs - hl) > 1e-9 * np.abs(hl)))[0]
    agree = {"loop": 0, "segmented": 0, "neither": 0}
    for k in diff[:20]:
        h = [v.cpu().numpy() for v in views[k]]
        o = pyref.hpd(h, weights=wv[k].cpu().numpy())
        agree["segmented" if abs(hs[k] - o) <= 1e-9 * abs(o) else ("loop" if abs(hl[k] - o) <= 1e-9 * abs(o) else "neither")] += 1
    return {"shells": nshell, "rays_traced": N * nshell, "rays_kept": int(mrays[1].shape[0]),
            "loop": entry(tl, mrays[1].shape[0], ll, nshell), "segmented": entry(ts, mrays[1].shape[0], ls, 1),
            "max_rel_diff": float(np.max(np.abs(hs[ok] - hl[ok]) / np.abs(hl[ok]))), "shells_differing": int(diff.size),
            "of_the_first_20_differing_the_numpy_reference_agrees_with": agree}


def kscale(pxf, num):
    import torch
    from pyxfocus_b200._call import bundle_alloc
    anal = pxf.analyses
    d = bundle_alloc(num, torch.device("cuda", 0), zero=True)
    gen = torch.Generator(device="cuda").manual_seed(0)
    d[1].normal_(generator=gen)
    d[2].normal_(generator=gen)
    out = {"rays": num}
    t, ref, l1 = timed(lambda: anal.hpd(d), reps=5)
    out["single_bundle_hpd"] = entry(t, num, l1, 1)
    out["single_bundle_hpd"]["algorithmic_GB_per_s"] = 2 * 16 * num / t / 1e9
    for nseg in (1, 31, 1000, 100000):
        sizes = np.full(nseg, num // nseg, dtype=np.int64)
        sizes[: num - int(sizes.sum())] += 1
        segs = pxf.Segments(sizes)
        t, h, ln = timed(lambda: anal.hpd(d, segments=segs), reps=5)
        e = entry(t, num, ln, 1)
        e["algorithmic_GB_per_s"] = 2 * 16 * num / t / 1e9
        if nseg == 1:
            e["equals_single_bundle_hpd"] = bool(h[0] == ref)
        out["segments_%d" % nseg] = e
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="multiply every ray count (rehearsal: e.g. 1e-3)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default="w1,w2,w3,k")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("segments_bench.py needs a CUDA device")
    import pyxfocus_b200 as pxf
    sc = a.scale
    res = {"info": device_info(), "scale": sc}
    todo = a.only.split(",")
    if "w1" in todo:
        res["W1"] = w1(pxf, max(2, int(1000 * min(sc, 1.))), max(1000, int(1e5 * sc)))
    if "w2" in todo:
        res["W2"] = w2(pxf, max(1000, int(1e7 * sc)))
    if "w3" in todo:
        res["W3"] = w3(pxf, max(100, int(1.25e8 / 260 * sc)))
    if "k" in todo:
        res["kernel_scaling"] = kscale(pxf, max(200000, int(1.25e8 * sc)))
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
