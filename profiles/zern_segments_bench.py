"""Segmented programs with one Zernike surface per segment against the per-program path they replace.

    python profiles/zern_segments_bench.py [--scale S] [--reps R] [--out FILE]

Workloads (same seeded inputs for both paths; every timing ends in a device synchronise, after a warm-up call):
  T  trace only: config 3's 14-op program (Zernike surface, Wolter-I pair, three vignette predicates) over 5e7 rays,
     as 1, 31, 1000 and 25 000 segments, each segment with its own 36-term figure realisation (25 000 segments =
     2000 rays each, below the 2048-ray tile: segments change inside tiles).  Against ONE Program.run of one such
     program over the same 5e7 rays.  Both out of place (the source bundle is read, a second bundle written), so
     every repetition does the same work.
  W  figure-error Monte Carlo: 1000 realisations x 1e5 rays, trace + compaction + hpd + rmsCentroid each.  The loop
     of examples.config3_fast(coeff=c_k) against examples.config3_tolerance_fast(coeffs); the kept counts and the
     hpd / rms of the two are compared in the same run.
Each entry reports the median and the spread (min, max) of R repetitions in ms, rays/s at the median, the libpxf
launch-count delta of one call and the kernel that traced.
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


def timed(fn, reps):
    """Wall times of reps calls of fn(), each ending in a synchronise (after one warm-up call), the last result and
    the launch-count delta of one call."""
    import torch
    import pyxfocus_b200 as pxf
    fn()
    torch.cuda.synchronize()
    ts, out, launches = [], None, None
    for _ in range(reps):
        torch.cuda.synchronize()
        l0 = pxf.launch_count()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
        launches = pxf.launch_count() - l0
    return ts, out, launches


def entry(ts, rays, launches, kernel=None):
    med = float(np.median(ts))
    e = {"ms_median": 1e3 * med, "ms_min": 1e3 * min(ts), "ms_max": 1e3 * max(ts), "reps": len(ts),
         "rays_per_s": rays / med, "launches": int(launches)}
    if kernel is not None:
        e["kernel"] = kernel
    return e


def trace(pxf, num, nsegs, reps):
    import torch
    from pyxfocus_b200._call import bundle_alloc
    ex = pxf.examples
    dev = torch.device("cuda", 0)
    src = pxf.sources.subannulus(220., 220.6, 100. / 220., num, zhat=-1., rng="philox", seed=0, device=dev)
    out = bundle_alloc(num, dev)
    alive = torch.empty(num, dtype=torch.uint8, device=dev)
    one = ex.config3_program(ex.zernike_coeff(36, 0))
    ts, _, launches = timed(lambda: one.run(src, alive=alive, out=out), reps)
    res = {"rays": num, "single_program": entry(ts, num, launches, pxf.last_trace_kernel()), "segmented": []}
    base = float(np.median(ts))
    for K in nsegs:
        sizes = [len(a) for a in np.array_split(np.arange(num), K)]
        t0 = time.perf_counter()
        sp = pxf.SegmentedProgram([ex.config3_program(ex.zernike_coeff(36, k)) for k in range(K)], sizes, device=dev)
        setup = time.perf_counter() - t0
        ts, _, launches = timed(lambda: sp.run(src, alive=alive, out=out), reps)
        e = entry(ts, num, launches, pxf.last_trace_kernel())
        e.update(segments=K, rays_per_segment_min=int(min(sizes)), table_mb=sp.table_host.numel() / 2 ** 20,
                 host_setup_s=setup, vs_single_program=float(np.median(ts)) / base)
        res["segmented"].append(e)
        del sp
    return res


def montecarlo(pxf, K, n, reps_loop, reps_seg):
    import torch
    ex = pxf.examples
    dev = torch.device("cuda", 0)
    coeffs = [ex.zernike_coeff(36, 1000 + k) for k in range(K)]

    def loop():
        res = [ex.config3_fast(n, rng="philox", rng_seed=7, device=dev, coeff=c) for c in coeffs]
        return [(int(r["rays"][1].shape[0]), r["hpd"], r["rms"]) for r in res]

    def seg():
        res = ex.config3_tolerance_fast(n, coeffs, rng="philox", rng_seed=7, device=dev)
        return [(int(r["rays"][1].shape[0]), r["hpd"], r["rms"]) for r in res]
    tl, rl, ll = timed(loop, reps_loop)
    ts, rs, ls = timed(seg, reps_seg)
    return {"realisations": K, "rays_per_realisation": n, "loop": entry(tl, K * n, ll), "segmented": entry(ts, K * n, ls),
            "speedup_median": float(np.median(tl) / np.median(ts)),
            "kept_equal": all(a[0] == b[0] for a, b in zip(rl, rs)),
            "max_rel_diff_hpd": max(abs(b[1] - a[1]) / abs(a[1]) for a, b in zip(rl, rs)),
            "max_rel_diff_rms": max(abs(b[2] - a[2]) / abs(a[2]) for a, b in zip(rl, rs))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1., help="multiplies every ray count (1 = the sizes above)")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import pyxfocus_b200 as pxf
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(0)
    res = {"info": device_info()}
    res["T_trace"] = trace(pxf, int(5e7 * a.scale), [1, 31, 1000, 25000], a.reps)
    res["W_montecarlo"] = montecarlo(pxf, 1000, int(1e5 * a.scale), max(3, a.reps // 2), a.reps)
    res["jit_status"] = pxf.jit_status()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
