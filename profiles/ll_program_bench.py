"""Legendre-Legendre shells as fused-program ops against the per-routine path they replace.

    python profiles/ll_program_bench.py [--scale S] [--reps R] [--out FILE]

Workloads (same seeded inputs for both paths; every timing ends in a device synchronise, after a warm-up call):
  P  trace only: the LL Wolter-I pair (transform, primaryLL, reflect, secondaryLL, reflect, flat) over 5e7 rays with
     every term up to order 5 on each mirror (36 terms), and again up to orders 3 (16 terms) and 7 (64 terms).  The
     five-launch sequence that ``fused`` ran before LL ops existed (transform | wolterprimll | reflect | woltersecll |
     reflect + flat) against ONE Program.run.  The first launch of the sequence and the program read the source
     bundle and write a second one, so every repetition does the same work; the results are compared bit for bit.
     The interpreter (PXF_JIT=0, registers capped for 1 CTA/SM) is timed once, in a child process.
  M  figure-error Monte Carlo: 1000 realisations x 1e5 rays (36 terms per mirror), trace + hpd + rmsCentroid each.
     The loop of examples.llpair_fast against examples.ll_tolerance_fast; ray counts and hpd / rms are compared.
Each entry reports the median and the spread (min, max) of R repetitions in ms, rays/s at the median, the libpxf
launch-count delta of one call and the kernel that traced.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
from zern_segments_bench import device_info, entry, timed  # noqa: E402

T_IN = (-0., -0., 8400., -0., -0., -0.)


def pair_terms(pxf, order):
    ex = pxf.examples
    ax, az = ex.ll_orders(order)
    return ex.ll_coeff(len(ax), 0), ex.ll_coeff(len(ax), 1), ax, az


def pair_case(pxf, src, out, work, order, reps, with_routines=True):
    import torch
    ex = pxf.examples
    cp, cs, ax, az = pair_terms(pxf, order)
    prog = ex.llpair_program(cp, cs, ax, az)
    num = src[1].shape[0]
    res = {"max_order": order, "terms_per_mirror": len(ax)}
    ts, _, launches = timed(lambda: prog.run(src, out=out), reps)
    res["program"] = entry(ts, num, launches, pxf.last_trace_kernel())
    if not with_routines:
        return res
    w = pxf.woltsurf
    head, mid, tail = pxf.Program().transform(*T_IN), pxf.Program().reflect(), pxf.Program().reflect().flat()

    def routines():
        head.run(src, out=work)
        w.wolterprimll(*work[1:], 220., 8400., 8500., 8400., .25, cp, ax, az)
        mid.run(work)
        w.woltersecll(*work[1:], 220., 8400., 1., 8400., 8300., .25, cs, ax, az)
        tail.run(work)
    ts, _, launches = timed(routines, reps)
    res["per_routine"] = entry(ts, num, launches)
    res["speedup_median"] = res["per_routine"]["ms_median"] / res["program"]["ms_median"]
    res["bits_equal"] = all(torch.equal(out[k].view(torch.int64), work[k].view(torch.int64)) for k in range(1, 10))
    return res


def trace(pxf, num, reps, with_routines=True):
    import torch
    from pyxfocus_b200._call import bundle_alloc
    dev = torch.device("cuda", 0)
    src = pxf.sources.subannulus(220., 220.6, .25, num, zhat=-1., rng="philox", seed=0, device=dev)
    out, work = bundle_alloc(num, dev), bundle_alloc(num, dev)
    return {"rays": num, "cases": [pair_case(pxf, src, out, work, order, reps, with_routines) for order in (5, 3, 7)]}


def interpreter(scale, reps):
    """P with the interpreter only, in a child process (PXF_JIT is read once per process)."""
    env = dict(os.environ, PXF_JIT="0")
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child-interp", "--scale", str(scale),
                        "--reps", str(reps)], env=env, capture_output=True, text=True, timeout=3000)
    if p.returncode != 0:
        return {"error": p.stderr[-2000:]}
    return json.loads(p.stdout.strip().splitlines()[-1])


def montecarlo(pxf, K, n, reps_loop, reps_seg):
    import torch
    ex = pxf.examples
    dev = torch.device("cuda", 0)
    ax, az = ex.ll_orders(5)
    real = [(ex.ll_coeff(36, 1000 + k), ex.ll_coeff(36, 2000 + k)) for k in range(K)]

    def loop():
        res = [ex.llpair_fast(n, cp, cs, ax, az, rng="philox", rng_seed=7, device=dev) for cp, cs in real]
        return [(int(r["rays"][1].shape[0]), r["hpd"], r["rms"]) for r in res]

    def seg():
        res = ex.ll_tolerance_fast(n, real, ax, az, rng="philox", rng_seed=7, device=dev)
        return [(int(r["rays"][1].shape[0]), r["hpd"], r["rms"]) for r in res]
    tl, rl, ll = timed(loop, reps_loop)
    kl = pxf.last_trace_kernel()
    ts, rs, ls = timed(seg, reps_seg)
    return {"realisations": K, "rays_per_realisation": n, "loop": entry(tl, K * n, ll),
            "segmented": entry(ts, K * n, ls), "loop_last_trace_kernel": kl,
            "speedup_median": float(np.median(tl) / np.median(ts)),
            "kept_equal": all(a[0] == b[0] for a, b in zip(rl, rs)),
            "max_rel_diff_hpd": max(abs(b[1] - a[1]) / abs(a[1]) for a, b in zip(rl, rs)),
            "max_rel_diff_rms": max(abs(b[2] - a[2]) / abs(a[2]) for a, b in zip(rl, rs))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1., help="multiplies every ray count (1 = the sizes above)")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child-interp", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    import torch
    import pyxfocus_b200 as pxf
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(0)
    if a.child_interp:
        r = trace(pxf, int(5e7 * a.scale), a.reps, with_routines=False)
        print(json.dumps({"cases": [{"max_order": c["max_order"], **c["program"]} for c in r["cases"]]}))
        return
    res = {"info": device_info()}
    res["P_trace"] = trace(pxf, int(5e7 * a.scale), a.reps)
    res["P_interpreter"] = interpreter(a.scale, a.reps)
    res["M_montecarlo"] = montecarlo(pxf, 1000, int(1e5 * a.scale), max(3, a.reps // 2), a.reps)
    res["jit_status"] = pxf.jit_status()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
