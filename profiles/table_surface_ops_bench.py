"""conicplus, legsurf, zernphase and the rotated Zernike surface as fused-program ops against the launch sequence
``fused`` ran before they were ops.

    python profiles/table_surface_ops_bench.py [--scale S] [--reps R] [--out FILE]

Workloads (same seeded inputs for every path; every timing ends in a device synchronise, after a warm-up call; old and
new paths are timed in alternating rounds within one process):
  C  four chains over 5e7 rays, out of place:
       asphere   transform, tracesphere, refract, transform, conicplus (8 terms), refract, transform, flat
       legsurf   transform, flat, legsurf (48 terms), transform, flat
       zernphase transform, flat, zernphase (36 terms), transform, flat
       zernrot   transform, zernsurfrot (36 + 10 terms), reflect, transform, flat
     Three ways:
       launches     what ``fused`` ran before: a program (the ops before) | the stand-alone routine | a program (the
                    ops after).  The first launch reads the source bundle and writes a second one.
       program      ONE Program.run, out of place (the run-time specialised kernel)
       interpreter  the same Program.run in a child process with PXF_JIT=0
     The rays come from the surfaces2.npz fixture bundle of each routine (drawn with replacement, positions jittered
     by ~1 um).  Results are compared bit for bit.
  S  segmented: 1000 segments x 1e5 rays, once with per-segment conicplus coefficients and once with a per-segment
     rot of the rotated Zernike surface: ONE SegmentedProgram.run against the loop of per-segment Program.run, out of
     place, compared bit for bit.
Each entry reports the median and the spread (min, max) in ms, rays/s at the median, the libpxf launch-count delta of
one call and the kernel that traced.
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
from surface_ops_bench import source  # noqa: E402
from zern_segments_bench import device_info, entry, timed  # noqa: E402

G = np.load(os.path.join(ROOT, "tests", "golden", "surfaces2.npz"))
RO, AO = G["z_rorder"], G["z_aorder"]          # 36 terms, radial orders <= 7
ASPH = np.array([(-1.) ** j * 10. ** (-6 - 3 * j) for j in range(8)])
LEG48 = (25., 30., 2., np.random.default_rng(5).normal(0., 1e-5, 48), np.arange(48) % 8, np.arange(48) // 8)


def rot_terms(P, rot):
    return P.tracezernrot(G["z_coeff"], RO, AO, G["z_coeff2"], RO[:10], AO[:10], 20., rot)


# name: (fixture, ops before, the op as a Program method, its stand-alone call on a bundle, ops after)
def chains(pxf):
    S = pxf.surfaces
    return {
        "asphere": ("conicplus_in",
                    lambda P: P.transform(0, 0, 0, 0, 0, 0).tracesphere(-900.).refract(1., 1.5).transform(0, 0, 2., 0, 0, 0),
                    lambda P: P.conicplus(800., -1.3, ASPH),
                    lambda r: S.conicplus(r, 800., -1.3, ASPH),
                    lambda P: P.refract(1.5, 1.).transform(0, 0, 50., 0, 0, 0).flat()),
        "legsurf": ("legsurf_in", lambda P: P.transform(0, 0, .1, 0, 0, 0).flat(),
                    lambda P: P.legsurf(*LEG48), lambda r: S.legSurf(r, *LEG48),
                    lambda P: P.transform(0, 0, 5., 0, 0, 0).flat()),
        "zernphase": ("zernphase_in", lambda P: P.transform(0, 0, .1, 0, 0, 0).flat(),
                      lambda P: P.zernphase(G["z_coeff"], RO, AO, 20., 5.e-4),
                      lambda r: S.zernphase(r, G["z_coeff"], 20., 5.e-4, rorder=RO, aorder=AO),
                      lambda P: P.transform(0, 0, 5., 0, 0, 0).flat()),
        "zernrot": ("zernrot_in", lambda P: P.transform(0, 0, 0, 0, 0, 0),
                    lambda P: rot_terms(P, .37),
                    lambda r: S.zernsurfrot(r, G["z_coeff"], G["z_coeff2"], 20., .37, rorder1=RO, aorder1=AO,
                                            rorder2=RO[:10], aorder2=AO[:10]),
                    lambda P: P.reflect().transform(0, 0, 5., 0, 0, 0).flat()),
    }


def alternate(fns, reps, rounds=4):
    """time each of fns in turn, rounds times, reps // rounds calls each: {index: (times, launch delta)}"""
    out = {k: ([], 0) for k in range(len(fns))}
    for _ in range(rounds):
        for k, fn in enumerate(fns):
            ts, _, launches = timed(fn, max(1, reps // rounds))
            out[k] = (out[k][0] + ts, launches)
    return out


def bits_equal(a, b):
    import torch
    return all(torch.equal(a[k].view(torch.int64), b[k].view(torch.int64)) for k in range(10))


def start_from(src, *bundles):
    """rows a path does not write keep the source's values, so whole bundles compare"""
    for b in bundles:
        for k in range(10):
            b[k].copy_(src[k])


def chain_case(pxf, spec, num, reps, interp_only=False):
    import torch
    from pyxfocus_b200._call import bundle_alloc
    key, before, op, call, after = spec
    dev = torch.device("cuda", 0)
    src = source(pxf, key, num, seed=11)
    out = bundle_alloc(num, dev)
    prog = after(op(before(pxf.Program())))

    def one():
        prog.run(src, out=out)
    if interp_only:
        ts, _, launches = timed(one, reps)
        return {"program": entry(ts, num, launches, pxf.last_trace_kernel())}
    work = bundle_alloc(num, dev)
    head, tail = before(pxf.Program()), after(pxf.Program())

    def launches_seq():
        head.run(src, out=work)
        call(work)
        tail.run(work)
    start_from(src, out, work)
    one()
    launches_seq()
    res = {"bits_equal": bits_equal(out, work)}
    one()
    kernel = pxf.last_trace_kernel()
    t = alternate([launches_seq, one], reps)
    res["launches"] = entry(t[0][0], num, t[0][1])
    res["program"] = entry(t[1][0], num, t[1][1], kernel)
    res["speedup_median"] = res["launches"]["ms_median"] / res["program"]["ms_median"]
    return res


def seg_programs(pxf, which, K):
    P = pxf.Program
    if which == "conicplus":
        return [P().transform(0, 0, 0, 0, 0, 0).conicplus(800., -1.3, ASPH * (1. + .001 * k)).refract(1., 1.5)
                .transform(0, 0, 50., 0, 0, 0).flat() for k in range(K)], "conicplus_in"
    return [rot_terms(P().transform(0, 0, 0, 0, 0, 0), .37 + .001 * k).reflect().transform(0, 0, 5., 0, 0, 0).flat()
            for k in range(K)], "zernrot_in"


def segmented(pxf, which, K, n, reps, interp_only=False):
    import torch
    from pyxfocus_b200._call import bundle_alloc
    dev = torch.device("cuda", 0)
    num = K * n
    progs, key = seg_programs(pxf, which, K)
    src = source(pxf, key, num, seed=12)
    out = bundle_alloc(num, dev)
    seg = pxf.SegmentedProgram(progs, [n] * K)

    def one():
        seg.run(src, out=out)
    if interp_only:
        ts, _, launches = timed(one, reps)
        return {"segmented": entry(ts, num, launches, pxf.last_trace_kernel())}
    work = bundle_alloc(num, dev)
    views_in = [[r[k * n:(k + 1) * n] for r in src] for k in range(K)]
    views_out = [[r[k * n:(k + 1) * n] for r in work] for k in range(K)]

    def loop():
        for k in range(K):
            progs[k].run(views_in[k], out=views_out[k])
    start_from(src, out, work)
    one()
    kernel = pxf.last_trace_kernel()
    loop()
    loop_kernel = pxf.last_trace_kernel()
    res = {"segments": K, "rays_per_segment": n, "bits_equal": bits_equal(out, work)}
    t = alternate([loop, one], max(4, reps // 2))
    res["loop"] = entry(t[0][0], num, t[0][1], loop_kernel)
    res["segmented"] = entry(t[1][0], num, t[1][1], kernel)
    res["speedup_median"] = res["loop"]["ms_median"] / res["segmented"]["ms_median"]
    return res


def interpreter(scale, reps):
    """C and S with the interpreter only (PXF_JIT=0 is read once per process: a child process)"""
    env = dict(os.environ, PXF_JIT="0")
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child-interp", "--scale", str(scale),
                        "--reps", str(reps)], env=env, capture_output=True, text=True, timeout=3000)
    if p.returncode != 0:
        return {"error": p.stderr[-2000:]}
    return json.loads(p.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1., help="multiplies every ray count (1 = the sizes above)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child-interp", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    import torch
    import pyxfocus_b200 as pxf
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(0)
    num, n = int(5e7 * a.scale), int(1e5 * a.scale)
    spec = chains(pxf)
    if a.child_interp:
        r = {name: chain_case(pxf, s, num, a.reps, interp_only=True)["program"] for name, s in spec.items()}
        for which in ("conicplus", "rot"):
            r["segmented_" + which] = segmented(pxf, which, 1000, n, a.reps, interp_only=True)["segmented"]
        print(json.dumps(r))
        return
    res = {"info": device_info(), "rays": num}
    res["C_chains"] = {name: chain_case(pxf, s, num, a.reps) for name, s in spec.items()}
    res["S_segmented"] = {which: segmented(pxf, which, 1000, n, a.reps) for which in ("conicplus", "rot")}
    res["interpreter"] = interpreter(a.scale, a.reps)
    res["jit_status"] = pxf.jit_status()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
