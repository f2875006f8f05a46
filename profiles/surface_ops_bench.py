"""The remaining scalar surfaces (sphere, cylinder, cylconic, paraxial lenses, torus, W-S back surfaces) as
fused-program ops against the launch sequence ``fused`` ran before they were ops.

    python profiles/surface_ops_bench.py [--scale S] [--reps R] [--out FILE]

Workloads (same seeded inputs for every path; every timing ends in a device synchronise, after a warm-up call):
  O  per op, trace only over 5e7 rays, out of place: transform, the op, refract (reflect behind the mirrors),
     transform, flatopd.  Three ways:
       launches     what ``fused`` ran before: a program (transform) | the stand-alone routine | a program (refract,
                    transform, flatopd).  The first launch reads the source bundle and writes a second one, so every
                    repetition does the same work.
       program      ONE Program.run, out of place (the run-time specialised kernel)
       interpreter  the same Program.run in a child process with PXF_JIT=0 (k_program<surf>)
     The rays come from the surfaces2.npz fixture bundle of each surface (drawn with replacement, positions jittered
     by ~1 um); the W-S secondary back surface gets the primary's output.  Results are compared bit for bit.
  S  segmented: 1000 segments x 1e5 rays through a refracting pair of spheres, every segment with its own radii:
     ONE SegmentedProgram.run against the loop of per-segment Program.run, out of place, compared bit for bit.
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

T_IN = (-0., -0., .5, -0., -0., -0.)
T_OUT = (-0., -0., -1., -0., -0., -0.)


def ops(alpha):
    # name: (Program method, scalars, fixture bundle, reflect behind it, stand-alone module, takes the opd row)
    return {
        "tracesphere": ("tracesphere", (15.,), "sphere_in", False, "surfacesf", False),
        "tracesphereopd": ("tracesphereopd", (15., 1.5), "sphere_in", False, "surfacesf", True),
        "tracecyl": ("tracecyl", (15.,), "cyl_in", False, "surfacesf", False),
        "tracecylopd": ("tracecylopd", (15., 1.2), "cyl_in", False, "surfacesf", True),
        "cylconic": ("cylconic", (1. / 400., -.7), "cylconic_in", True, "surfacesf", False),
        "paraxial": ("paraxial", (350.,), "paraxial_in", False, "surfacesf", False),
        "paraxialy": ("paraxialy", (-120.,), "paraxial_in", False, "surfacesf", False),
        "torus": ("torus", (150., 900.), "torus_in", True, "surfacesf", False),
        "wsprimaryback": ("wsprimaryback", (alpha, 1.e4, 1., .4), "wsback_in", True, "woltsurf", False),
        "wssecondaryback": ("wssecondaryback", (alpha, 1.e4, 1., .4), "wsback_in", True, "woltsurf", False),
    }


def source(pxf, key, num, seed):
    """num rays of the fixture bundle ``key`` (drawn with replacement on the device, x and y jittered by ~1 um)"""
    import torch
    from pyxfocus_b200._call import bundle_alloc
    fix = np.load(os.path.join(ROOT, "tests", "golden", "surfaces2.npz"))[key]
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    idx = torch.randint(0, fix.shape[1], (num,), generator=g, device=dev)
    rows = bundle_alloc(num, dev)
    for k in range(10):
        rows[k].copy_(torch.from_numpy(np.ascontiguousarray(fix[k])).to(dev)[idx])
    for k in (1, 2):
        rows[k].add_(torch.randn(num, generator=g, device=dev, dtype=torch.float64), alpha=1e-3)
    return rows


def op_program(pxf, spec):
    meth, args, _, refl = spec[:4]
    p = getattr(pxf.Program().transform(*T_IN), meth)(*args)
    p.reflect() if refl else p.refract(1., 1.5)
    return p.transform(*T_OUT).flatopd(1.)


def op_bundle(pxf, name, spec, num):
    src = source(pxf, spec[2], num, seed=11)
    if name == "wssecondaryback":
        # the secondary's rays come off the primary
        pxf.woltsurf.wsprimaryback(*src[1:], *spec[1])
        pxf.transformationsf.reflect(*src[4:])
    return src


def op_case(pxf, name, spec, num, reps, interp_only=False):
    import torch
    from pyxfocus_b200._call import bundle_alloc
    dev = torch.device("cuda", 0)
    src = op_bundle(pxf, name, spec, num)
    out = bundle_alloc(num, dev)
    prog = op_program(pxf, spec)
    ts, _, launches = timed(lambda: prog.run(src, out=out), reps)
    res = {"program": entry(ts, num, launches, pxf.last_trace_kernel())}
    if interp_only:
        return res
    meth, args, _, refl, mod, with_opd = spec
    work = bundle_alloc(num, dev)
    head = pxf.Program().transform(*T_IN)
    tail = (pxf.Program().reflect() if refl else pxf.Program().refract(1., 1.5)).transform(*T_OUT).flatopd(1.)
    routine = getattr(getattr(pxf, mod), meth)

    def launches_seq():
        head.run(src, out=work)
        routine(*(work if with_opd else work[1:]), *args)
        tail.run(work)
    # the head does not touch opd: one checked pass starts from the source's, the timed ones run on whatever is there
    work[0].copy_(src[0])
    launches_seq()
    res["bits_equal"] = all(torch.equal(out[k].view(torch.int64), work[k].view(torch.int64)) for k in range(10))
    ts, _, launches = timed(launches_seq, reps)
    res["launches"] = entry(ts, num, launches)
    res["speedup_median"] = res["launches"]["ms_median"] / res["program"]["ms_median"]
    return res


def lens(pxf, k):
    return (pxf.Program().transform(-0., -0., 5. + .001 * k, -0., -0., -0.).tracesphereopd(20. + .01 * k, 1.)
            .refract(1., 1.5).transform(0., 0., -10., 0., 0., 0.).tracesphere(40. + .01 * k).refract(1.5, 1.)
            .flatopd(1.))


def segmented(pxf, K, n, reps, interp_only=False):
    import torch
    from pyxfocus_b200._call import bundle_alloc
    dev = torch.device("cuda", 0)
    num = K * n
    src = source(pxf, "sphere_in", num, seed=12)
    out = bundle_alloc(num, dev)
    progs = [lens(pxf, k) for k in range(K)]
    seg = pxf.SegmentedProgram(progs, [n] * K)
    ts, _, launches = timed(lambda: seg.run(src, out=out), reps)
    res = {"segments": K, "rays_per_segment": n, "segmented": entry(ts, num, launches, pxf.last_trace_kernel())}
    if interp_only:
        return res
    work = bundle_alloc(num, dev)
    views_in = [[r[k * n:(k + 1) * n] for r in src] for k in range(K)]
    views_out = [[r[k * n:(k + 1) * n] for r in work] for k in range(K)]

    def loop():
        for k in range(K):
            progs[k].run(views_in[k], out=views_out[k])
    ts, _, launches = timed(loop, max(3, reps // 2))
    res["loop"] = entry(ts, num, launches, pxf.last_trace_kernel())
    res["speedup_median"] = res["loop"]["ms_median"] / res["segmented"]["ms_median"]
    res["bits_equal"] = all(torch.equal(out[k].view(torch.int64), work[k].view(torch.int64)) for k in range(10))
    return res


def interpreter(scale, reps):
    """O and S with the interpreter only (PXF_JIT=0 is read once per process: a child process)"""
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
    spec = ops(float(pxf.conicsolve.woltparam(220., 1.e4)[0]))
    num = int(5e7 * a.scale)
    if a.child_interp:
        r = {name: op_case(pxf, name, s, num, a.reps, interp_only=True)["program"] for name, s in spec.items()}
        r["segmented"] = segmented(pxf, 1000, int(1e5 * a.scale), a.reps, interp_only=True)["segmented"]
        print(json.dumps(r))
        return
    res = {"info": device_info(), "rays": num}
    res["O_ops"] = {name: op_case(pxf, name, s, num, a.reps) for name, s in spec.items()}
    res["S_segmented"] = segmented(pxf, 1000, int(1e5 * a.scale), a.reps)
    res["interpreter"] = interpreter(a.scale, a.reps)
    res["jit_status"] = pxf.jit_status()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
