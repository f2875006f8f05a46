"""radgratW and grat as fused-program ops against the three launches ``fused`` needed before them.

At 5e7 rays, out of place, each grating inside the chain  transform, flat, GRATING, transform, flat  runs as
  - one launch: the whole chain as one program (the new ops);
  - three launches: program (transform, flat) out of place | stand-alone pxf_radgratw / pxf_grat in place on the
    output | program (transform, flat) in place on the output -- what ``fused`` ran when it met the grating.
The two are alternated in one process, timed with CUDA events (median of the repetitions), and their outputs are
compared bit for bit (NaN for NaN).  The bundle (8 GB in and out) is far larger than L2.  ``--path`` picks the kernels: the
run-time specialised chain (default) or the interpreter (PXF_JIT=0, set by the parent before the library loads).
Without ``--path`` the script runs both in child processes and writes one JSON with the card's name and power limit.

    python profiles/grating_ops_bench.py --out profiles/grating_ops_bench_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def run_path(num, reps):
    import numpy as np
    import torch

    import pyxfocus_b200 as pxf
    from pyxfocus_b200 import transformationsf
    from pyxfocus_b200._call import bundle_alloc
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    src = bundle_alloc(num, dev)
    src[0].zero_()
    src[1].copy_(torch.rand(num, dtype=torch.float64, device=dev, generator=g) * 100 - 50)
    src[2].copy_(torch.rand(num, dtype=torch.float64, device=dev, generator=g) * 100 - 50)
    src[3].copy_(torch.rand(num, dtype=torch.float64, device=dev, generator=g) - .5)
    src[4].copy_(torch.rand(num, dtype=torch.float64, device=dev, generator=g) * .1 - .05)
    src[5].copy_(torch.rand(num, dtype=torch.float64, device=dev, generator=g) * .1 - .05)
    src[6].copy_(-torch.sqrt(1 - src[4] ** 2 - src[5] ** 2))
    for k in (7, 8):
        src[k].zero_()
    src[9].fill_(1.)
    wave = 3.6 + 3.6 * torch.rand(num, dtype=torch.float64, device=dev, generator=g)
    order = torch.randint(-3, 4, (num,), device=dev, generator=g).to(torch.float64)
    T1, T2 = (0., 0., 10., .01, .02, 0.), (1., -2., 5., 0., -.01, .03)
    head = pxf.Program().transform(*T1).flat()
    tail = pxf.Program().transform(*T2).flat()
    cases = {
        "radgratw": (pxf.Program().transform(*T1).flat().radgratw(wave, 2., -3.).transform(*T2).flat(),
                     lambda o: transformationsf.radgratw(o[1], o[2], o[4], o[5], o[6], wave, 2., -3.)),
        "grat": (pxf.Program().transform(*T1).flat().grat(160., order, wave).transform(*T2).flat(),
                 lambda o: transformationsf.grat(o[1], o[2], o[4], o[5], o[6], 160., order, wave)),
    }
    out_a, out_b = bundle_alloc(num, dev), bundle_alloc(num, dev)
    res = {}
    for name, (one, alone) in cases.items():
        def single():
            one.run(src, out=out_a)

        def three():
            head.run(src, out=out_b)
            alone(out_b)
            tail.run(out_b)
        for f in (single, three, single, three):        # warm-up (module loads, kernel compiles)
            f()
        kern = None
        times = {"single": [], "three": []}
        for _ in range(reps):
            for key, f in (("single", single), ("three", three)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                f()
                e1.record()
                e1.synchronize()
                times[key].append(e0.elapsed_time(e1))
                if key == "single":
                    kern = pxf.last_trace_kernel()
        # bits, NaN for NaN (the sign of a NaN follows the compiler's operand order)
        a_, b_ = ([o[k].cpu().numpy() for k in range(10)] for o in (out_a, out_b))
        same = all(np.array_equal(np.isnan(x), np.isnan(y)) and
                   np.array_equal(x.view(np.int64)[~np.isnan(x)], y.view(np.int64)[~np.isnan(y)]) for x, y in zip(a_, b_))
        nan_rays = int(np.isnan(a_[6]).sum())
        res[name] = dict(single_ms=float(np.median(times["single"])), three_ms=float(np.median(times["three"])),
                         single_ms_all=times["single"], three_ms_all=times["three"], kernel=kern, bit_identical=same,
                         nan_rays=nan_rays)
        res[name]["speedup"] = res[name]["three_ms"] / res[name]["single_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num", type=int, default=50_000_000)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--path", choices=["chain", "interp"])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.path:
        print(json.dumps(run_path(a.num, a.reps)))
        return
    result = dict(card=card(), num=a.num, reps=a.reps, layout="out of place",
                  chain="transform, flat, GRATING, transform, flat")
    for path in ("chain", "interp"):
        env = dict(os.environ, PXF_JIT="0" if path == "interp" else "1")
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--path", path, "--num", str(a.num), "--reps",
                            str(a.reps)], env=env, capture_output=True, text=True, check=True)
        result[path] = json.loads(r.stdout.strip().splitlines()[-1])
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
