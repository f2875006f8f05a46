"""Executed by tests/test_gpu_surface_ops.py in two processes -- PXF_JIT=0 (interpreter only) and PXF_JIT_MIN_RAYS=0
(every program specialised at run time) -- and prints one line per case: name, sha256 of the traced rows and alive
flags, and the kernel that ran.  The digests must be identical."""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pyxfocus_b200 as pxf  # noqa: E402
from surface_cases import LAYOUT, SEG, SINGLE, single_name, single_program, source  # noqa: E402
from util import to_dev  # noqa: E402


def digest(rows, alive):
    h = hashlib.sha256()
    for t in rows + ([alive] if alive is not None else []):
        h.update(t.cpu().numpy().tobytes())
    return h.hexdigest()[:24]


def main():
    for family in sorted(SEG):
        make, key = SEG[family]
        for oop in (False, True):
            progs = [make(pxf, k) for k in range(len(LAYOUT))]
            rays = to_dev(source(key, int(np.sum(LAYOUT)), seed=1))
            out = [torch.zeros_like(r) for r in rays] if oop else None
            alive = pxf.SegmentedProgram(progs, LAYOUT).run(rays, out=out)
            print("seg_%s_oop%d %s %s" % (family, int(oop), digest(out if oop else rays, alive),
                                          pxf.last_trace_kernel().replace(" ", "_")), flush=True)
    for name in sorted(SINGLE):
        for vig in (False, True):
            h = source(SINGLE[name][2], 20_000, seed=2)
            rays = to_dev(h)
            alive = single_program(pxf, name, vig_rows=h if vig else None).run(rays)
            print("%s %s %s" % (single_name(name, vig), digest(rays, alive),
                                pxf.last_trace_kernel().replace(" ", "_")), flush=True)


if __name__ == "__main__":
    main()
