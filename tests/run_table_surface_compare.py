"""Executed by tests/test_gpu_table_surface_ops.py in two processes -- PXF_JIT=0 (interpreter only) and
PXF_JIT_MIN_RAYS=0 (every program specialised at run time) -- and prints one line per case: name, sha256 of the traced
rows and alive flags, and the kernel that ran.  The digests must be identical."""
import hashlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pyxfocus_b200 as pxf  # noqa: E402
from table_surface_cases import PROGRAMS, SEGMENTED, source  # noqa: E402
from util import to_dev  # noqa: E402


def digest(rows, alive):
    h = hashlib.sha256()
    for t in rows + ([alive] if alive is not None else []):
        h.update(t.cpu().numpy().tobytes())
    return h.hexdigest()[:24]


def main():
    for name in sorted(PROGRAMS):
        for vig in (False, True):
            rays = to_dev(source(name, 20_000, seed=2))
            out = [torch.zeros_like(r) for r in rays]
            alive = PROGRAMS[name](pxf, vig).run(rays, out=out)
            print("%s_vig%d %s %s" % (name, int(vig), digest(out, alive), pxf.last_trace_kernel().replace(" ", "_")),
                  flush=True)
    for name in sorted(SEGMENTED):
        progs, sizes, key = SEGMENTED[name](pxf, 31)
        rays = to_dev(source(key, sum(sizes), seed=3))
        alive = pxf.SegmentedProgram(progs, sizes).run(rays)
        print("seg_%s %s %s" % (name, digest(rays, alive), pxf.last_trace_kernel().replace(" ", "_")), flush=True)


if __name__ == "__main__":
    main()
