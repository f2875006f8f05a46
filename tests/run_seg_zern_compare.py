"""Executed by tests/test_gpu_segmented_zern.py in two processes -- PXF_JIT=0 (interpreter only) and
PXF_JIT_MIN_RAYS=0 (every program specialised at run time) -- and prints one line per case: name, sha256 of the
traced rows and alive flags, and the kernel that ran.  The digests must be identical."""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pyxfocus_b200 as pxf  # noqa: E402
from seg_zern_cases import CASES, LAYOUT, case_name, program, source  # noqa: E402
from util import to_dev  # noqa: E402


def main():
    for chain, with_nr, oop in CASES:
        progs = [program(pxf, chain, k, with_nr) for k in range(len(LAYOUT))]
        rays = to_dev(source(chain, int(np.sum(LAYOUT)), seed=1))
        out = [torch.zeros_like(r) for r in rays] if oop else None
        alive = pxf.SegmentedProgram(progs, LAYOUT).run(rays, out=out)
        h = hashlib.sha256()
        for t in (out if oop else rays) + ([alive] if alive is not None else []):
            h.update(t.cpu().numpy().tobytes())
        print("%s %s %s" % (case_name(chain, with_nr, oop), h.hexdigest()[:24],
                            pxf.last_trace_kernel().replace(" ", "_")), flush=True)


if __name__ == "__main__":
    main()
