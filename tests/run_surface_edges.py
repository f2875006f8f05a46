"""Executed by tests/test_gpu_surface_edges.py in two processes -- PXF_JIT=0 (interpreter only) and PXF_JIT_MIN_RAYS=0
(every program specialised at run time) -- on the edge bundles of tests/surface_edge_cases.py: every fused-program op
alone and followed by ``flat``, and the segmented families with per-segment scalars at the edges.  Writes the traced
rows and the kernel that ran to the .npz named on the command line; the parent compares them with the oracle."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pyxfocus_b200 as pxf  # noqa: E402
import surface_edge_cases as E  # noqa: E402
from util import to_dev, to_host  # noqa: E402


def op_program(name, flat):
    case = E.CASES[name]
    p = getattr(pxf.Program(), case.routine)(*case.args)
    return p.flat() if flat else p


def main(path):
    res = {}
    for name in E.PROGRAM:
        for flat in (False, True):
            if flat and E.CASES[name].special:
                continue
            rays = to_dev(E.bundle(name)[0])
            op_program(name, flat).run(rays)
            key = "%s_flat%d" % (name, int(flat))
            for k, r in enumerate(to_host(rays)):
                res["%s_row%d" % (key, k)] = r
            res[key + "_kernel"] = np.array(pxf.last_trace_kernel())
    for family in sorted(E.SEG):
        rays = to_dev(E.seg_bundle(family)[0])
        progs = [E.SEG[family][1](pxf.Program, k) for k in range(len(E.LAYOUT))]
        pxf.SegmentedProgram(progs, E.LAYOUT).run(rays)
        key = "seg_" + family
        for k, r in enumerate(to_host(rays)):
            res["%s_row%d" % (key, k)] = r
        res[key + "_kernel"] = np.array(pxf.last_trace_kernel())
    np.savez(path, **res)


if __name__ == "__main__":
    main(sys.argv[1])
