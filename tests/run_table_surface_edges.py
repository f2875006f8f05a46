"""Executed by tests/test_gpu_table_surface_ops.py in two processes -- PXF_JIT=0 (interpreter only) and
PXF_JIT_MIN_RAYS=0 (every program specialised at run time) -- on the conicplus / legsurf edge bundles of
tests/surface_edge_cases.py: each op alone and followed by ``flat``, as a program and as a segmented program of three
segments (the middle one empty).  Writes the traced rows and the kernel that ran to the .npz named on the command line;
the parent compares them with the oracle."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pyxfocus_b200 as pxf  # noqa: E402
import surface_edge_cases as E  # noqa: E402
from util import to_dev, to_host  # noqa: E402

EDGE = sorted(n for n, c in E.CASES.items() if c.routine in ("conicplus", "conicplusopd", "legsurf"))


def op_program(name, flat):
    case = E.CASES[name]
    p = getattr(pxf.Program(), case.routine)(*case.args)
    return p.flat() if flat else p


def seg_sizes(n):
    return [n // 2, 0, n - n // 2]


def main(path):
    res = {}
    for name in EDGE:
        for flat in (False, True):
            for seg in (False, True):
                inp = E.bundle(name)[0]
                rays = to_dev(inp)
                if seg:
                    sizes = seg_sizes(inp[1].shape[0])
                    pxf.SegmentedProgram([op_program(name, flat) for _ in sizes], sizes).run(rays)
                else:
                    op_program(name, flat).run(rays)
                key = "%s_flat%d_seg%d" % (name, int(flat), int(seg))
                for k, r in enumerate(to_host(rays)):
                    res["%s_row%d" % (key, k)] = r
                res[key + "_kernel"] = np.array(pxf.last_trace_kernel())
    np.savez(path, **res)


if __name__ == "__main__":
    main(sys.argv[1])
