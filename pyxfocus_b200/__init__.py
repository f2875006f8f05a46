"""pyxfocus_b200 -- a B200 (sm_100a) ray-trace engine behind the PyXFocus Python API.

Drop-in module layout (same names as the reference package)::

    import pyxfocus_b200.sources as sources
    import pyxfocus_b200.surfaces as surf
    import pyxfocus_b200.transformations as tran
    import pyxfocus_b200.analyses as anal

and, one level down, replacements for the four f2py Fortran modules with the f2py
signatures: ``transformationsf``, ``surfacesf``, ``woltsurf``, ``zernsurf``.

The ray bundle is a list of ten float64 CUDA tensors ``[opd,x,y,z,l,m,n,ux,uy,uz]``.  All
arithmetic runs in hand-written CUDA kernels inside ``libpxf.so`` (C ABI: ``include/pxf.h``).
There is no CPU fallback: importing the package without the built library raises.
"""
from . import _lib

_lib.lib()      # fail loudly if libpxf.so is missing

from . import conicsolve, program, sources, transformations, surfaces, analyses, dist, host  # noqa: E402,F401
from . import transformationsf, surfacesf, woltsurf, zernsurf, reconstruct, southwell, examples  # noqa: E402,F401
from .program import FanAux, Program, SegmentedProgram, Segments, fused  # noqa: E402,F401
from ._lib import OPT_WS_LIBM, OPT_WS_RETRACE, OPT_WS_GRAZE_PPM, PxfError, jit_status, last_trace_kernel, launch_count, set_option  # noqa: E402,F401

__version__ = "0.1.0"
