"""Legendre-Legendre shells in fused programs: the term lists, programs, layouts and input bundles shared by
tests/test_gpu_ll_program.py and tests/run_ll_compare.py (host side only: numpy in, numpy out)."""
import numpy as np

from oracle import pyref
from pyxfocus_b200 import examples as ex

# segments straddle the 2048-ray tile boundaries, some are empty
LAYOUT = [0, 1, 2047, 2048, 2049, 3, 0, 50001, 7]
KINDS = (0, 1, 2)             # wolterprimLL, woltersecLL, ellipsoidWoltLL
ORDERS = (3, 5, 7)
S_ELL = 2.5e5


def terms(order, seed):
    """Every term up to ``order`` in both directions, random coefficients [mm]."""
    axial, az = ex.ll_orders(order)
    return ex.ll_coeff(len(axial), seed), axial, az


def add_ll(prog, kind, order, seed):
    c, ax, az = terms(order, seed)
    if kind == 0:
        return prog.wolterprimll(220., 8400., 8500., 8400., .25, c, ax, az)
    if kind == 1:
        return prog.woltersecll(220., 8400., 1., 8400., 8300., .25, c, ax, az)
    return prog.ellipsoidwoltll(220., 8400., 1., S_ELL, 8500., 8400., .25, c, ax, az)


def routine(of_or_pxf, rows, kind, order, seed):
    """The per-routine call the LL op replaces (``woltsurf`` of the package or of the C oracle) on nine rows."""
    c, ax, az = terms(order, seed)
    w = of_or_pxf.woltsurf
    if kind == 0:
        w.wolterprimll(*rows, 220., 8400., 8500., 8400., .25, c, ax, az)
    elif kind == 1:
        w.woltersecll(*rows, 220., 8400., 1., 8400., 8300., .25, c, ax, az)
    else:
        w.ellipsoidwoltll(*rows, 220., 8400., 1., S_ELL, 8500., 8400., .25, c, ax, az)


# the z window of the vignette predicate behind each kind's shell: it cuts part of the bundle
ZCUT = {0: (8430., 8470.), 1: (8330., 8370.), 2: (8430., 8470.)}
T_IN = (-0., -0., 8400., -0., -0., -0.)          # transformations.transform(rays, 0, 0, -8400, 0, 0, 0), recorded


def single_program(pxf, kind, order, vig):
    """transform, [wolterprimary, reflect for the secondary], the LL shell, reflect, [vignette on z]."""
    p = pxf.Program().transform(*T_IN)
    if kind == 1:
        p.wolterprimary(220., 8400., 1.).reflect()
    add_ll(p, kind, order, 10 * kind + order)
    p.reflect()
    if vig:
        p.vignette_box(3, *ZCUT[kind])
    return p


SINGLE = [(kind, order, vig) for kind in KINDS for order in ORDERS for vig in (False, True)]


def single_name(kind, order, vig):
    return "k%d_n%d_vig%d" % (kind, order, int(vig))


def seg_program(pxf, k):
    """Program of segment k: the LL pair, the primary's kind alternating between wolterprimLL and ellipsoidWoltLL and
    both orders cycling through 3, 5, 7 (so one bundle holds every order at each LL position)."""
    p = pxf.Program().transform(-0., -0., 8400. + .5 * k, -0., -0., -0.)
    add_ll(p, 0 if k % 2 == 0 else 2, ORDERS[k % 3], 100 + k)
    p.reflect()
    add_ll(p, 1, ORDERS[(k + 1) % 3], 200 + k)
    return p.reflect().flat()


def seg_segment_routines(of_or_pxf, rows, k):
    """seg_program(k) as per-routine calls on ten host or device rows."""
    tf = of_or_pxf.transformationsf
    tf.transform(*rows[1:], -0., -0., 8400. + .5 * k, -0., -0., -0.)
    routine(of_or_pxf, rows[1:], 0 if k % 2 == 0 else 2, ORDERS[k % 3], 100 + k)
    tf.reflect(*rows[4:])
    routine(of_or_pxf, rows[1:], 1, ORDERS[(k + 1) % 3], 200 + k)
    tf.reflect(*rows[4:])
    of_or_pxf.surfacesf.flat(*rows[1:])


def source(num, seed=0):
    """Host bundle of the LL pair: the sub-annulus of the reference fixture."""
    np.random.seed(seed)
    return pyref.subannulus(220., 220.6, .25, num, zhat=-1.)
