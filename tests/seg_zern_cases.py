"""Segmented programs with one Zernike surface per segment: the layouts, tables, programs and input bundles shared by
tests/test_gpu_segmented_zern.py and tests/run_seg_zern_compare.py (host side only: numpy in, numpy out)."""
import numpy as np

from oracle import pyref
from pyxfocus_b200 import examples as ex

# segments straddle the 2048-ray tile boundaries, some are empty
LAYOUT = [0, 1, 2047, 2048, 2049, 3, 0, 50001, 7]


def zern_table(k):
    """Term list of segment k: 36 terms (n <= 7), 10 terms (n <= 3), a single term, all zeros -- in turn -- with a
    radius of its own."""
    kind = k % 4
    if kind == 0:
        ro, ao = ex.zernike_orders(7)
        c = ex.zernike_coeff(len(ro), 100 + k)
    elif kind == 1:
        ro, ao = ex.zernike_orders(3)
        c = ex.zernike_coeff(len(ro), 100 + k, sigma=3e-4)
    elif kind == 2:
        # one term: the reference sizes its tables from the term count, so a single term is piston (n = 0)
        ro, ao, c = np.array([0]), np.array([0]), np.array([2.5e-4])
    else:
        ro, ao = ex.zernike_orders(7)
        c = np.zeros(len(ro))
    return c, ro, ao, 62.5 + 1.5 * k


def zern_nr(k):
    return 1. + .01 * k


def program(pxf, chain, k, with_nr):
    """Program of segment k: ``chain`` 'c3' = config 3's 14-op program (three vignette predicates), 'tzr' = transform,
    zernsurf, reflect.  ``with_nr``: tracezernOPD (nr of its own per segment) instead of tracezern."""
    c, ro, ao, rad = zern_table(k)
    nr = zern_nr(k) if with_nr else None
    P = pxf.Program
    if chain == "tzr":
        return P().transform(-1. - .1 * k, 2., 100., -1e-3, 2e-3 * k, -.3).zernsurf(c, ro, ao, rad, nr).reflect()
    return (P().transform(-220.3, 0., 100., 0., 0., 0.).zernsurf(c, ro, ao, rad, nr).reflect()
            .transform(0., 0., 0., -np.pi, 0., 0.).flatopd(1.).transform(220.3, 0., 8600., 0., 0., 0.)
            .wolterprimary(220., 8400., 1.).reflect().vignette_box(3, 8426., 8526.).vignette_abs(2, 50.)
            .woltersecondary(220., 8400., 1.).reflect().vignette_mag().flat())


def source(chain, num, seed=0):
    """Host bundle the chain is meant for: config 3's sub-annulus, or a 60 mm beam for the 3-op chain."""
    np.random.seed(seed)
    if chain == "tzr":
        return pyref.circularbeam(60., num)
    return pyref.subannulus(220., 220.6, 100. / 220., num, zhat=-1.)


CASES = [(chain, with_nr, oop) for chain in ("c3", "tzr") for with_nr in (False, True) for oop in (False, True)]


def case_name(chain, with_nr, oop):
    return "%s_nr%d_oop%d" % (chain, int(with_nr), int(oop))
