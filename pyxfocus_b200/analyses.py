"""Mirror of the hot-path part of the reference's ``analyses.py`` on the device ray bundle:
``centroid`` (analyses.py:16-22), ``rmsCentroid`` (:24-30), ``rmsX/rmsY`` (:46-58), ``rho``
(:60-71), ``rhocdf`` (:73-86), ``hpd`` (:88-97), ``analyticImagePlane`` (:118-133), plus
``findimageplane`` (named by the reference's examples, defined nowhere in it; see below).

Everything is reductions / order statistics computed by libpxf kernels: block+warp
reductions for the sums, an exact radix *select* on the IEEE bit patterns of the radii for
the unweighted median, a hand-written radix sort + scan for the weighted branch.  Scalars are
returned as Python floats like numpy scalars in the reference.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._call import stream_ptr
from .program import flush


def _w(weights, x):
    if weights is None:
        return None
    w = torch.as_tensor(weights, dtype=torch.float64, device=x.device).contiguous()
    if w.shape != x.shape:
        raise ValueError("weights must have one entry per ray")
    return w


def _ptr(t):
    return t.data_ptr() if t is not None else None


# ---- segmented bundles: ``segments=`` (a ``program.Segments``) gives every quantity per segment, as an
# np.ndarray[nseg], in a number of launches that does not depend on nseg and ONE read-back of the nseg results.
# A segment with no rays, or with zero total weight, gives NaN for every quantity.
def _seg_sums(mode, x, y, w, segments, z=None, l=None, m=None, n=None, ab=None):
    """Device [nseg, 16] per-segment sums of ``pxf_sums_segmented``."""
    segments.check(x.shape[0], x.device)
    dev = x.device
    L = _lib.lib()
    out = torch.empty((segments.nseg, 16), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        scratch = torch.empty(int(L.pxf_sums_segmented_scratch_bytes(x.shape[0], segments.nseg)), dtype=torch.uint8,
                              device=dev)
        _lib.check(L.pxf_sums_segmented(mode, x.data_ptr(), y.data_ptr(), _ptr(z), _ptr(l), _ptr(m), _ptr(n), _ptr(w),
                                        x.shape[0], segments.start_dev.data_ptr(), segments.nseg, _ptr(ab), out.data_ptr(),
                                        scratch.data_ptr(), stream_ptr(dev)))
    return out


def _nan_where_empty(v, S0):
    v = np.array(v, dtype=np.float64)
    v[S0 == 0] = np.nan
    return v


def _seg_rms(x, y, w, segments):
    sums = _seg_sums(0, x, y, w, segments)
    cxy = torch.empty((segments.nseg, 2), dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_centroids_segmented(sums.data_ptr(), segments.nseg, cxy.data_ptr(), stream_ptr(x.device)))
    S = _seg_sums(1, x, y, w, segments, ab=cxy).cpu().numpy()
    with np.errstate(divide="ignore", invalid="ignore"):
        return _nan_where_empty(np.sqrt(S[:, 1] / S[:, 0]), S[:, 0])


def centroid(rays, weights=None, segments=None):
    """Centroid of the rays in the xy plane (np.average semantics).  ``segments``: ``(cx[nseg], cy[nseg])``."""
    flush(rays)
    x, y = rays[1:3]
    w = _w(weights, x)
    if segments is not None:
        S = _seg_sums(0, x, y, w, segments).cpu().numpy()
        with np.errstate(divide="ignore", invalid="ignore"):
            return _nan_where_empty(S[:, 1] / S[:, 0], S[:, 0]), _nan_where_empty(S[:, 2] / S[:, 0], S[:, 0])
    cx, cy = ctypes.c_double(), ctypes.c_double()
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_centroid(x.data_ptr(), y.data_ptr(), _ptr(w), x.shape[0], ctypes.byref(cx),
                                           ctypes.byref(cy), stream_ptr(x.device)))
    return cx.value, cy.value


def rmsCentroid(rays, weights=None, segments=None):
    """RMS distance of the rays from their centroid in the xy plane (``segments``: per segment, about its own
    centroid)."""
    flush(rays)
    x, y = rays[1:3]
    w = _w(weights, x)
    if segments is not None:
        return _seg_rms(x, y, w, segments)
    out = ctypes.c_double()
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_rmscentroid(x.data_ptr(), y.data_ptr(), _ptr(w), x.shape[0], ctypes.byref(out),
                                              stream_ptr(x.device)))
    return out.value


def _rms1(v, weights, segments=None):
    # 1-D analogue of rmsCentroid: feed the same row as x and a zero-extent y
    w = _w(weights, v)
    zero = torch.zeros_like(v)
    if segments is not None:
        return _seg_rms(v, zero, w, segments)
    out = ctypes.c_double()
    with torch.cuda.device(v.device):
        _lib.check(_lib.lib().pxf_rmscentroid(v.data_ptr(), zero.data_ptr(), _ptr(w), v.shape[0],
                                              ctypes.byref(out), stream_ptr(v.device)))
    return out.value


def rmsX(rays, weights=None, segments=None):
    """RMS from centroid in the X direction (analyses.py:46-51)."""
    flush(rays)
    return _rms1(rays[1], weights, segments)


def rmsY(rays, weights=None, segments=None):
    """RMS from centroid in the Y direction (analyses.py:53-58)."""
    flush(rays)
    return _rms1(rays[2], weights, segments)


def rho(rays, weights=None, cent=False):
    """Distance of every ray from the centroid (cent=True) or the origin (analyses.py:60-71)."""
    flush(rays)
    x, y = rays[1:3]
    if cent is True:
        cx, cy = centroid(rays, weights=weights)
    else:
        cx, cy = 0., 0.
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_rho(x.data_ptr(), y.data_ptr(), x.shape[0], cx, cy, out.data_ptr(),
                                      stream_ptr(x.device)))
    return out


def argsort(keys):
    """(sorted keys, int64 permutation) by the library's stable LSD radix sort."""
    dev = keys.device
    num = keys.shape[0]
    L = _lib.lib()
    ks = torch.empty_like(keys)
    idx = torch.empty(num, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        scratch = torch.empty(int(L.pxf_sort_scratch_bytes(num)), dtype=torch.uint8, device=dev)
        _lib.check(L.pxf_argsort(keys.data_ptr(), num, ks.data_ptr(), idx.data_ptr(), scratch.data_ptr(),
                                 stream_ptr(dev)))
    return ks, idx


def rhocdf(rays, weights=None, cent=True):
    """Radial CDF of the ray distribution: (sorted radii, cumulative weight / max)
    (analyses.py:73-86)."""
    r = rho(rays, weights=weights, cent=cent)
    dev = r.device
    num = r.shape[0]
    w = _w(weights, r)
    L = _lib.lib()
    rs, idx = argsort(r)
    cdf = torch.empty_like(r)
    with torch.cuda.device(dev):
        scratch = torch.empty(int(L.pxf_scan_scratch_bytes(num)), dtype=torch.uint8, device=dev)
        if w is None:
            w = torch.ones_like(r)
        _lib.check(L.pxf_cumsum_gather(w.data_ptr(), idx.data_ptr(), num, cdf.data_ptr(), scratch.data_ptr(),
                                       stream_ptr(dev)))
    cdf = cdf / cdf.max()
    return rs, cdf


def hpd(rays, weights=None, cent=True, sums=None, segments=None):
    """Half-power diameter about the centroid (the reference ignores ``cent``,
    analyses.py:90).  Unweighted: 2*median(r).  Weighted:
    r[argmin|cdf-.75|] - r[argmin|cdf-.25|].
    ``sums`` (unweighted only): the centroid sums ``Program.run(..., sums=...)`` produced for
    this very bundle; saves the pass over x,y that computes them.
    ``segments``: the HPD of every segment about its own centroid (np.ndarray[nseg]); not with ``sums``."""
    flush(rays)
    x, y = rays[1:3]
    w = _w(weights, x)
    if segments is not None:
        if sums is not None:
            raise ValueError("hpd: segments= and sums= cannot be combined")
        return _hpd_seg(x, y, w, segments)
    out = ctypes.c_double()
    with torch.cuda.device(x.device):
        if sums is not None and w is None:
            _lib.check(_lib.lib().pxf_hpd_with_sums(x.data_ptr(), y.data_ptr(), x.shape[0], sums.data_ptr(),
                                                    ctypes.byref(out), stream_ptr(x.device)))
        else:
            _lib.check(_lib.lib().pxf_hpd(x.data_ptr(), y.data_ptr(), _ptr(w), x.shape[0], ctypes.byref(out),
                                          stream_ptr(x.device)))
    return out.value


def _hpd_seg(x, y, w, segments, mode=0, raw=False):
    """Per-segment ``pxf_hpd_segmented``; segments it flags (bracket miss / candidate overflow: rare) are resolved
    by the five-pass select on their slice.  ``raw``: the [nseg, 4] {HPD, lower, upper, valid} rows."""
    sums = _seg_sums(0, x, y, w, segments)
    dev, num, ns = x.device, x.shape[0], segments.nseg
    L = _lib.lib()
    out = torch.empty((ns, 4), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        ws = torch.empty(int(L.pxf_hpd_segmented_workspace_bytes(num, ns, 0 if w is None else 1)), dtype=torch.uint8,
                         device=dev)
        _lib.check(L.pxf_hpd_segmented(x.data_ptr(), y.data_ptr(), _ptr(w), num, segments.start_dev.data_ptr(), ns,
                                       sums.data_ptr(), out.data_ptr(), ws.data_ptr(), mode, stream_ptr(dev)))
        h = out.cpu().numpy()
        bad = np.nonzero(h[:, 3] == 0)[0]
        if bad.size:
            fws = hpd_workspace(0, dev)
            for k in bad:
                a, b = int(segments.start[k]), int(segments.start[k + 1])
                _lib.check(L.pxf_hpd_from_sums_dev(x[a:].data_ptr(), y[a:].data_ptr(), b - a, sums[k].data_ptr(),
                                                   out[k].data_ptr(), fws.data_ptr(), 1, stream_ptr(dev)))
            h[bad] = out[bad].cpu().numpy()
    return h if raw else h[:, 0].copy()


def hpd_workspace(num, device):
    """Scratch tensor for ``hpd_enqueue`` on bundles of up to ``num`` rays."""
    return torch.empty(int(_lib.lib().pxf_hpd_workspace_bytes(int(num))) + 64, dtype=torch.uint8, device=device)


def hpd_enqueue(rays, out, workspace, sums=None, mode=0):
    """Unweighted ``hpd`` without the read-back: everything is enqueued on the current stream and the
    result lands in ``out`` (device float64[4] = [HPD, lower middle radius, upper middle radius,
    valid]).  For pipelines that analyse many bundles back to back and read the numbers at the end.
    ``valid`` == 0 (bracket miss / ties piled in one bin: ~never) means: call again with mode=1."""
    flush(rays)
    x, y = rays[1:3]
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_hpd_from_sums_dev(x.data_ptr(), y.data_ptr(), x.shape[0],
                                                    sums.data_ptr() if sums is not None else None, out.data_ptr(),
                                                    workspace.data_ptr(), mode, stream_ptr(x.device)))
    return out


def analyticImagePlane(rays, weights=None, segments=None):
    """Axial shift to the best image plane, Ron Elsner's analytic method (analyses.py:118-133)."""
    flush(rays)
    x, y, z, l, m, n = rays[1:7]
    w = _w(weights, x)
    if segments is not None:
        h = imageplane_sums(rays, weights, segments=segments).cpu().numpy()
        W = h[:, 0]
        with np.errstate(divide="ignore", invalid="ignore"):
            # pxf_analyticimageplane's arithmetic, per segment
            ax_, ay_, aln, amn = h[:, 1] / W, h[:, 2] / W, h[:, 3] / W, h[:, 4] / W
            bx = h[:, 5] / W - ax_ * aln
            ax = h[:, 7] / W - aln * aln
            by = h[:, 6] / W - ay_ * amn
            ay = h[:, 8] / W - amn * amn
            return _nan_where_empty(-(bx + by) / (ax + ay), W)
    out = ctypes.c_double()
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_analyticimageplane(x.data_ptr(), y.data_ptr(), l.data_ptr(), m.data_ptr(),
                                                     n.data_ptr(), _ptr(w), x.shape[0], ctypes.byref(out),
                                                     stream_ptr(x.device)))
    return out.value


def imageplane_sums(rays, weights=None, at_z0=False, segments=None):
    """The nine weighted sums behind ``analyticImagePlane`` / ``findimageplane`` as a device
    tensor [S0, Sx, Sy, Sa, Sb, Sxa, Syb, Saa, Sbb] with a=l/n, b=m/n (one pass, 40 B/ray).
    ``at_z0``: take x, y where each ray crosses z = 0, (x - z a, y - z b) (48 B/ray) -- what a plane scan needs
    when the rays are not on the plane; ``analyticImagePlane`` itself ignores z (analyses.py:122-131).
    ``segments``: a device [nseg, 9] tensor, one row of sums per segment."""
    flush(rays)
    x, y, z, l, m, n = rays[1:7]
    w = _w(weights, x)
    if segments is not None:
        return _seg_sums(3 if at_z0 else 2, x, y, w, segments, z=z, l=l, m=m, n=n)[:, :9]
    L = _lib.lib()
    dev = x.device
    out = torch.zeros(16, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        scratch = torch.empty(int(L.pxf_sums_scratch_bytes()), dtype=torch.uint8, device=dev)
        if at_z0:
            _lib.check(L.pxf_sums_z(x.data_ptr(), y.data_ptr(), z.data_ptr(), l.data_ptr(), m.data_ptr(), n.data_ptr(),
                                    _ptr(w), x.shape[0], out.data_ptr(), scratch.data_ptr(), stream_ptr(dev)))
        else:
            _lib.check(L.pxf_sums(2, x.data_ptr(), y.data_ptr(), l.data_ptr(), m.data_ptr(), n.data_ptr(), _ptr(w),
                                  x.shape[0], 0., 0., out.data_ptr(), scratch.data_ptr(), stream_ptr(dev)))
    return out[:9]


def findimageplane(rays, zscan, num, weights=None, sums=None, moved=0., segments=None):
    """Scan the axial offset over ``linspace(-zscan, zscan, num)`` and return the offset of
    minimum RMS spot radius about the centroid.

    PARITY UNPINNED: the reference *calls* ``findimageplane(zscan,num)`` from its examples
    (examples/axro/WSverify.py:74-77,161-164) but ships no definition (SURVEY.md 8c).  This
    follows the legacy behaviour those call sites imply (move the plane by dz, trace to it,
    take rmsCentroid, keep the best dz).  Propagating a ray by dz changes (x,y) by
    (l/n, m/n)*dz, so RMS^2(dz) is an exact quadratic in dz whose coefficients are the nine
    sums of ``analyticImagePlane`` (taken where the rays cross z = 0, so rays that are off the plane -- e.g.
    after ``transform(rays,0,0,dz,...)`` without a ``flat`` -- scan as the literal loop would): one pass over the
    bundle instead of ``num`` passes.  ``sums`` / ``moved``: sums from an earlier ``imageplane_sums(rays,
    at_z0=True)`` and the z offset the frame has been moved by since (``transform(rays,0,0,moved,...)``): a second,
    finer scan then costs no pass at all.
    ``segments``: the offset of every segment (np.ndarray[nseg]); ``sums`` is then the [nseg, 9] output of
    ``imageplane_sums(rays, at_z0=True, segments=...)`` and ``moved`` a scalar or one offset per segment."""
    if segments is not None:
        S = (sums if sums is not None else imageplane_sums(rays, weights, at_z0=True, segments=segments)).cpu().numpy()
        S = S.copy()
        mv = np.broadcast_to(np.asarray(moved, dtype=np.float64), (S.shape[0],))
        sh = mv != 0.
        for k, j in ((1, 3), (2, 4), (5, 7), (6, 8)):
            S[sh, k] += mv[sh] * S[sh, j]
        W = S[:, 0]
        with np.errstate(divide="ignore", invalid="ignore"):
            mx, my, ma, mb = S[:, 1] / W, S[:, 2] / W, S[:, 3] / W, S[:, 4] / W
            vxx = S[:, 7] / W - ma * ma + S[:, 8] / W - mb * mb
            cxa = S[:, 5] / W - mx * ma + S[:, 6] / W - my * mb
        dz = np.linspace(-zscan, zscan, int(num))
        merit = 2 * dz[None, :] * cxa[:, None] + dz[None, :] ** 2 * vxx[:, None]
        return _nan_where_empty(dz[np.argmin(merit, axis=1)], W)
    S = (sums if sums is not None else imageplane_sums(rays, weights, at_z0=True)).cpu().numpy().copy()
    if moved != 0.:
        # the new z = 0 plane lies `moved` further along: x0' = x0 + moved a, y0' = y0 + moved b
        S[1] += moved * S[3]; S[2] += moved * S[4]; S[5] += moved * S[7]; S[6] += moved * S[8]
    W = S[0]
    mx, my, ma, mb = S[1] / W, S[2] / W, S[3] / W, S[4] / W
    vxx = S[7] / W - ma * ma + S[8] / W - mb * mb            # Var(a)+Var(b)
    cxa = S[5] / W - mx * ma + S[6] / W - my * mb            # Cov(x,a)+Cov(y,b)
    dz = np.linspace(-zscan, zscan, int(num))
    # RMS^2(dz) = RMS^2(0) + 2 dz Cov + dz^2 Var ; the constant does not move the argmin
    merit = 2 * dz * cxa + dz ** 2 * vxx
    return float(dz[np.argmin(merit)])


def _plane_sums(rays, weights, segments=None):
    if segments is not None:
        S = imageplane_sums(rays, weights, segments=segments).cpu().numpy().T      # [9, nseg]
        with np.errstate(divide="ignore", invalid="ignore"):
            return _nan_where_empty(S / S[0], np.broadcast_to(S[0], S.shape))
    S = imageplane_sums(rays, weights).cpu().numpy()
    W = S[0]
    return S / W


def analyticYPlane(rays, weights=None, segments=None):
    """Axial shift to the best line focus in y (analyses.py:135-144); same one-pass sums as
    ``analyticImagePlane``."""
    a = _plane_sums(rays, weights, segments)      # [1, <x>, <y>, <l/n>, <m/n>, <x l/n>, <y m/n>, <(l/n)^2>, <(m/n)^2>]
    by = a[6] - a[2] * a[4]
    ay = a[8] - a[4] ** 2
    if segments is not None:
        with np.errstate(divide="ignore", invalid="ignore"):
            return -by / ay
    return float(-by / ay)


def analyticXPlane(rays, weights=None, segments=None):
    """Axial shift to the best line focus in x (analyses.py:146-155)."""
    a = _plane_sums(rays, weights, segments)
    bx = a[5] - a[1] * a[3]
    ax = a[7] - a[3] ** 2
    if segments is not None:
        with np.errstate(divide="ignore", invalid="ignore"):
            return -bx / ax
    return float(-bx / ax)


def hpdY(rays, weights=None):
    """HPD in the y direction about the mean y (analyses.py:99-116).  |y-cy| is the radius of the
    point (0, y), so this is ``hpd`` on a bundle whose x row is zero: sqrt(0 + (y-cy)^2) = |y-cy|
    exactly."""
    flush(rays)
    y = rays[2]
    zero = torch.zeros_like(y)
    fake = [rays[0], zero, y] + list(rays[3:])
    return hpd(fake, weights=weights)


def rmsPoint(rays, point, weights=None):
    """RMS distance of the rays from a point: a ten-row ray or an (x,y,z) triple (analyses.py:33-45)."""
    flush(rays)
    off = 1 if np.size(point) == 10 else 0
    px, py, pz = (float(point[off + k]) for k in range(3))
    x, y, z = rays[1:4]
    w = _w(weights, x)
    out = ctypes.c_double()
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_rmspoint(x.data_ptr(), y.data_ptr(), z.data_ptr(), _ptr(w), x.shape[0], px, py, pz,
                                           ctypes.byref(out), stream_ptr(x.device)))
    return out.value


def measureOPD(rays, point):
    """Distance of every ray from a point -- a ten-row ray or an (x,y,z) triple (analyses.py:232-244); a device tensor."""
    flush(rays)
    off = 1 if len(point) == 10 else 0
    px, py, pz = (float(point[off + k]) for k in range(3))
    x, y, z = rays[1:4]
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_distance(x.data_ptr(), y.data_ptr(), z.data_ptr(), out.data_ptr(), x.shape[0], px, py, pz,
                                           None, stream_ptr(x.device)))
    return out


def indAngle(rays, ind=None, normal=None):
    """Incidence angle against the current or a given surface normal (analyses.py:164-182); returns a
    device tensor (one pxf_indangle launch; ``ind`` -- bool mask or index array -- selects rays like numpy
    indexing does in the reference, through the library's compaction / gather kernels)."""
    flush(rays)
    l, m, n, ux, uy, uz = rays[4:10]
    dev = l.device
    num = l.shape[0]
    ang = torch.empty_like(l)
    nrm = None if normal is None else (ctypes.c_double * 3)(*[float(v) for v in normal])
    L = _lib.lib()
    with torch.cuda.device(dev):
        _lib.check(L.pxf_indangle(l.data_ptr(), m.data_ptr(), n.data_ptr(), ux.data_ptr(), uy.data_ptr(), uz.data_ptr(),
                                  ang.data_ptr(), num, nrm, None, stream_ptr(dev)))
    if ind is None:
        return ang
    from .transformations import take
    return take([ang], ind)[0]


def grazeAngle(rays, ind=None):
    """Graze angle against the current surface normal (analyses.py:184-187)."""
    return np.pi / 2 - indAngle(rays, ind=ind)


# ---- OPD-map pipeline: scattered-data interpolation and wavefront integration (analyses.py:189-230, 305-334) ----
_GRID_METHODS = {"nearest": 0, "linear": 1, "cubic": 2}


def griddata(px, py, values, qx, qy, method="linear"):
    """``scipy.interpolate.griddata((px, py), values, (qx, qy), method)`` for 'nearest' / 'linear' / 'cubic' on the
    device (``pxf_griddata``: the Delaunay triangle of every query point by pivoting to the empty circumcircle; 'cubic' is
    scipy's Clough-Tocher interpolant with its global gradient estimate; NaN outside the convex hull).  All five
    arguments are equally long (points) / equally shaped (queries) float64 CUDA tensors."""
    if method not in _GRID_METHODS:
        raise ValueError("Unknown interpolation method %r for 2 dimensional data" % (method,))
    dev = px.device
    shape = qx.shape
    px, py, values = (t.contiguous() for t in (px, py, values))
    fx, fy = qx.reshape(-1).contiguous(), qy.reshape(-1).contiguous()
    out = torch.empty_like(fx)
    L = _lib.lib()
    nfail = ctypes.c_int64(0)
    with torch.cuda.device(dev):
        scratch = torch.empty(int(L.pxf_griddata_scratch_bytes(px.shape[0])), dtype=torch.uint8, device=dev)
        _lib.check(L.pxf_griddata(px.data_ptr(), py.data_ptr(), values.data_ptr(), px.shape[0], fx.data_ptr(), fy.data_ptr(),
                                  out.data_ptr(), fx.shape[0], _GRID_METHODS[method], ctypes.byref(nfail),
                                  scratch.data_ptr(), stream_ptr(dev)))
    if nfail.value:
        raise _lib.PxfError("griddata: %d query points have no unique Delaunay triangle (degenerate point set: "
                            "duplicate, collinear or exactly cocircular points) -- %s"
                            % (nfail.value, (L.pxf_last_error() or b"").decode()))
    return out.reshape(shape)


def delaunay_neighbors(px, py):
    """Delaunay neighbours of every point, counter-clockwise: ``(ring, degree, is_hull_vertex)`` -- an int32
    ``[N, max_degree]`` tensor padded with -1, and two uint8 ``[N]`` tensors."""
    dev = px.device
    n = px.shape[0]
    L = _lib.lib()
    ring = torch.empty((n, int(L.pxf_delaunay_max_degree())), dtype=torch.int32, device=dev)
    deg = torch.empty(n, dtype=torch.uint8, device=dev)
    hull = torch.empty(n, dtype=torch.uint8, device=dev)
    px, py = px.contiguous(), py.contiguous()
    with torch.cuda.device(dev):
        scratch = torch.empty(int(L.pxf_griddata_scratch_bytes(n)), dtype=torch.uint8, device=dev)
        _lib.check(L.pxf_delaunay_neighbors(px.data_ptr(), py.data_ptr(), n, ring.data_ptr(), deg.data_ptr(), hull.data_ptr(),
                                            scratch.data_ptr(), stream_ptr(dev)))
    return ring, deg, hull


def _bbox(x, y):
    L = _lib.lib()
    box = (ctypes.c_double * 4)()
    with torch.cuda.device(x.device):
        scratch = torch.empty(int(L.pxf_bbox_scratch_bytes()), dtype=torch.uint8, device=x.device)
        _lib.check(L.pxf_bbox(x.data_ptr(), y.data_ptr(), x.shape[0], box, scratch.data_ptr(), stream_ptr(x.device)))
    return list(box)


def interpolateVec(rays, I, Nx, Ny, xr=None, yr=None, method='linear', polar=False, interpVec=None):
    """Interpolate ray vector ``I`` (or ``interpVec``) onto an Nx x Ny grid spanning the rays' x/y range
    (analyses.py:189-230).  Returns ``(res, dx, dy)``; ``res`` is a (Ny, Nx) CUDA tensor."""
    flush(rays)
    x, y = rays[1:3]
    dev = x.device
    vec = rays[I] if interpVec is None else torch.as_tensor(interpVec, dtype=torch.float64, device=dev)
    if xr is None:
        box = _bbox(x, y)
        xr, yr = box[0:2], box[2:4]
    gx, gy = np.meshgrid(np.linspace(xr[0], xr[1], Nx), np.linspace(yr[0], yr[1], Ny))
    dx = np.diff(gx)[0][0]
    dy = np.diff(np.transpose(gy))[0][0]
    qx, qy = torch.from_numpy(gx).to(dev), torch.from_numpy(gy).to(dev)
    if polar is not True:
        return griddata(x, y, vec, qx, qy, method=method), dx, dy
    # two polar charts (cut along -x and along -y), then the median of the two maps
    L = _lib.lib()

    def chart(px, py):
        flat_x, flat_y = px.reshape(-1).contiguous(), py.reshape(-1).contiguous()
        rho, a1, a2 = (torch.empty_like(flat_x) for _ in range(3))
        with torch.cuda.device(dev):
            _lib.check(L.pxf_polar_coords(flat_x.data_ptr(), flat_y.data_ptr(), flat_x.shape[0], rho.data_ptr(),
                                          a1.data_ptr(), a2.data_ptr(), stream_ptr(dev)))
        return rho.reshape(px.shape), a1.reshape(px.shape), a2.reshape(px.shape)
    rho, t1, t2 = chart(x, y)
    rhog, g1, g2 = chart(qx, qy)
    res1 = griddata(rho, t1, vec, rhog, g1, method=method)
    res2 = griddata(rho, t2, vec, rhog, g2, method=method)
    res = torch.empty_like(res1)
    with torch.cuda.device(dev):
        _lib.check(L.pxf_nanmedian2(res1.data_ptr(), res2.data_ptr(), res1.numel(), res.data_ptr(), stream_ptr(dev)))
    return res, dx, dy


def wavefront(rays, Nx, Ny, method='cubic', polar=False, maxiter=10000):
    """Interpolate the beam slopes onto a grid and integrate the wavefront (analyses.py:305-334): ``interpolateVec`` of
    m and l, a one-pixel border, missing data -> 100., Southwell reconstruction (criterion 1e-12, step dx).  Returns
    ``(phase, x, y)`` without the border, as numpy arrays like the reference (NaN where there is no data).

    As shipped the reference cannot run this function: ``man.padRect`` lives in the un-vendored ``utilities.imaging``
    package (taken here as a one-pixel NaN frame, which is what the ``[1:-1,1:-1]`` at the end strips), and
    ``reconstruct.reconstruct`` is called without its required ``maxiter`` (here a keyword, default as in
    ``southwell.southwell``)."""
    from . import reconstruct as _rec
    ys, dx, dy = interpolateVec(rays, 5, Nx, Ny, method=method, polar=polar)
    xs, dx, dy = interpolateVec(rays, 4, Nx, Ny, method=method, polar=polar)

    def framed(t):
        a = np.full((t.shape[0] + 2, t.shape[1] + 2), np.nan, order='F')
        a[1:-1, 1:-1] = t.cpu().numpy()
        return a
    xs, ys = framed(xs), framed(ys)
    hole = np.isnan(xs)
    phase = np.zeros(xs.shape, order='F')
    phase[hole] = 100.
    xs[hole] = 100.
    ys[np.isnan(ys)] = 100.
    phase = _rec.reconstruct(ys, xs, 1e-12, dx, phase, maxiter)
    phase[phase == 100] = np.nan
    xs[xs == 100] = np.nan
    ys[ys == 100] = np.nan
    return phase[1:-1, 1:-1], xs[1:-1, 1:-1], ys[1:-1, 1:-1]


# ---- scalar set-up formulas of analyses.py that do not touch a ray bundle (host numpy, as in the reference) ----
def radialGrad(x, y, hubscale, yaw, hubdist):
    """x and y derivatives of a radial grating's phase function at the points (x, y) (analyses.py:402-428).  As in the
    reference the hub shift is applied to the UNROTATED y (``y2 = y + hubdist``, :415)."""
    x2 = x * np.cos(yaw) + y * np.sin(yaw)
    y2 = y + hubdist
    rho = np.sqrt(x2 ** 2 + y2 ** 2)
    theta = np.arctan2(-x2, y2)
    gx = hubscale * (np.cos(theta) / rho)
    gy = -hubscale * (np.sin(theta) / rho)
    return gx * np.cos(-yaw) + gy * np.sin(-yaw), -gx * np.sin(-yaw) + gy * np.cos(-yaw)


def sellmeier(wave, B, C):
    """Refractive index from Sellmeier coefficients, one value per wavelength (analyses.py:430-446)."""
    w2 = np.reshape(wave, [np.size(wave), 1]) ** 2
    B = np.reshape(B, [1, np.size(B)])
    C = np.reshape(C, [1, np.size(C)])
    return np.sqrt(1 + np.sum(np.dot(w2, B) / (w2 - C), axis=1))

