"""Mirror of the reference's ``transformations.py`` on the device ray bundle.

Same function names, argument order and semantics (file:line cited per function).  ``rays``
is a list of ten 1-D float64 CUDA tensors.  Differences from the reference, all invisible to
results:

* ``ind=`` (bool mask, index array or ``np.where`` tuple) is executed as a per-ray predicate
  inside the kernel instead of gather -> Fortran -> scatter copies
  (transformations.py:20-27,54-61,106-109,152-166);
* ``vignette`` is an order-preserving ballot/prefix stream compaction kernel instead of ten
  numpy fancy-index copies (transformations.py:214-225);
* inside ``with program.fused(rays):`` unmasked calls are recorded and run as one kernel.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from . import transformationsf as tran
from ._call import bundle_alloc, stream_ptr, to_mask
from .program import flush, recorder_for


def copy_rays(rays):
    """transformations.py:7-8"""
    flush(rays)
    out = bundle_alloc(rays[1].shape[0], rays[1].device)
    for i in range(10):
        out[i].copy_(rays[i])
    return out


def _update_coords_fwd(coords, dx, dy, dz, rx, ry, rz):
    rotm = rotationM(rx, ry, rz)
    tranm = translationM(dx, dy, dz)
    rotmi = rotationM(rx, ry, rz, inverse=True)
    tranmi = translationM(-dx, -dy, -dz)
    coords[0] = np.dot(rotm, coords[0])
    coords[1] = np.dot(np.dot(rotm, tranm), coords[1])
    coords[2] = np.dot(coords[2], rotmi)
    coords[3] = np.dot(coords[3], np.dot(tranmi, rotmi))


def transform(rays, dx, dy, dz, rx, ry, rz, ind=None, coords=None):
    """Coordinate transformation: translation, then Rx, Ry, Rz (transformations.py:11-44).
    All six arguments are negated before the kernel, as the reference does (:29)."""
    x, y, z, l, m, n, ux, uy, uz = rays[1:]
    prog = recorder_for(rays) if ind is None else None
    if prog is not None:
        prog.transform(-dx, -dy, -dz, -rx, -ry, -rz)
    else:
        flush(rays)
        tran.transform(x, y, z, l, m, n, ux, uy, uz, -dx, -dy, -dz, -rx, -ry, -rz, mask=ind)
    if coords is not None:
        _update_coords_fwd(coords, dx, dy, dz, rx, ry, rz)
    return


def itransform(rays, dx, dy, dz, rx, ry, rz, coords=None, ind=None):
    """Inverse transformation: -rz, -ry, -rx, then translation (transformations.py:47-77)."""
    x, y, z, l, m, n, ux, uy, uz = rays[1:]
    prog = recorder_for(rays) if ind is None else None
    if prog is not None:
        prog.itransform(-dx, -dy, -dz, -rx, -ry, -rz)
    else:
        flush(rays)
        tran.itransform(x, y, z, l, m, n, ux, uy, uz, -dx, -dy, -dz, -rx, -ry, -rz, mask=ind)
    if coords is not None:
        rotm = rotationM(rx, ry, rz, inverse=True)
        tranm = translationM(-dx, -dy, -dz)
        rotmi = rotationM(rx, ry, rz)
        tranmi = translationM(dx, dy, dz)
        coords[0] = np.dot(rotm, coords[0])
        coords[1] = np.dot(np.dot(tranm, rotm), coords[1])
        coords[2] = np.dot(coords[2], rotmi)
        coords[3] = np.dot(coords[3], np.dot(rotmi, tranmi))
    return


def pointTo(rays, x0, y0, z0, reverse=-1.):
    """Point all direction cosines toward (x0,y0,z0) (transformations.py:91-100); one pxf_pointto launch."""
    flush(rays)
    x, y, z, l, m, n = rays[1:7]
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().pxf_pointto(x.data_ptr(), y.data_ptr(), z.data_ptr(), l.data_ptr(), m.data_ptr(),
                                          n.data_ptr(), x.shape[0], float(x0), float(y0), float(z0), float(reverse),
                                          None, stream_ptr(x.device)))
    return


def reflect(rays, ind=None):
    """Reflect about the surface normal (transformations.py:102-112)."""
    l, m, n, ux, uy, uz = rays[4:]
    prog = recorder_for(rays) if ind is None else None
    if prog is not None:
        prog.reflect()
        return
    flush(rays)
    tran.reflect(l, m, n, ux, uy, uz, mask=ind)
    return


def refract(rays, n1, n2):
    """Refract from index n1 into n2 (transformations.py:114-121)."""
    l, m, n, ux, uy, uz = rays[4:]
    prog = recorder_for(rays)
    if prog is not None:
        prog.refract(n1, n2)
        return
    tran.refract(l, m, n, ux, uy, uz, n1, n2)
    return


def radgrat(rays, dpermm, order, wave, ind=None):
    """Infinite radial grating in the x-y plane (transformations.py:124-172).  A scalar
    ``wave`` uses ``radgrat`` (sign of n kept); an array (numpy or tensor) uses ``radgratw``
    (sign taken from y), the reference's own dispatch (:146-149).  Inside ``fused`` an array with one
    entry per ray is recorded (a device tensor is read when the program runs, a host array is copied now)."""
    x, y, z, l, m, n = rays[1:7]
    is_arr = isinstance(wave, (np.ndarray, torch.Tensor)) and np.ndim(wave) > 0
    if is_arr and np.size(wave) == 1 and ind is not None:
        # reference: type(wave)==ndarray picks radgratw but a size-1 array is passed whole (:156-159)
        wave = torch.as_tensor(wave, dtype=torch.float64).reshape(1).expand(x.shape[0]).contiguous()
    if is_arr:
        prog = recorder_for(rays) if ind is None else None
        if prog is not None and prog.can_hold_arrays():
            # converted as the stand-alone call converts its intent(in) array (_call.Staged.input)
            w = torch.as_tensor(wave).to(device=x.device, dtype=torch.float64).contiguous()
            if w.dim() == 1 and w.shape[0] == x.shape[0]:
                prog.radgratw(w, dpermm, order)
                return
        flush(rays)
        tran.radgratw(x, y, l, m, n, wave, dpermm, order, mask=ind)
        return
    prog = recorder_for(rays) if ind is None else None
    if prog is not None:
        prog.radgrat(float(wave), dpermm, order)
        return
    flush(rays)
    tran.radgrat(x, y, l, m, n, float(wave), dpermm, order, mask=ind)
    return


def grat(rays, d, order, wave, ind=None):
    """Linear grating with grooves along +y (transformations.py:200-212).  ``order`` and
    ``wave`` are per-ray arrays (scalars are broadcast).  Recorded inside ``fused`` unless ``ind`` is
    given."""
    x, y, z, l, m, n = rays[1:7]
    num = x.shape[0]

    def vec(v):
        t = torch.as_tensor(v, dtype=torch.float64, device=x.device)
        return t.expand(num).contiguous() if t.dim() == 0 else t.contiguous()
    order, wave = vec(order), vec(wave)
    prog = recorder_for(rays) if ind is None else None
    if (prog is not None and prog.can_hold_arrays() and order.dim() == wave.dim() == 1
            and order.shape[0] == wave.shape[0] == num):
        prog.grat(d, order, wave)
        return
    flush(rays)
    tran.grat(x, y, l, m, n, d, order, wave, mask=ind)
    return


def take(rows, ind):
    """``[r[ind] for r in rows]`` for equally long float64 device rows: a bool mask is an order-preserving
    compaction, an index array (or ``np.where`` tuple) a gather that may repeat / reorder like numpy fancy
    indexing.  One library pass over all rows."""
    rows = list(rows)
    dev = rows[0].device
    num = rows[0].shape[0]
    nr = len(rows)
    L = _lib.lib()
    s = stream_ptr(dev)
    if _is_mask(ind, num):
        with torch.cuda.device(dev):
            flags = to_mask(ind, num, dev)
            scratch = torch.empty(int(L.pxf_compact_scratch_bytes(num)), dtype=torch.uint8, device=dev)
            count = ctypes.c_int64(0)
            _lib.check(L.pxf_compact_count(flags.data_ptr(), num, scratch.data_ptr(), ctypes.byref(count), s))
            out = bundle_alloc(count.value, dev, nrows=nr)
            pin = (ctypes.c_void_p * nr)(*[r.data_ptr() for r in rows])
            pout = (ctypes.c_void_p * nr)(*[r.data_ptr() for r in out])
            _lib.check(L.pxf_compact_scatter(pin, pout, nr, flags.data_ptr(), num, scratch.data_ptr(), s))
        return out
    idx = ind[0] if isinstance(ind, tuple) else ind
    if not isinstance(idx, torch.Tensor):
        idx = np.ascontiguousarray(idx)          # (a reversed / strided numpy view cannot be wrapped directly)
    idx = torch.as_tensor(idx, device=dev).long().contiguous()
    if idx.numel() and (int(idx.min()) < -num or int(idx.max()) >= num):
        raise IndexError("index out of bounds for %d rays" % num)
    idx = torch.where(idx < 0, idx + num, idx)
    count = idx.shape[0]
    out = bundle_alloc(count, dev, nrows=nr)
    pin = (ctypes.c_void_p * nr)(*[r.data_ptr() for r in rows])
    pout = (ctypes.c_void_p * nr)(*[r.data_ptr() for r in out])
    tab = torch.empty(256, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.pxf_gather_rows(pin, pout, nr, idx.data_ptr(), count, tab.data_ptr(), s))
    return out


def vignette(rays, ind=None):
    """Remove vignetted rays (transformations.py:214-225).  ``ind`` selects the rays to KEEP
    (bool mask / index array / ``np.where`` tuple); default keeps ``l^2+m^2+n^2 > .1``.
    Returns a new bundle; order is preserved."""
    flush(rays)
    if ind is not None:
        return take(rays, ind)
    dev = rays[1].device
    num = rays[1].shape[0]
    with torch.cuda.device(dev):
        flags = torch.empty(num, dtype=torch.uint8, device=dev)
        _lib.check(_lib.lib().pxf_vignette_flags(rays[4].data_ptr(), rays[5].data_ptr(), rays[6].data_ptr(), num,
                                                 flags.data_ptr(), stream_ptr(dev)))
        return compact(rays, flags)


def compact(rays, flags, extra=None):
    """Order-preserving stream compaction of all ten rows by a uint8 flag row.  ``extra``: further per-ray float64
    rows (e.g. the weights that the reference scripts index with the same mask, ``weights = weights[ind]``)
    compacted in the same pass; returns ``(bundle, [extra rows])`` then."""
    dev = rays[1].device
    num = rays[1].shape[0]
    L = _lib.lib()
    s = stream_ptr(dev)
    extra = [] if extra is None else list(extra)
    for e in extra:
        if not e.is_cuda or e.dtype != torch.float64 or not e.is_contiguous() or e.shape[0] != num:
            raise ValueError("extra rows must be contiguous float64 CUDA tensors with one entry per ray")
    with torch.cuda.device(dev):
        scratch = torch.empty(int(L.pxf_compact_scratch_bytes(num)), dtype=torch.uint8, device=dev)
        count = ctypes.c_int64(0)
        _lib.check(L.pxf_compact_count(flags.data_ptr(), num, scratch.data_ptr(), ctypes.byref(count), s))
        out = bundle_alloc(count.value, dev, nrows=10 + len(extra))
        nr = 10 + len(extra)
        pin = (ctypes.c_void_p * nr)(*[r.data_ptr() for r in list(rays) + extra])
        pout = (ctypes.c_void_p * nr)(*[r.data_ptr() for r in out])
        _lib.check(L.pxf_compact_scatter(pin, pout, nr, flags.data_ptr(), num, scratch.data_ptr(), s))
    if extra:
        return out[:10], out[10:]
    return out


def surviving_indices(flags):
    """``np.where(flags)[0]`` on the device (int64), via the same prefix kernels."""
    dev = flags.device
    num = flags.shape[0]
    L = _lib.lib()
    s = stream_ptr(dev)
    with torch.cuda.device(dev):
        scratch = torch.empty(int(L.pxf_compact_scratch_bytes(num)), dtype=torch.uint8, device=dev)
        count = ctypes.c_int64(0)
        _lib.check(L.pxf_compact_count(flags.data_ptr(), num, scratch.data_ptr(), ctypes.byref(count), s))
        idx = torch.empty(count.value, dtype=torch.int64, device=dev)
        _lib.check(L.pxf_compact_indices(flags.data_ptr(), num, scratch.data_ptr(), idx.data_ptr(), s))
    return idx


def _is_mask(ind, num):
    if isinstance(ind, tuple):
        ind = ind[0]
    if isinstance(ind, torch.Tensor):
        return ind.dtype == torch.bool
    return np.asarray(ind).dtype == np.bool_


# ------------------------------------------------------------------ 4x4 bookkeeping (host numpy)
def _rotation_matrix(angle, axis):
    """Homogeneous right-handed rotation about a coordinate axis (the subset of Gohlke's
    ``rotation_matrix`` the reference uses via transformMod, transformations.py:242-244)."""
    c, s = np.cos(angle), np.sin(angle)
    M = np.identity(4)
    i = int(np.argmax(np.abs(axis)))
    j, k = (i + 1) % 3, (i + 2) % 3
    M[j, j] = c
    M[j, k] = -s
    M[k, j] = s
    M[k, k] = c
    return M


def newCoords():
    """Identity matrices establishing a coordinate system (transformations.py:228-232)."""
    return [np.identity(4)] * 4


def rotationM(rx, ry, rz, inverse=False):
    """Rotation matrix, rotations applied in X,Y,Z order (transformations.py:234-248)."""
    if inverse is True:
        rx, ry, rz = -rx, -ry, -rz
    r1 = _rotation_matrix(-rx, [1, 0, 0])
    r2 = _rotation_matrix(-ry, [0, 1, 0])
    r3 = _rotation_matrix(-rz, [0, 0, 1])
    if inverse is True:
        return np.dot(r1, np.dot(r2, r3))
    return np.dot(r3, np.dot(r2, r1))


def translationM(tx, ty, tz):
    """Translation matrix (transformations.py:250-255)."""
    M = np.identity(4)
    M[:3, 3] = [-tx, -ty, -tz]
    return M


def applyT(rays, coords, inverse=False):
    """Apply a transformation matrix to the bundle; rotations only for the direction cosines
    and normals (transformations.py:257-280).  Returns a new bundle (one copy + one pxf_applyt launch)."""
    flush(rays)
    i = 2 if inverse is True else 0
    dev = rays[1].device
    P = np.ascontiguousarray(coords[i + 1], dtype=np.float64)
    R = np.ascontiguousarray(coords[i], dtype=np.float64)
    if P.shape != (4, 4) or R.shape != (4, 4):
        raise ValueError("coords must hold 4x4 matrices")
    num = rays[1].shape[0]
    out = bundle_alloc(num, dev)
    for k in range(10):
        out[k].copy_(rays[k])
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().pxf_applyt(*[r.data_ptr() for r in out[1:]], num, P.ctypes.data, R.ctypes.data,
                                         stream_ptr(dev)))
    return out


def _mean_tilts(rays):
    """(mean l, mean m) of the bundle by the library's deterministic tree reduction (pxf_centroid on rows 4, 5)."""
    l, m = rays[4], rays[5]
    a, b = ctypes.c_double(), ctypes.c_double()
    with torch.cuda.device(l.device):
        _lib.check(_lib.lib().pxf_centroid(l.data_ptr(), m.data_ptr(), None, l.shape[0], ctypes.byref(a), ctypes.byref(b),
                                           stream_ptr(l.device)))
    return a.value, b.value


def steerY(rays, coords=None):
    """Rotate the reference frame until the mean y tilt vanishes (transformations.py:78-82)."""
    flush(rays)
    while abs(_mean_tilts(rays)[1]) > 1e-6:
        transform(rays, 0, 0, 0, -_mean_tilts(rays)[1], 0, 0, coords=coords)
        flush(rays)          # inside `with fused(rays)` the transform is only recorded: run it before re-reading the mean
    return


def steerX(rays, coords=None):
    """Rotate the reference frame until the mean x tilt vanishes (transformations.py:84-88)."""
    flush(rays)
    while abs(_mean_tilts(rays)[0]) > 1e-6:
        transform(rays, 0, 0, 0, 0, -_mean_tilts(rays)[0], 0, coords=coords)
        flush(rays)
    return


def applyTPos(x, y, z, coords, inverse=False):
    """Apply the accumulated coordinate transformation to a list of points
    (transformations.py:283-290); host or device arrays, returns three arrays of the same kind."""
    i = 2 if inverse is True else 0
    M = np.asarray(coords[i + 1], dtype=np.float64)
    if isinstance(x, torch.Tensor):
        Mt = torch.as_tensor(M, device=x.device)
        pos = torch.stack([x, y, z, torch.ones_like(x)])
        out = Mt @ pos
        return [out[0], out[1], out[2]]
    pos = [x, y, z, np.ones(np.size(x))]
    return np.dot(M, pos)[:3]


def skew(vec):
    """Skew-symmetric cross-product matrix (transformations.py:292-293)."""
    return np.array([[0, -vec[2], vec[1]], [vec[2], 0, -vec[0]], [-vec[1], vec[0], 0]])
