"""ctypes binding of ``libpxf.so`` (the C ABI declared in ``include/pxf.h``).

This is the only place the shared library is opened.  There is no CPU fallback:
if the library is missing, ``lib()`` raises; if no CUDA device is present the
entry points return ``PXF_ERR_CUDA`` and ``check()`` raises ``PxfError``.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpxf.so")

_c = ctypes
_dp = _c.c_void_p          # device / host double*  (passed as integer addresses)
_vp = _c.c_void_p
_d = _c.c_double
_i64 = _c.c_int64
_i32 = _c.c_int32
_u64 = _c.c_uint64
_sz = _c.c_size_t
_st = _c.c_void_p          # pxf_stream_t


class PxfError(RuntimeError):
    """Raised when a libpxf entry point returns a non-zero status (the analogue of
    ``<f2py module>.error``)."""


class pxf_op(ctypes.Structure):
    _fields_ = [("code", _i32), ("reserved", _i32), ("p", _d * 6)]


class pxf_program_aux(ctypes.Structure):
    _fields_ = [("wave", _c.c_void_p), ("count", _c.c_void_p), ("count_max", _c.c_void_p), ("cap", _i32),
                ("reserved", _i32)]


# name -> (restype, [argtypes]).  Order follows include/pxf.h.
_NINE = [_dp] * 9
SIGNATURES = {
    "pxf_version": (_c.c_int, []),
    "pxf_last_error": (_c.c_char_p, []),
    "pxf_launch_count": (_i64, []),
    "pxf_set_option": (_c.c_int, [_i32, _i32]),
    "pxf_newton_cap": (_c.c_int, []),
    # transformationsf
    "pxf_transform": (_c.c_int, _NINE + [_i64] + [_d] * 6 + [_vp, _st]),
    "pxf_itransform": (_c.c_int, _NINE + [_i64] + [_d] * 6 + [_vp, _st]),
    "pxf_reflect": (_c.c_int, [_dp] * 6 + [_i64, _vp, _st]),
    "pxf_refract": (_c.c_int, [_dp] * 6 + [_i64, _d, _d, _vp, _st]),
    "pxf_pointto": (_c.c_int, [_dp] * 6 + [_i64, _d, _d, _d, _d, _vp, _st]),
    "pxf_distance": (_c.c_int, [_dp] * 4 + [_i64, _d, _d, _d, _vp, _st]),
    "pxf_applyt": (_c.c_int, _NINE + [_i64, _vp, _vp, _st]),
    "pxf_indangle": (_c.c_int, [_dp] * 7 + [_i64, _vp, _vp, _st]),
    "pxf_radgrat": (_c.c_int, [_dp] * 5 + [_d, _i64, _d, _d, _vp, _st]),
    "pxf_radgratw": (_c.c_int, [_dp] * 6 + [_i64, _d, _d, _vp, _st]),
    "pxf_grat": (_c.c_int, [_dp] * 5 + [_i64, _d, _dp, _dp, _vp, _st]),
    # surfacesf
    "pxf_flat": (_c.c_int, _NINE + [_i64, _vp, _st]),
    "pxf_flatopd": (_c.c_int, _NINE + [_dp, _i64, _d, _vp, _st]),
    "pxf_conic": (_c.c_int, _NINE + [_i64, _d, _d, _vp, _st]),
    "pxf_conicopd": (_c.c_int, [_dp] * 10 + [_i64, _d, _d, _d, _vp, _st]),
    "pxf_tracesphere": (_c.c_int, _NINE + [_i64, _d, _vp, _st]),
    "pxf_tracesphereopd": (_c.c_int, [_dp] * 10 + [_i64, _d, _d, _vp, _st]),
    "pxf_tracecyl": (_c.c_int, _NINE + [_i64, _d, _vp, _st]),
    "pxf_tracecylopd": (_c.c_int, [_dp] * 10 + [_i64, _d, _d, _vp, _st]),
    "pxf_cylconic": (_c.c_int, _NINE + [_i64, _d, _d, _vp, _st]),
    "pxf_paraxial": (_c.c_int, _NINE + [_i64, _d, _vp, _st]),
    "pxf_paraxialy": (_c.c_int, _NINE + [_i64, _d, _vp, _st]),
    "pxf_torus": (_c.c_int, _NINE + [_i64, _d, _d, _vp, _st]),
    "pxf_conicplus": (_c.c_int, _NINE + [_i64, _d, _d, _vp, _i32, _vp, _st]),
    "pxf_conicplusopd": (_c.c_int, [_dp] * 10 + [_i64, _d, _d, _vp, _i32, _d, _vp, _st]),
    "pxf_legsurf": (_c.c_int, _NINE + [_i64, _d, _d, _d, _vp, _vp, _vp, _i32, _vp, _st]),
    # woltsurf
    "pxf_wsprimaryback": (_c.c_int, _NINE + [_i64, _d, _d, _d, _d, _vp, _st]),
    "pxf_wssecondaryback": (_c.c_int, _NINE + [_i64, _d, _d, _d, _d, _vp, _st]),
    "pxf_wolterprimary": (_c.c_int, _NINE + [_i64, _d, _d, _d, _vp, _st]),
    "pxf_wolterprimaryopd": (_c.c_int, [_dp] * 10 + [_i64, _d, _d, _d, _d, _vp, _st]),
    "pxf_woltersecondary": (_c.c_int, _NINE + [_i64, _d, _d, _d, _vp, _st]),
    "pxf_woltersine": (_c.c_int, _NINE + [_i64, _d, _d, _d, _d, _vp, _st]),
    "pxf_wsprimary": (_c.c_int, _NINE + [_i64, _d, _d, _d, _vp, _st]),
    "pxf_wssecondary": (_c.c_int, _NINE + [_i64, _d, _d, _d, _vp, _st]),
    "pxf_spocone": (_c.c_int, _NINE + [_i64, _d, _d, _vp, _st]),
    "pxf_wolterprimll": (_c.c_int, _NINE + [_i64] + [_d] * 5 + [_vp, _vp, _vp, _i32, _vp, _st]),
    "pxf_woltersecll": (_c.c_int, _NINE + [_i64] + [_d] * 6 + [_vp, _vp, _vp, _i32, _vp, _st]),
    "pxf_ellipsoidwoltll": (_c.c_int, _NINE + [_i64] + [_d] * 7 + [_vp, _vp, _vp, _i32, _vp, _st]),
    # zernsurf (coeff/rorder/aorder are HOST pointers)
    "pxf_tracezern": (_c.c_int, _NINE + [_i64, _vp, _vp, _vp, _i32, _d, _vp, _st]),
    "pxf_tracezernopd": (_c.c_int, [_dp] * 10 + [_i64, _vp, _vp, _vp, _i32, _d, _d, _vp, _st]),
    "pxf_zernphase": (_c.c_int, [_dp] * 10 + [_i64, _vp, _vp, _vp, _i32, _d, _d, _vp, _st]),
    "pxf_tracezernrot": (_c.c_int, _NINE + [_i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _d, _d, _vp, _st]),
    # fused program
    "pxf_trace_program": (_c.c_int, [_vp, _i64, _vp, _i32, _vp, _st]),
    "pxf_trace_program_to": (_c.c_int, [_vp, _vp, _i64, _vp, _i32, _vp, _st]),
    "pxf_trace_program_sums": (_c.c_int, [_vp, _vp, _i64, _vp, _i32, _vp, _dp, _vp, _st]),
    "pxf_jit_compile": (_i32, [_vp, _i32, _i32, _vp]),
    "pxf_jit_status": (_c.c_char_p, []),
    "pxf_last_trace_kernel": (_c.c_char_p, []),
    "pxf_trace_program_aux": (_c.c_int, [_vp, _vp, _i64, _vp, _i32, _vp, _vp, _dp, _vp, _st]),
    # vignetting / compaction
    "pxf_vignette_flags": (_c.c_int, [_dp] * 3 + [_i64, _vp, _st]),
    "pxf_compact_scratch_bytes": (_sz, [_i64]),
    "pxf_compact_count": (_c.c_int, [_vp, _i64, _vp, _vp, _st]),
    "pxf_compact_scatter": (_c.c_int, [_vp, _vp, _i32, _vp, _i64, _vp, _st]),
    "pxf_compact_indices": (_c.c_int, [_vp, _i64, _vp, _vp, _st]),
    "pxf_gather_rows": (_c.c_int, [_vp, _vp, _i32, _vp, _i64, _vp, _st]),
    # analyses
    "pxf_sums_scratch_bytes": (_sz, []),
    "pxf_sums": (_c.c_int, [_i32] + [_dp] * 6 + [_i64, _d, _d, _dp, _vp, _st]),
    "pxf_sums_z": (_c.c_int, [_dp] * 7 + [_i64, _dp, _vp, _st]),
    "pxf_rho": (_c.c_int, [_dp, _dp, _i64, _d, _d, _dp, _st]),
    "pxf_select_state_bytes": (_sz, []),
    "pxf_select_begin": (_c.c_int, [_vp, _i64, _i64, _st]),
    "pxf_select_hist": (_c.c_int, [_dp, _dp, _dp, _i64, _dp, _i32, _i32, _vp, _st]),
    "pxf_select_hist_ptr": (_vp, [_vp]),
    "pxf_select_nan_ptr": (_vp, [_vp]),
    "pxf_select_narrow": (_c.c_int, [_i32, _vp, _st]),
    "pxf_select_finish": (_c.c_int, [_vp, _i64, _dp, _st]),
    "pxf_select_schedule": (_c.c_int, [_i32, _vp, _vp]),
    "pxf_centroid_from_sums": (_c.c_int, [_dp, _dp, _st]),
    "pxf_bracket_min_num": (_i64, []),
    "pxf_bracket_samples": (_i32, []),
    "pxf_bracket_capacity": (_i64, [_i64]),
    "pxf_bracket_sample_ranks": (None, [_i32, _vp, _vp]),
    "pxf_select_sample": (_c.c_int, [_dp, _dp, _i64, _dp, _i32, _dp, _st]),
    "pxf_bracket_collect": (_c.c_int, [_dp, _dp, _i64, _dp, _dp, _dp, _i64, _vp, _st]),
    "pxf_select_begin_bracket": (_c.c_int, [_vp, _i64, _i64, _vp, _i64, _st]),
    "pxf_select_hist_keys": (_c.c_int, [_dp, _i64, _vp, _i32, _i32, _vp, _st]),
    "pxf_sample_pack": (_c.c_int, [_dp, _dp, _i64, _dp, _i32, _dp, _st]),
    "pxf_sample_radii": (_c.c_int, [_dp, _i32, _i32, _dp, _dp, _dp, _st]),
    "pxf_fastsel_bytes": (_sz, []),
    "pxf_fast_nbins": (_i32, []),
    "pxf_fast_fincap": (_i32, []),
    "pxf_small_select": (_c.c_int, [_dp, _vp, _i32, _i32, _i64, _i64, _i32, _vp, _dp, _st]),
    "pxf_cand_hist": (_c.c_int, [_dp, _i64, _vp, _dp, _vp, _st]),
    "pxf_cand_scan": (_c.c_int, [_vp, _vp, _i64, _i64, _vp, _st]),
    "pxf_cand_gather": (_c.c_int, [_dp, _i64, _vp, _dp, _vp, _dp, _vp, _st]),
    "pxf_hpd_workspace_bytes": (_sz, [_i64]),
    "pxf_hpd_unweighted_dev": (_c.c_int, [_dp, _dp, _i64, _dp, _vp, _i32, _st]),
    "pxf_hpd_from_sums_dev": (_c.c_int, [_dp, _dp, _i64, _dp, _dp, _vp, _i32, _st]),
    "pxf_hpd_with_sums": (_c.c_int, [_dp, _dp, _i64, _dp, _vp, _st]),
    "pxf_segment_counts": (_c.c_int, [_vp, _i64, _vp, _i32, _vp, _st]),
    "pxf_sums_segmented_scratch_bytes": (_sz, [_i64, _i32]),
    "pxf_sums_segmented": (_c.c_int, [_i32] + [_dp] * 7 + [_i64, _vp, _i32, _dp, _dp, _vp, _st]),
    "pxf_centroids_segmented": (_c.c_int, [_dp, _i32, _dp, _st]),
    "pxf_hpd_segmented_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "pxf_hpd_segmented": (_c.c_int, [_dp, _dp, _dp, _i64, _vp, _i32, _dp, _dp, _vp, _i32, _st]),
    "pxf_centroid": (_c.c_int, [_dp, _dp, _dp, _i64, _vp, _vp, _st]),
    "pxf_rmscentroid": (_c.c_int, [_dp, _dp, _dp, _i64, _vp, _st]),
    "pxf_hpd": (_c.c_int, [_dp, _dp, _dp, _i64, _vp, _st]),
    "pxf_rmspoint": (_c.c_int, [_dp, _dp, _dp, _dp, _i64, _d, _d, _d, _vp, _st]),
    "pxf_analyticimageplane": (_c.c_int, [_dp] * 6 + [_i64, _vp, _st]),
    "pxf_hpd_weighted": (_c.c_int, [_dp, _dp, _dp, _i64, _vp, _st]),
    "pxf_hpd_weighted_sorted": (_c.c_int, [_dp, _dp, _dp, _i64, _vp, _st]),
    "pxf_hpd_weighted_bracket": (_c.c_int, [_dp, _dp, _dp, _i64, _vp, _vp, _st]),
    "pxf_wq_state_bytes": (_sz, []),
    "pxf_wq_min_num": (_i64, []),
    "pxf_wq_samples": (_i32, [_i64]),
    "pxf_wq_capacity": (_i64, [_i64]),
    "pxf_wq_sample": (_c.c_int, [_dp, _dp, _dp, _i64, _dp, _i32, _dp, _dp, _st]),
    "pxf_wq_brackets": (_c.c_int, [_dp, _dp, _i32, _i32, _vp, _st]),
    "pxf_wq_collect_scratch_bytes": (_sz, []),
    "pxf_wq_collect": (_c.c_int, [_dp, _dp, _dp, _i64, _dp, _vp, _dp, _dp, _dp, _dp, _i64, _vp, _st]),
    "pxf_wq_below_ptr": (_vp, [_vp, _i32]),
    "pxf_wq_argmin_scratch_bytes": (_sz, []),
    "pxf_wq_argmin": (_c.c_int, [_dp, _dp, _i64, _dp, _dp, _d, _dp, _vp, _st]),
    "pxf_wq_merge_state_bytes": (_sz, []),
    "pxf_wq_merge_klo_ptr": (_vp, [_vp]),
    "pxf_wq_merge_result_ptr": (_vp, [_vp]),
    "pxf_wq_merge_begin": (_c.c_int, [_vp, _i64, _i64, _i64, _i64, _st]),
    "pxf_wq_merge_probe": (_c.c_int, [_vp, _dp, _i64, _vp, _dp, _i64, _vp, _i32, _dp, _st]),
    "pxf_wq_merge_narrow": (_c.c_int, [_vp, _dp, _dp, _dp, _d, _d, _i32, _st]),
    "pxf_wq_merge_final_probe": (_c.c_int, [_vp, _dp, _i64, _vp, _dp, _i64, _vp, _dp, _st]),
    "pxf_wq_merge_finish": (_c.c_int, [_vp, _dp, _dp, _dp, _d, _d, _st]),
    "pxf_sort_scratch_bytes": (_sz, [_i64]),
    "pxf_argsort": (_c.c_int, [_dp, _i64, _dp, _vp, _vp, _st]),
    "pxf_argsort_digits": (_c.c_int, [_dp, _i64, _dp, _vp, _vp, _i32, _st]),
    "pxf_scan_scratch_bytes": (_sz, [_i64]),
    "pxf_cumsum_gather": (_c.c_int, [_dp, _vp, _i64, _dp, _vp, _st]),
    # reconstruct
    "pxf_reconstruct": (_c.c_int, [_dp, _dp, _i32, _i32, _d, _d, _dp, _dp, _i32, _vp, _st]),
    "pxf_southwellbin_scratch_bytes": (_sz, [_i64, _i32, _i32]),
    "pxf_southwellbin": (_c.c_int, [_dp, _dp, _dp, _dp, _i64, _d, _dp, _dp, _dp, _i32, _i32, _vp, _st]),
    # scattered-data interpolation
    "pxf_griddata_scratch_bytes": (_sz, [_i64]),
    "pxf_bbox_scratch_bytes": (_sz, []),
    "pxf_bbox": (_c.c_int, [_dp, _dp, _i64, _vp, _vp, _st]),
    "pxf_polar_coords": (_c.c_int, [_dp, _dp, _i64, _dp, _dp, _dp, _st]),
    "pxf_nanmedian2": (_c.c_int, [_dp, _dp, _i64, _dp, _st]),
    "pxf_delaunay_max_degree": (_c.c_int, []),
    "pxf_delaunay_neighbors": (_c.c_int, [_dp, _dp, _i64, _vp, _vp, _vp, _vp, _st]),
    "pxf_griddata": (_c.c_int, [_dp, _dp, _dp, _i64, _dp, _dp, _dp, _i64, _i32, _vp, _vp, _st]),
    # sources
    "pxf_source": (_c.c_int, [_i32, _vp, _i64, _i64, _u64, _d, _d, _d, _d, _st]),
    "pxf_source_segmented": (_c.c_int, [_i32, _vp, _i64, _i64, _u64, _i32, _vp, _dp, _st]),
    "pxf_zern_table_bytes": (_sz, []),
    "pxf_zern_table_fill": (_i32, [_vp, _vp, _vp, _i32, _d, _i32, _d, _vp]),
    "pxf_segmented_table_bytes": (_sz, [_i32, _i32]),
    "pxf_segmented_table_fill": (_c.c_int, [_vp, _i32, _i32, _vp, _vp]),
    "pxf_segmented_table_bytes_zern": (_sz, [_i32, _i32]),
    "pxf_segmented_table_fill_zern": (_c.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "pxf_ll_table_bytes": (_sz, []),
    "pxf_ll_table_fill": (_i32, [_i32, _d, _d, _d, _d, _d, _d, _d, _vp, _vp, _vp, _i32, _vp]),
    "pxf_zern_table_fill_rot": (_i32, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _d, _d, _vp]),
    "pxf_conicplus_table_bytes": (_sz, []),
    "pxf_conicplus_table_fill": (_i32, [_d, _d, _vp, _i32, _i32, _d, _vp]),
    "pxf_legsurf_table_bytes": (_sz, []),
    "pxf_legsurf_table_fill": (_i32, [_d, _d, _d, _vp, _vp, _vp, _i32, _vp]),
    "pxf_segmented_table_bytes_ll": (_sz, [_i32, _i32]),
    "pxf_segmented_table_fill_ll": (_c.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "pxf_trace_program_segmented": (_c.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _st]),
    "pxf_source_from_uniform": (_c.c_int, [_i32, _vp, _i64, _dp, _dp, _d, _d, _d, _d, _st]),
    "pxf_source_grid": (_c.c_int, [_i32, _vp, _i64, _i64, _i64, _i64, _d, _d, _d, _st]),
    "pxf_source_beam": (_c.c_int, [_i32, _vp, _i64, _i64, _u64, _vp, _st]),
    "pxf_source_beam_from_draws": (_c.c_int, [_i32, _vp, _i64, _dp, _dp, _dp, _vp, _st]),
    # host-buffer entry point
    "pxf_host_trace_program": (_c.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "pxf_host_trace_program_hint": (_c.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _c.c_uint32]),
    "pxf_host_release": (None, []),
}

_lib = None


def lib():
    """Open libpxf.so (once) and declare every entry point.  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "pyxfocus_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` (or `make -C pyxfocus_b200/csrc`).  There is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().pxf_last_error()
        raise PxfError("libpxf error %d: %s" % (rc, msg.decode() if msg else ""))


OPT_WS_LIBM = 1
OPT_WS_RETRACE = 2
OPT_WS_GRAZE_PPM = 3


def set_option(option, value):
    """Process-wide library option (include/pxf.h, enum pxf_option)."""
    check(lib().pxf_set_option(int(option), int(value)))


def last_trace_kernel():
    """Name of the kernel the last trace launched (built-in chain, run-time specialised chain, or interpreter)."""
    return lib().pxf_last_trace_kernel().decode()


def jit_status():
    return lib().pxf_jit_status().decode()


def launch_count():
    return int(lib().pxf_launch_count())
