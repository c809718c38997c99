"""ctypes binding of the C ABI in include/chronoclust_b200.h.

The shared library is built in-tree by chronoclust_b200/build.py (nvcc, sm_100a).  There is no CPU
fallback: if the library cannot be loaded, or no CUDA device is present when a handle is created, the
caller gets an exception.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libchronoclust_b200.so")
_LIB = None

i32, i64, f64, u8 = C.c_int32, C.c_int64, C.c_double, C.c_uint8
vp = C.c_void_p


class Params(C.Structure):
    _fields_ = [("D", i32), ("device", i32), ("eps2", f64), ("upsilon_eps", f64), ("upsilon_eps2", f64),
                ("delta", f64), ("delta2", f64), ("beta", f64), ("k", f64), ("chunk", i32),
                ("bsv_bmin", i32), ("bsv_iters", i32), ("bsv_stream", i32), ("off_csr_min_m", i32), ("reserved0", i32)]


class Stats(C.Structure):
    _fields_ = [(n, i64) for n in (
        "points", "nearest_pairs", "upgrades", "created", "downgraded", "deleted", "kernel_launches", "borderline_pairs",
        "bsv_blocks", "bsv_rounds", "bsv_mismatches", "bsv_cuts_unknown", "bsv_cuts_rounds", "bsv_cuts_capacity",
        "bsv_late_topk", "bsv_outlier_stage_cells", "bsv_replayed_cells", "bsv_light_rounds", "bsv_serial_cells", "bsv_pdl")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


# every symbol include/chronoclust_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "ccb_create": (C.c_int, [C.POINTER(Params), C.POINTER(vp)]),
    "ccb_destroy": (None, [vp]),
    "ccb_last_error": (C.c_char_p, [vp]),
    "ccb_stream": (vp, [vp]),
    "ccb_get_stats": (C.c_int, [vp, C.POINTER(Stats)]),
    "ccb_reset": (C.c_int, [vp]),
    "ccb_fp64_peak": (C.c_int, [i32, vp, i32, i32, i32, vp, C.POINTER(f64)]),
    "ccb_enable_timing": (C.c_int, [vp, i32]),
    "ccb_get_timing": (C.c_int, [vp, C.POINTER(f64 * 16), C.POINTER(i64 * 16), i32]),
    "ccb_set_dnrm2": (C.c_int, [vp, vp]),
    "ccb_begin_timepoint": (C.c_int, [vp, f64, f64, i64, i32, f64]),
    "ccb_ingest": (C.c_int, [vp, vp, i64, i64, vp, vp]),
    "ccb_ingest_device": (C.c_int, [vp, vp, i64, i64, vp, vp]),
    "ccb_ingest_ex": (C.c_int, [vp, vp, i32, i32, i64, i64, vp, vp, vp, vp]),
    "ccb_ingest_cols": (C.c_int, [vp, vp, i32, i32, i64, i64, i32, vp, vp, vp, vp, vp]),
    "ccb_ingest_tx": (C.c_int, [vp, vp, i32, i32, i64, i64, i32, vp, vp, vp, vp, vp, vp]),
    "ccb_offline": (C.c_int, [vp, C.POINTER(i64)]),
    "ccb_counts": (C.c_int, [vp, C.POINTER(i64 * 4)]),
    "ccb_export_list": (C.c_int, [vp, i32] + [vp] * 7),
    "ccb_import_list": (C.c_int, [vp, i32, i64] + [vp] * 7),
    "ccb_set_counters": (C.c_int, [vp, i64, i64]),
    "ccb_cluster_sizes": (C.c_int, [vp, C.POINTER(i64 * 3)]),
    "ccb_export_clusters": (C.c_int, [vp] + [vp] * 8),
    "ccb_export_offline": (C.c_int, [vp] + [vp] * 4),
    "ccb_nearest": (C.c_int, [i32, vp, vp, i64, i64, i32, vp, vp, i64, f64, vp, vp]),
    "ccb_assoc_nearest": (C.c_int, [i32, vp, vp, vp, i64, vp, i64, i32, f64, vp, vp]),
    "ccb_assoc_nearest2": (C.c_int, [i32, vp, vp, vp, i64, vp, i64, i32, f64, vp, vp, vp]),
    "ccb_colminmax": (C.c_int, [i32, vp, vp, i64, i64, i32, vp, vp]),
    "ccb_colminmax_ex": (C.c_int, [i32, vp, vp, i32, i64, i64, i32, vp, vp]),
    "ccb_arcsinh": (C.c_int, [i32, vp, vp, i32, i64, i64, i32, vp, vp]),
    "ccb_ingest_scaled": (C.c_int, [vp, vp, i64, i64, vp, vp, vp, vp]),
    "ccb_off_neighbours": (C.c_int, [i32, vp, vp, i64, i32, i64, i64, f64, f64, vp, vp, vp, C.POINTER(i64)]),
    "ccb_off_subspace": (C.c_int, [i32, vp, vp, i64, i32, i64, i64, vp, vp, f64, vp]),
    "ccb_off_weighted": (C.c_int, [i32, vp, vp, i64, i32, i64, i64, vp, vp, f64, f64, vp]),
    "ccb_off_clusters": (C.c_int, [i32, vp, i64, vp, vp, vp, f64, i64, i32, vp, vp, vp, vp]),
    "ccb_offc_rowinfo": (C.c_int, [i32, vp, vp, i64, i64, i64, vp, vp]),
    "ccb_offc_fill": (C.c_int, [i32, vp, vp, i64, i64, i64, vp, vp, vp]),
    "ccb_off_clusters_csr": (C.c_int, [i32, vp, i64, vp, vp, vp, vp, vp, f64, i64, vp, vp, vp, vp]),
    "ccb_group_stats": (C.c_int, [i32, vp, vp, i32, i64, i64, i32, vp, i32, i32, vp, vp, vp, vp, vp]),
    "ccb_cluster_stats": (C.c_int, [vp, vp, i64, i32, i32, vp, vp, vp, vp, vp]),
}


DTYPE_F64, DTYPE_F32 = 0, 1  # CCB_DTYPE_*

CATEGORIES = ["chain_p", "nearest", "verify", "maintenance", "offline", "misc", "copy", "speculate", "lists", "chain_o",
              "olist", "derive", "decide", "commit", "reserved14", "reserved15"]


class CCBError(RuntimeError):
    pass


def lib():
    """Loads the CUDA library; raises if it is missing (never falls back to a CPU path)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise CCBError(f"{SO_PATH} is missing: build it with `python -m chronoclust_b200.build` "
                           "(or __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _LIB = L
    return _LIB


def check(rc, handle=None):
    if rc != 0:
        msg = lib().ccb_last_error(handle)
        raise CCBError(f"chronoclust_b200 error {rc}: {msg.decode() if msg else '?'}")


def ptr(a):
    return None if a is None else a.ctypes.data_as(vp)


def scipy_dnrm2_pointer():
    """Address of the BLAS dnrm2 numba binds for np.linalg.norm (the reference's Euclidean norm,
    predeconmc_functions.py:16-17): scipy.linalg.cython_blas.__pyx_capi__['dnrm2']."""
    import scipy.linalg.cython_blas as cb

    cap = cb.__pyx_capi__["dnrm2"]
    C.pythonapi.PyCapsule_GetName.restype = C.c_char_p
    C.pythonapi.PyCapsule_GetName.argtypes = [C.py_object]
    C.pythonapi.PyCapsule_GetPointer.restype = vp
    C.pythonapi.PyCapsule_GetPointer.argtypes = [C.py_object, C.c_char_p]
    return C.pythonapi.PyCapsule_GetPointer(cap, C.pythonapi.PyCapsule_GetName(cap))
