"""ctypes binding of libdbgsom_b200.so (the C ABI declared in include/dbgsom_b200.h).

The library is the product's only compute path: if it cannot be loaded, `load()` raises
and nothing falls back to the CPU.
"""

from __future__ import annotations

import ctypes as C
import os

_LIB = None
LIB_NAME = "libdbgsom_b200.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

ABI_VERSION = 10
COLSTATS_PARTS = 256  # DBGSOM_COLSTATS_PARTS
SELECT_OFF, SELECT_FLAG, SELECT_REFINE = 0, 1, 2
MAX_CAND = 8
BMU_SIMT = 0
BMU_TENSOR = 1
HOPS_MAX_M = 28000

c_void_p, c_int, c_int32, c_int64, c_size_t, c_float, c_double = (
    C.c_void_p, C.c_int, C.c_int32, C.c_int64, C.c_size_t, C.c_float, C.c_double,
)


class BmuArgs(C.Structure):
    _fields_ = [
        ("d_X", c_void_p),
        ("d_X16_hi", c_void_p),
        ("d_X16_lo", c_void_p),
        ("d_xnorm16", c_void_p),
        ("N", c_int64),
        ("D", c_int32),
        ("ldx", c_int64),
        ("ld16", c_int64),
        ("d_W", c_void_p),
        ("d_W32", c_void_p),
        ("d_W16_hi", c_void_p),
        ("d_W16_lo", c_void_p),
        ("d_wnorm", c_void_p),
        ("d_Wb16", c_void_p),
        ("d_bias_scale", c_void_p),
        ("d_wmax", c_void_p),
        ("d_proto_of_col", c_void_p),
        ("scale", c_float),
        ("M", c_int32),
        ("Mpad", c_int32),
        ("proto_stride", c_int32),
        ("ties_any", c_int32),
        ("n_bmu", c_int32),
        ("backend", c_int32),
        ("n_pass", c_int32),
        ("bound_scale", c_float),
        ("tie_rel", c_float),
        ("strict", c_int32),
        ("want_dist", c_int32),
        ("d_idx", c_void_p),
        ("d_dist", c_void_p),
        ("d_stats", c_void_p),
        ("d_workspace", c_void_p),
        ("workspace_bytes", c_size_t),
        ("d_row_perm", c_void_p),
        ("d_tile_mask", c_void_p),
        ("d_tile_bound", c_void_p),
        ("select", c_int32),
        ("select_granule", c_int32),
    ]


class AccumulateArgs(C.Structure):
    _fields_ = [
        ("d_X", c_void_p),
        ("N", c_int64),
        ("D", c_int32),
        ("ldx", c_int64),
        ("d_bmu", c_void_p),
        ("d_W", c_void_p),
        ("M", c_int32),
        ("inv_total_variance", c_double),
        ("d_part", c_void_p),
        ("d_labels", c_void_p),
        ("n_classes", c_int32),
        ("d_class_hist", c_void_p),
        ("d_workspace", c_void_p),
        ("workspace_bytes", c_size_t),
    ]


class SmoothArgs(C.Structure):
    _fields_ = [
        ("d_part", c_void_p),
        ("d_hop", c_void_p),
        ("ldh", c_int64),
        ("d_kernel_lut", c_void_p),
        ("lut_len", c_int32),
        ("M", c_int32),
        ("D", c_int32),
        ("pack_rows", c_int32),
        ("d_W_in", c_void_p),
        ("d_W_out", c_void_p),
        ("d_change", c_void_p),
        ("d_workspace", c_void_p),
        ("workspace_bytes", c_size_t),
        ("row_begin", c_int32),
        ("row_end", c_int32),
    ]


# name -> (restype, argtypes); every symbol include/dbgsom_b200.h declares
SIGNATURES = {
    "dbgsom_abi_version": (c_int, []),
    "dbgsom_status_string": (C.c_char_p, [c_int]),
    "dbgsom_check_device": (c_int, [c_int]),
    "dbgsom_colstats": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "dbgsom_colstats_weighted": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dbgsom_prepare_x16": (
        c_int,
        [c_void_p, c_int64, c_int, c_int64, c_void_p, c_float, c_void_p, c_void_p, c_int64, c_void_p, c_void_p],
    ),
    "dbgsom_prepare_x16_sorted": (
        c_int,
        [c_void_p, c_int64, c_int, c_int64, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p],
    ),
    "dbgsom_bmu_select_supported": (c_int, [c_int64, c_int64, c_int32, c_int32, c_int32]),
    "dbgsom_accumulate_perm_offset": (c_size_t, [c_int64, c_int32]),
    "dbgsom_prepare_w": (
        c_int,
        [c_void_p, c_int, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p,
         c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "dbgsom_exclude_duplicates": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dbgsom_tile_bounds": (
        c_int, [c_void_p, c_int, c_int, c_void_p, c_float, c_void_p, c_void_p, c_int, c_void_p, c_void_p]
    ),
    "dbgsom_prepare_bias": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dbgsom_bmu_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "dbgsom_bmu": (c_int, [C.POINTER(BmuArgs), c_void_p]),
    "dbgsom_bmu_candidates": (c_int, [C.POINTER(BmuArgs), c_void_p]),
    "dbgsom_bmu_resolve": (c_int, [C.POINTER(BmuArgs), c_void_p]),
    "dbgsom_accumulate_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "dbgsom_accumulate": (c_int, [C.POINTER(AccumulateArgs), c_void_p]),
    "dbgsom_accumulate_weighted": (c_int, [C.POINTER(AccumulateArgs), c_void_p, c_void_p, c_void_p]),
    "dbgsom_smooth_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "dbgsom_smooth": (c_int, [C.POINTER(SmoothArgs), c_void_p]),
    "dbgsom_apply_row_ops": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "dbgsom_gather_rows": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "dbgsom_node_stats": (
        c_int, [c_void_p, c_int32, c_void_p, c_int32, c_int64, c_void_p, c_int32, c_double, c_void_p, c_void_p]
    ),
    "dbgsom_node_stats_weighted": (
        c_int,
        [c_void_p, c_int32, c_void_p, c_int32, c_int64, c_void_p, c_int32, c_double, c_void_p, c_void_p, c_void_p],
    ),
    "dbgsom_umatrix": (c_int, [c_void_p, c_int32, c_int32, c_int64, c_void_p, c_void_p, c_void_p]),
    "dbgsom_label_hist": (
        c_int, [c_void_p, c_int32, c_void_p, c_int64, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]
    ),
    "dbgsom_label_hist_weighted_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "dbgsom_label_hist_weighted": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_size_t,
         c_void_p],
    ),
    "dbgsom_hops": (c_int, [c_void_p, c_int32, c_void_p, c_int64, c_void_p]),
    "dbgsom_sparse_code_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "dbgsom_sparse_code": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
         c_size_t, c_void_p],
    ),
}


class NativeError(RuntimeError):
    pass


def load():
    """Load the shared library once; raise NativeError if it is missing or mismatched."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} not found. Build it with `python -m dbgsom_b200.build` (needs nvcc); "
            "dbgsom_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise NativeError(f"{LIB_NAME} does not export {name}; rebuild it") from exc
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.dbgsom_abi_version() != ABI_VERSION:
        raise NativeError(f"{LIB_NAME} has ABI {lib.dbgsom_abi_version()}, expected {ABI_VERSION}; rebuild it")
    _LIB = lib
    return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().dbgsom_status_string(status)
        raise NativeError(f"{what} failed with status {status}: {msg.decode() if msg else '?'}")
