"""ctypes binding of libscann_b200.so (include/scann_b200.h).  No torch types cross this boundary:
host buffers are numpy arrays, device buffers are raw pointers (e.g. ``tensor.data_ptr()``)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

OK = 0
INVALID_ARGUMENT = 3
RESOURCE_EXHAUSTED = 8
FAILED_PRECONDITION = 9
OUT_OF_RANGE = 11
UNIMPLEMENTED = 12
INTERNAL = 13
UNAVAILABLE = 14
_CODE_NAMES = {
    0: "OK", 1: "CANCELLED", 2: "UNKNOWN", 3: "INVALID_ARGUMENT", 4: "DEADLINE_EXCEEDED", 5: "NOT_FOUND",
    6: "ALREADY_EXISTS", 7: "PERMISSION_DENIED", 8: "RESOURCE_EXHAUSTED", 9: "FAILED_PRECONDITION", 10: "ABORTED",
    11: "OUT_OF_RANGE", 12: "UNIMPLEMENTED", 13: "INTERNAL", 14: "UNAVAILABLE", 15: "DATA_LOSS",
    16: "UNAUTHENTICATED",
}

SQL2, L2, DOT = 0, 1, 2
TREEAH_RAW_BY_POSITION, TREEAH_BORROW_RAW = 1, 2
HOST, DEVICE = 0, 1

# every symbol include/scann_b200.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "scann_last_error", "scann_version", "scann_device_count",
    "scann_bf_create", "scann_bf_search", "scann_bf_search_radius", "scann_bf_destroy", "scann_bf_path_stats", "scann_sq8_path_stats",
    "scann_sq8_quantize", "scann_sq8_create", "scann_sq8_search", "scann_sq8_destroy",
    "scann_part_create", "scann_part_select", "scann_part_destroy", "scann_part_update",
    "scann_treeah_create", "scann_treeah_create_ex", "scann_treeah_search", "scann_treeah_search_filtered", "scann_treeah_search_with_params", "scann_treeah_destroy", "scann_treeah_last_scan_bytes",
    "scann_treeah_set_profiling", "scann_treeah_get_profile", "scann_treeah_search_begin", "scann_treeah_search_end", "scann_treeah_search_abort", "scann_treeah_partition",
    "scann_treeah_set_filter", "scann_treeah_path_stats", "scann_treeah_tc_profile",
    "scann_lut16_build", "scann_lut16_scan", "scann_pq_encode", "scann_merge_topk", "scann_merge_topk_packed", "scann_tc_scores",
    "scann_ivf_create", "scann_ivf_search", "scann_ivf_destroy",
    "scann_kmtree_create", "scann_kmtree_build", "scann_kmtree_info", "scann_kmtree_export", "scann_kmtree_search_leaves",
    "scann_kmtree_destroy",
    "scann_kmeans_fit", "scann_pq_train", "scann_treeah_build", "scann_ivf_build", "scann_treeah_set_reorder",
]


class ScannError(Exception):
    """Mirror of the reference's ScannError {code, message} (src/error.rs:72-76)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"{_CODE_NAMES.get(code, code)}: {message}")
        self.code = code
        self.message = message


_lib = None


def lib_path() -> str:
    return _build.LIB


def load():
    """Loads the CUDA library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ScannError(UNAVAILABLE, f"{path} is not built; run __graft_entry__.build() "
                                      "(there is no CPU fallback for the product path)")
    L = C.CDLL(path)
    vp, sz, i32, f32 = C.c_void_p, C.c_size_t, C.c_int, C.c_float
    L.scann_last_error.restype = C.c_char_p
    L.scann_version.restype = i32
    L.scann_device_count.argtypes = [C.POINTER(i32)]
    L.scann_bf_create.argtypes = [vp, sz, sz, sz, i32, i32, i32, C.POINTER(vp)]
    L.scann_bf_search.argtypes = [vp, vp, sz, sz, sz, vp, vp, vp, i32, vp]
    L.scann_bf_search_radius.argtypes = [vp, vp, sz, sz, f32, sz, vp, vp, vp, i32, vp]
    L.scann_bf_destroy.argtypes = [vp]
    L.scann_bf_path_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.scann_sq8_path_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.scann_bf_destroy.restype = None
    L.scann_sq8_quantize.argtypes = [vp, sz, sz, sz, vp, vp, i32, i32]
    L.scann_sq8_create.argtypes = [vp, sz, sz, f32, i32, i32, i32, C.POINTER(vp)]
    L.scann_sq8_search.argtypes = [vp, vp, sz, sz, sz, vp, vp, vp, i32, vp]
    L.scann_sq8_destroy.argtypes = [vp]
    L.scann_sq8_destroy.restype = None
    L.scann_part_create.argtypes = [vp, sz, sz, i32, i32, C.POINTER(vp)]
    L.scann_part_select.argtypes = [vp, vp, sz, sz, sz, vp, vp, i32, vp]
    L.scann_part_destroy.argtypes = [vp]
    L.scann_part_update.argtypes = [vp, vp, i32]
    L.scann_part_destroy.restype = None
    L.scann_treeah_create.argtypes = [vp, sz, sz, vp, sz, vp, vp, vp, sz, vp, sz, sz, i32, i32, i32, i32,
                                      C.POINTER(vp)]
    L.scann_treeah_create_ex.argtypes = [vp, sz, sz, vp, sz, vp, vp, vp, sz, vp, sz, sz, i32, i32, C.c_uint32, i32, i32,
                                         C.POINTER(vp)]
    L.scann_treeah_search.argtypes = [vp, vp, sz, sz, sz, sz, sz, vp, vp, vp, vp, vp, vp, i32, vp]
    L.scann_treeah_search_filtered.argtypes = [vp, vp, sz, sz, sz, sz, sz, vp, sz, sz, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    L.scann_treeah_search_with_params.argtypes = [vp, vp, sz, sz, sz, sz, sz, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    L.scann_treeah_destroy.argtypes = [vp]
    L.scann_treeah_destroy.restype = None
    L.scann_treeah_last_scan_bytes.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.scann_treeah_search_begin.argtypes = [vp, vp, sz, sz, sz, sz, sz, vp, vp, vp]
    L.scann_treeah_set_filter.argtypes = [vp, vp, sz, i32]
    L.scann_treeah_partition.argtypes = [vp, vp, sz, sz, sz, vp, vp]
    L.scann_treeah_search_end.argtypes = [vp, vp, vp, vp, vp, vp]
    L.scann_treeah_search_abort.argtypes = [vp]
    L.scann_treeah_path_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.scann_treeah_tc_profile.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64),
                                          C.POINTER(C.c_uint64)]
    L.scann_treeah_set_profiling.argtypes = [vp, i32]
    L.scann_treeah_get_profile.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.scann_lut16_build.argtypes = [vp, sz, sz, vp, sz, vp, vp, vp, vp, i32, i32]
    L.scann_lut16_scan.argtypes = [vp, sz, sz, vp, vp, i32, i32]
    L.scann_pq_encode.argtypes = [vp, sz, sz, vp, sz, sz, vp, vp, vp, i32, i32]
    L.scann_merge_topk.argtypes = [vp, vp, sz, sz, sz, vp, vp, vp, i32, i32, vp]
    L.scann_ivf_create.argtypes = [vp, sz, sz, vp, vp, sz, vp, sz, sz, vp, sz, sz, vp, i32, i32, C.POINTER(vp)]
    L.scann_ivf_search.argtypes = [vp, i32, vp, sz, sz, sz, sz, i32, i32, vp, vp, vp, i32, vp]
    L.scann_ivf_destroy.argtypes = [vp]
    L.scann_ivf_destroy.restype = None
    L.scann_merge_topk_packed.argtypes = [vp, sz, sz, sz, vp, vp, vp, i32, vp]
    L.scann_tc_scores.argtypes = [vp, sz, sz, vp, i32, sz, sz, f32, i32, vp, vp, vp, sz, vp, i32]
    u64 = C.c_uint64
    L.scann_kmeans_fit.argtypes = [vp, sz, sz, sz, sz, i32, u64, f32, vp, i32, i32]
    L.scann_pq_train.argtypes = [vp, sz, sz, sz, vp, vp, sz, sz, i32, u64, vp, i32, i32]
    L.scann_treeah_build.argtypes = [vp, sz, sz, sz, sz, sz, sz, i32, u64, i32, i32, i32, i32, i32, C.POINTER(vp)]
    L.scann_ivf_build.argtypes = [vp, sz, sz, sz, sz, i32, u64, i32, i32, C.POINTER(vp)]
    L.scann_treeah_set_reorder.argtypes = [vp, i32]
    L.scann_kmtree_create.argtypes = [vp, vp, vp, vp, vp, sz, sz, sz, i32, C.POINTER(vp)]
    L.scann_kmtree_build.argtypes = [vp, sz, sz, sz, sz, sz, sz, i32, u64, i32, i32, C.POINTER(vp)]
    L.scann_kmtree_info.argtypes = [vp] + [C.POINTER(sz)] * 5
    L.scann_kmtree_export.argtypes = [vp] * 9
    L.scann_kmtree_search_leaves.argtypes = [vp, vp, sz, sz, sz, vp, vp, vp, vp, i32, vp]
    L.scann_kmtree_destroy.argtypes = [vp]
    L.scann_kmtree_destroy.restype = None
    for name in SYMBOLS:
        fn = getattr(L, name)
        if name not in ("scann_last_error", "scann_version") and not name.endswith("_destroy"):
            fn.restype = C.c_int32
    _lib = L
    return L


def check(status: int):
    if status != OK:
        msg = load().scann_last_error()
        raise ScannError(status, msg.decode("utf-8", "replace") if msg else "")


def device_count() -> int:
    n = C.c_int(0)
    st = load().scann_device_count(C.byref(n))
    return n.value if st == OK else 0


def require_gpu():
    if device_count() <= 0:
        raise ScannError(UNAVAILABLE, "no CUDA device: the scann-rust_b200 product path has no CPU fallback")


def np_ptr(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def as_f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)
