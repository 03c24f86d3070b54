"""ctypes binding of libnrb200.so (the C-ABI declared in include/nrb200.h).

There is deliberately no fallback: if the shared library is missing, importing this module
raises, and on a machine without an sm_100 GPU the compute entry points return
NRB_ERR_NO_DEVICE which `check()` turns into a RuntimeError.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# NRB_LIB selects another build of the same library (e.g. libnrb200_trace.so, `make trace`)
LIB_PATH = os.environ.get("NRB_LIB") or os.path.join(_PKG, "libnrb200.so")

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
PATH_AUTO, PATH_SIMT, PATH_TC, PATH_TC1, PATH_TC16 = 0, 1, 2, 3, 4
MAX_K = 128
SMALL_MAX_NQ = 64  # NRB_SMALL_MAX_NQ

# every symbol include/nrb200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "nrb_version", "nrb_last_error", "nrb_device_info", "nrb_launch_count",
    "nrb_profile_enable", "nrb_profile_read",
    "nrb_pack_rows", "nrb_pack_rows_h16", "nrb_gather_rows", "nrb_gather_i64", "nrb_normalize_l2",
    "nrb_search_flat_workspace", "nrb_search_flat", "nrb_fallback_query_count", "nrb_plan_flat_describe",
    "nrb_kmeans_update_workspace", "nrb_kmeans_update", "nrb_kmeans_partial_sums", "nrb_kmeans_means",
    "nrb_rand_perm_host", "nrb_split_clusters_host", "nrb_split_clusters",
    "nrb_kmeans_train_workspace", "nrb_kmeans_train",
    "nrb_ivf_build_lists_workspace", "nrb_ivf_build_lists",
    "nrb_ivf_search_workspace", "nrb_ivf_search",
    "nrb_merge_topk", "nrb_expand_lists", "nrb_csr_contains",
    "nrb_pack_topk", "nrb_merge_topk_packed",
    "nrb_search_small_workspace", "nrb_search_small", "nrb_search_small_host",
    "nrb_ivf_scan_small_workspace", "nrb_ivf_scan_small", "nrb_split_table_f64",
    "nrb_id_select_workspace", "nrb_id_select", "nrb_map_ids",
    "nrb_search_small_sel", "nrb_search_small_host_sel", "nrb_ivf_scan_small_sel", "nrb_sel_keys",
    "nrb_pack_topk_ids", "nrb_merge_topk_packed_ids", "nrb_exclude_topk",
    "nrb_csr_compact_workspace", "nrb_csr_compact",
]


class Matrix(C.Structure):
    """struct nrb_matrix"""
    _fields_ = [("raw", C.c_void_p), ("hi", C.c_void_p), ("lo", C.c_void_p), ("norms", C.c_void_p),
                ("n", C.c_int64), ("d", C.c_int32), ("kp", C.c_int32), ("max_norm", C.c_float),
                ("h16_scale", C.c_float), ("h16", C.c_void_p), ("h16_row_scale", C.c_void_p)]


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C newsrecommend_b200/csrc`. newsrecommend_b200 has no CPU / eager fallback.")

lib = C.CDLL(LIB_PATH)

_vp, _i64, _i32, _sz = C.c_void_p, C.c_int64, C.c_int32, C.c_size_t
_mp = C.POINTER(Matrix)

lib.nrb_version.restype = C.c_int
lib.nrb_last_error.argtypes = [C.c_char_p, C.c_int]
lib.nrb_device_info.argtypes = [C.POINTER(C.c_int)] * 3
lib.nrb_launch_count.restype = _i64
lib.nrb_profile_enable.argtypes = [C.c_int]
lib.nrb_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int)]
lib.nrb_pack_rows.argtypes = [_vp, _i64, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp]
lib.nrb_pack_rows_h16.argtypes = [_vp, _i64, _i32, _i64, _i32, C.c_float, _vp, _vp, _vp]
lib.nrb_gather_rows.argtypes = [_vp, _i32, _vp, _i64, _vp, _vp]
lib.nrb_gather_i64.argtypes = [_vp, _vp, _i64, _vp, _vp]
lib.nrb_normalize_l2.argtypes = [_vp, _i64, _i32, _i64, _vp]
lib.nrb_search_flat_workspace.restype = _sz
lib.nrb_search_flat_workspace.argtypes = [_i64, _i64, _i32, _i32]
lib.nrb_search_flat.argtypes = [_mp, _mp, _i32, _i32, _i64, _vp, _vp, _vp, _sz, _i32, _vp]
lib.nrb_fallback_query_count.restype = _i64
lib.nrb_plan_flat_describe.argtypes = [_i64, _i64, _i32, _i32, _vp]
lib.nrb_kmeans_update_workspace.restype = _sz
lib.nrb_kmeans_update_workspace.argtypes = [_i64, _i32, _i32]
lib.nrb_kmeans_update.argtypes = [_vp, _i64, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _sz, _vp]
lib.nrb_kmeans_partial_sums.argtypes = [_vp, _i64, _i32, _i32, _vp, _i32, _vp, _vp, _sz, _vp]
lib.nrb_kmeans_means.argtypes = [_vp, _i32, _i32, _vp, _vp, _vp]
lib.nrb_rand_perm_host.argtypes = [_vp, _i64, _i64]
lib.nrb_split_clusters_host.argtypes = [_i32, _i32, _i64, _vp, _vp]
lib.nrb_split_clusters.argtypes = [_i32, _i32, _i64, _vp, _vp, _vp, _vp]
lib.nrb_kmeans_train_workspace.restype = _sz
lib.nrb_kmeans_train_workspace.argtypes = [_i64, _i32, _i32]
lib.nrb_kmeans_train.argtypes = [_mp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _sz, _vp]
lib.nrb_ivf_build_lists_workspace.restype = _sz
lib.nrb_ivf_build_lists_workspace.argtypes = [_i64, _i32]
lib.nrb_ivf_build_lists.argtypes = [_vp, _i64, _i32, _vp, _vp, _vp, _sz, _vp]
lib.nrb_ivf_search_workspace.restype = _sz
lib.nrb_ivf_search_workspace.argtypes = [_i64, _i32, _i32, _i32, _i32, _i32]
lib.nrb_ivf_search.argtypes = [_mp, _mp, _vp, _i32, _i32, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _sz,
                               _i32, _vp]
lib.nrb_merge_topk.argtypes = [_vp, _vp, _i32, _i64, _i32, _i32, _vp, _vp, _vp]
lib.nrb_pack_topk.argtypes = [_vp, _vp, _i64, _i64, _vp, _vp]
lib.nrb_merge_topk_packed.argtypes = [_vp, _vp, _i32, _i64, _i32, _i32, _vp, _vp, _vp]
lib.nrb_search_small_workspace.restype = _sz
lib.nrb_search_small_workspace.argtypes = [_i64, _i64, _i32]
lib.nrb_search_small.argtypes = [_vp, _i64, _i32, _i32, _mp, _i32, _i32, _i64, _vp, _vp, _vp, _sz, _vp]
lib.nrb_search_small_host.argtypes = [_mp, _vp, _i32, _i32, _i32, _i32, _i64, _vp, _vp, _vp]
lib.nrb_ivf_scan_small_workspace.restype = _sz
lib.nrb_ivf_scan_small_workspace.argtypes = [_i64, _i32, _i32, _i64, _i32]
lib.nrb_ivf_scan_small.argtypes = [_vp, _i64, _i32, _i32, _mp, _vp, _i32, _i32, _vp, _vp, _i32, _i32, _i32, _vp, _vp,
                                   _vp, _sz, _vp]
lib.nrb_split_table_f64.argtypes = [_vp, _i64, _i32, _vp, _vp, _vp]
lib.nrb_expand_lists.argtypes = [_vp, _vp, _vp, _vp, _i64, _vp, _vp]
lib.nrb_csr_contains.argtypes = [_vp, _vp, _vp, _i64, _vp, _vp]
lib.nrb_id_select_workspace.restype = _sz
lib.nrb_id_select_workspace.argtypes = [_i64]
lib.nrb_id_select.argtypes = [_vp, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _sz, _vp]
lib.nrb_map_ids.argtypes = [_vp, _vp, _i64, _vp]
lib.nrb_search_small_sel.argtypes = lib.nrb_search_small.argtypes + [_vp, _i64]
lib.nrb_search_small_host_sel.argtypes = lib.nrb_search_small_host.argtypes + [_vp, _i64]
lib.nrb_ivf_scan_small_sel.argtypes = lib.nrb_ivf_scan_small.argtypes + [_vp, _i64]
lib.nrb_sel_keys.argtypes = [_vp, _i64, _vp, _i64, _i64, _vp, _vp]
lib.nrb_pack_topk_ids.argtypes = [_vp, _vp, _i64, _vp, _vp]
lib.nrb_merge_topk_packed_ids.argtypes = [_vp, _i32, _i64, _i32, _i32, _vp, _vp, _vp]
lib.nrb_exclude_topk.argtypes = [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp]
lib.nrb_csr_compact_workspace.restype = _sz
lib.nrb_csr_compact_workspace.argtypes = [_i64]
lib.nrb_csr_compact.argtypes = [_vp, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _sz, _vp]


def last_error() -> str:
    buf = C.create_string_buffer(512)
    lib.nrb_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def check(rc: int, what: str = "") -> int:
    """Raise RuntimeError (what faiss's SWIG layer turns a FaissException into) on failure."""
    if rc < 0:
        raise RuntimeError(f"libnrb200 {what} failed (code {rc}): {last_error()}")
    return rc


def profile_enable(on: bool) -> None:
    lib.nrb_profile_enable(1 if on else 0)


def profile_read():
    """(total ms, launches) of the dominant kernel since the last read."""
    ms, n = C.c_double(0), C.c_int(0)
    lib.nrb_profile_read(C.byref(ms), C.byref(n))
    return ms.value, n.value


def launch_count() -> int:
    return int(lib.nrb_launch_count())
