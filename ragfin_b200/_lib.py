"""ctypes binding of the C ABI in include/ragfin.h (libragfin.so, built for sm_100a).

The library is the product: there is no Python or CPU fallback.  If it has not been built,
importing this module raises with the build command.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# RAGFIN_LIB selects another build of the SAME library (e.g. one made with EXTRA=-DRAGFIN_TIMING_EXPERIMENTS);
# it is not a fallback: a missing file raises like the default does.
SO_PATH = os.environ.get("RAGFIN_LIB") or os.path.join(CSRC, "libragfin.so")

# every symbol include/ragfin.h declares
SYMBOLS = (
    "ragfin_abi_version", "ragfin_create", "ragfin_create_view", "ragfin_add", "ragfin_add_synthetic", "ragfin_add_synthetic_topics", "ragfin_count", "ragfin_reserve",
    "ragfin_delete", "ragfin_live_count", "ragfin_read_live_mask", "ragfin_compact",
    "ragfin_set_id_base", "ragfin_search", "ragfin_search_host", "ragfin_search_filtered", "ragfin_search_filtered_host", "ragfin_search_range", "ragfin_search_range_host", "ragfin_search_grouped", "ragfin_search_grouped_host", "ragfin_merge_topk", "ragfin_read_rows", "ragfin_read_sweep_rows",
    "ragfin_last_search_stats", "ragfin_profile", "ragfin_profile_read", "ragfin_save", "ragfin_load", "ragfin_set_gemm_min_batch", "ragfin_set_gemm_cluster", "ragfin_set_gemm_variant", "ragfin_set_bound_pass", "ragfin_set_scan_variant", "ragfin_set_append_mode", "ragfin_set_fused", "ragfin_set_pipelined", "ragfin_debug_fused_counts", "ragfin_debug_fused_times", "ragfin_debug_fused_ctas", "ragfin_debug_fused_tile_order", "ragfin_debug_gemm_scores", "ragfin_debug_plan", "ragfin_destroy", "ragfin_last_error",
    "ragfin_exchange_create", "ragfin_exchange_handle", "ragfin_exchange_connect", "ragfin_exchange_allgather_merge", "ragfin_fused_eligible", "ragfin_search_sharded", "ragfin_search_sharded_host", "ragfin_exchange_destroy",
)

OK, EINVAL, ECUDA, ENOMEM, EUNSUPPORTED = 0, -1, -2, -3, -4


class RagfinError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"ragfin error {code}: {message}")
        self.code = code


class SearchStats(ctypes.Structure):
    _fields_ = [("launches", ctypes.c_int32), ("path", ctypes.c_int32),
                ("queries_rescanned", ctypes.c_int32), ("cand_per_query", ctypes.c_int32)]


_lib = None


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(
            f"{SO_PATH} is missing: build it with `make -C {CSRC}` (or `python -c 'import __graft_entry__ as g; "
            f"g.build()'`). ragfin_b200 has no CPU fallback.")
    L = ctypes.CDLL(SO_PATH)
    vp, i32, i64, u64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64
    L.ragfin_abi_version.argtypes, L.ragfin_abi_version.restype = [], ctypes.c_int
    L.ragfin_create.argtypes = [ctypes.POINTER(vp), i32, i32, i64, i32]
    L.ragfin_create_view.argtypes = [vp, ctypes.POINTER(vp)]
    L.ragfin_add.argtypes = [vp, vp, i64, i32, vp]
    L.ragfin_add_synthetic.argtypes = [vp, u64, i64, i64, i32, i32, vp]
    L.ragfin_add_synthetic_topics.argtypes = [vp, u64, i64, i64, i64, i32, vp]
    L.ragfin_count.argtypes = [vp, ctypes.POINTER(i64)]
    L.ragfin_delete.argtypes = [vp, vp, i64, ctypes.POINTER(i64)]
    L.ragfin_live_count.argtypes = [vp, ctypes.POINTER(i64)]
    L.ragfin_read_live_mask.argtypes = [vp, vp]
    L.ragfin_compact.argtypes = [vp]
    L.ragfin_set_id_base.argtypes = [vp, i64]
    L.ragfin_reserve.argtypes = [vp, i64]
    L.ragfin_search.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    L.ragfin_search_host.argtypes = [vp, vp, i32, i32, vp, vp]
    L.ragfin_search_filtered.argtypes = [vp, vp, i32, i32, vp, i64, vp, vp, vp]
    L.ragfin_search_filtered_host.argtypes = [vp, vp, i32, i32, vp, i64, vp, vp]
    L.ragfin_search_range.argtypes = [vp, vp, i32, i32, vp, vp, i64, vp, vp, vp]   # range: ctypes.c_float * 2 {radius, range_filter}
    L.ragfin_search_range_host.argtypes = [vp, vp, i32, i32, vp, vp, i64, vp, vp]
    L.ragfin_search_grouped.argtypes = [vp, vp, i32, i32, vp, i32, vp, i64, vp, vp, vp]
    L.ragfin_search_grouped_host.argtypes = [vp, vp, i32, i32, vp, i32, i32, vp, i64, vp, vp]
    L.ragfin_merge_topk.argtypes = [vp, vp, i32, i32, i32, i64, i64, i64, vp, vp, i32, vp]
    L.ragfin_profile.argtypes = [vp, i32]
    L.ragfin_save.argtypes = [vp, ctypes.c_char_p]
    L.ragfin_load.argtypes = [ctypes.POINTER(vp), ctypes.c_char_p, i64, i32]
    L.ragfin_set_gemm_min_batch.argtypes = [vp, i32]
    L.ragfin_set_gemm_cluster.argtypes = [vp, i32]
    L.ragfin_set_gemm_variant.argtypes = [vp, i32]
    L.ragfin_set_bound_pass.argtypes = [vp, i32]
    L.ragfin_exchange_create.argtypes = [ctypes.POINTER(vp), i32, i32, i64, i32]
    L.ragfin_exchange_handle.argtypes = [vp, vp]
    L.ragfin_exchange_connect.argtypes = [vp, vp]
    L.ragfin_exchange_allgather_merge.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp]
    L.ragfin_exchange_destroy.argtypes = [vp]
    L.ragfin_fused_eligible.argtypes = [vp, i32, i32, ctypes.POINTER(i32)]
    L.ragfin_search_sharded.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp]
    L.ragfin_search_sharded_host.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    L.ragfin_exchange_destroy.restype = None
    L.ragfin_set_scan_variant.argtypes = [vp, i32]
    L.ragfin_set_append_mode.argtypes = [vp, i32]
    L.ragfin_set_fused.argtypes = [vp, i32, i64]
    L.ragfin_set_pipelined.argtypes = [vp, i32]
    L.ragfin_debug_fused_counts.argtypes = [vp, i32, vp, vp]
    L.ragfin_debug_fused_times.argtypes = [vp, vp]
    L.ragfin_debug_fused_ctas.argtypes = [vp, vp, vp]
    L.ragfin_debug_fused_tile_order.argtypes = [i32, vp]
    L.ragfin_debug_gemm_scores.argtypes = [vp, vp, i32, vp, vp]
    L.ragfin_debug_plan.argtypes = [i32, i64, i32, i32, i32, ctypes.POINTER(i64)]
    L.ragfin_profile_read.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i32)]
    L.ragfin_read_rows.argtypes = [vp, i64, i64, vp, ctypes.POINTER(i32)]
    L.ragfin_read_sweep_rows.argtypes = [vp, i64, i64, vp, ctypes.POINTER(i32)]
    L.ragfin_last_search_stats.argtypes = [vp, ctypes.POINTER(SearchStats)]
    for name in SYMBOLS:
        if name not in ("ragfin_destroy", "ragfin_last_error", "ragfin_exchange_destroy"):
            getattr(L, name).restype = ctypes.c_int
    L.ragfin_destroy.argtypes, L.ragfin_destroy.restype = [vp], None
    L.ragfin_last_error.argtypes, L.ragfin_last_error.restype = [], ctypes.c_char_p
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise RagfinError(rc, load().ragfin_last_error().decode("utf-8", "replace"))
