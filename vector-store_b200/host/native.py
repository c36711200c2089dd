"""ctypes binding of libvsb200.so — the same symbols the Rust FFI crate binds (INTEGRATION.md)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# VSB200_LIB: an instrumented build of the same library (tools/ profiling runs); never a different backend
_LIB_PATH = os.environ.get("VSB200_LIB") or os.path.join(os.path.dirname(_HERE), "libvsb200.so")

VSB_OK, VSB_EINVAL, VSB_EDIM, VSB_EDUPKEY, VSB_EFULL, VSB_EOOM, VSB_ECUDA, VSB_ENCCL = range(8)
STATUS_NAMES = ["OK", "EINVAL", "EDIM", "EDUPKEY", "EFULL", "EOOM", "ECUDA", "ENCCL"]


class VsbError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"vsb200 {STATUS_NAMES[status] if 0 <= status < 8 else status}: {message}")
        self.status = status


class VsbOptions(C.Structure):
    _fields_ = [("dimensions", C.c_uint32), ("metric", C.c_int32), ("storage", C.c_int32),
                ("connectivity", C.c_uint32), ("expansion_add", C.c_uint32), ("expansion_search", C.c_uint32),
                ("device", C.c_int32), ("flags", C.c_uint32), ("seed", C.c_uint64),
                ("n_devices", C.c_int32), ("device_ids", C.c_int32 * 8)]


class VsbSearchParams(C.Structure):
    _fields_ = [("expansion_search", C.c_uint32), ("max_iterations", C.c_uint32), ("n_seeds", C.c_uint32),
                ("min_graph_size", C.c_uint32), ("search_width", C.c_uint32), ("stream_threshold", C.c_uint32),
                ("filter_exact_below_pct", C.c_uint32), ("expansion_add", C.c_uint32), ("traversal", C.c_uint32),
                ("reserved", C.c_uint32)]


class VsbStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("kernel_launches", "distance_evals", "parent_expansions", "queries",
                                          "n_slots", "n_graphed", "graph_degree", "row_bytes", "n_seed_rows",
                                          "hbm_bytes", "convert_ns", "seed_ns", "graph_search_ns", "exact_ns",
                                          "merge_ns", "convert_launches", "seed_launches", "graph_search_launches",
                                          "exact_launches", "merge_launches", "tc_launches",
                                          "exact_certified", "exact_fallback", "exact_scanned", "extra_seeds")]


class VsbBuildStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rows", "allpairs_rows", "allpairs_flops", "allpairs_ns", "prune_ns",
                                          "stream_rows", "stream_evals", "stream_parents", "stream_ns",
                                          "refine_rows", "refine_evals", "refine_parents", "refine_ns", "seeds_ns",
                                          "compact_ns", "total_ns", "traversal_row_bytes")]


XCHG_HANDLE_BYTES = 64

# every symbol include/vsb200.h declares: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("vsb_create", C.c_int, [C.POINTER(VsbOptions), C.POINTER(_P)]),
    ("vsb_destroy", None, [_P]),
    ("vsb_reserve", C.c_int, [_P, C.c_uint64]),
    ("vsb_capacity", C.c_uint64, [_P]),
    ("vsb_size", C.c_uint64, [_P]),
    ("vsb_add", C.c_int, [_P, _P, _P, C.c_uint64]),
    ("vsb_add_dev", C.c_int, [_P, _P, _P, C.c_uint64]),
    ("vsb_add_each", C.c_int, [_P, _P, _P, C.c_uint64, _P, C.POINTER(C.c_uint64)]),
    ("vsb_remove", C.c_int, [_P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    ("vsb_contains", C.c_int, [_P, C.c_uint64]),
    ("vsb_build", C.c_int, [_P]),
    ("vsb_insert_pending", C.c_int, [_P]),
    ("vsb_export_graph", C.c_int, [_P, _P, _P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    ("vsb_set_search_params", C.c_int, [_P, C.POINTER(VsbSearchParams)]),
    ("vsb_get_stats", C.c_int, [_P, C.POINTER(VsbStats)]),
    ("vsb_get_build_stats", C.c_int, [_P, C.POINTER(VsbBuildStats)]),
    ("vsb_get_options", C.c_int, [_P, C.POINTER(VsbOptions)]),
    ("vsb_set_instrumented", C.c_int, [_P, C.c_int]),
    ("vsb_set_kernel_timing", C.c_int, [_P, C.c_int]),
    ("vsb_search", C.c_int, [_P, _P, C.c_uint64, C.c_uint32, _P, _P, _P]),
    ("vsb_search_exact", C.c_int, [_P, _P, C.c_uint64, C.c_uint32, _P, _P, _P]),
    ("vsb_search_filtered", C.c_int, [_P, _P, C.c_uint64, C.c_uint32, _P, C.c_uint64, _P, _P, _P]),
    ("vsb_search_filtered_multi", C.c_int, [_P, _P, C.c_uint64, C.c_uint32, _P, C.c_uint32, C.c_uint64, _P, _P, _P, _P]),
    ("vsb_search_dev", C.c_int, [_P, _P, C.c_uint64, C.c_uint32, _P, _P, _P, _P, C.c_int]),
    ("vsb_merge_topk_dev", C.c_int, [_P, _P, C.c_uint32, C.c_uint64, C.c_uint32, _P, _P, _P, C.c_int, _P]),
    ("vsb_batcher_create", C.c_int, [_P, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(_P)]),
    ("vsb_batcher_destroy", None, [_P]),
    ("vsb_batcher_search", C.c_int, [_P, _P, C.c_uint32, _P, _P, _P]),
    ("vsb_batcher_stats", C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ("vsb_batcher_add", C.c_int, [_P, C.c_uint64, _P]),
    ("vsb_batcher_flush", C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ("vsb_set_create", C.c_int, [C.POINTER(VsbOptions), C.c_uint32, C.POINTER(_P)]),
    ("vsb_set_destroy", None, [_P]),
    ("vsb_set_add", C.c_int, [_P, C.c_uint64, _P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    ("vsb_set_remove", C.c_int, [_P, C.c_uint64, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    ("vsb_set_remove_partition", C.c_int, [_P, C.c_uint64]),
    ("vsb_set_search", C.c_int, [_P, C.c_uint64, _P, C.c_uint64, C.c_uint32, _P, C.c_uint64, _P, _P, _P]),
    ("vsb_set_count", C.c_uint64, [_P, C.c_uint16]),
    ("vsb_set_partitions", C.c_uint64, [_P]),
    ("vsb_set_index", _P, [_P, C.c_uint64]),
    ("vsb_xchg_create", C.c_int, [C.c_int32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint64, C.POINTER(_P)]),
    ("vsb_xchg_allgather_bytes", C.c_int, [_P, _P, C.c_uint64, C.POINTER(_P), _P, _P]),
    ("vsb_xchg_destroy", None, [_P]),
    ("vsb_xchg_local_handle", C.c_int, [_P, _P]),
    ("vsb_xchg_open", C.c_int, [_P, _P]),
    ("vsb_xchg_allgather_merge", C.c_int, [_P, _P, _P, C.c_uint64, C.c_uint32, _P, _P, _P, _P]),
    ("vsb_xchg_check", C.c_int, [_P, _P]),
    ("vsb_save", C.c_int, [_P, C.c_char_p]),
    ("vsb_load", C.c_int, [C.c_char_p, C.c_int32, C.POINTER(_P)]),
    ("vsb_merge_topk_strided_dev", C.c_int, [_P, _P, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, _P, _P,
                                             _P, C.c_int, _P]),
    ("vsb_f32_to_b1x8", None, [_P, C.c_uint64, _P]),
    ("vsb_last_error", C.c_char_p, []),
    ("vsb_version", C.c_char_p, []),
]

_lib = None


def lib_path() -> str:
    return _LIB_PATH


def lib() -> C.CDLL:
    """Loads libvsb200.so.  There is no fallback: a missing library is a hard error."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise ImportError(f"{_LIB_PATH} is missing — run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a).  vsb200 has no CPU or PyTorch fallback.")
        l = C.CDLL(_LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(l, name)  # AttributeError = ABI drift between header and library
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status: int) -> None:
    if status != VSB_OK:
        msg = lib().vsb_last_error()
        raise VsbError(status, msg.decode() if msg else "")


def version() -> str:
    return lib().vsb_version().decode()
