"""ctypes binding of libzebra_b200.so (the C ABI declared in include/zebra_b200.h).

There is no CPU fallback: if the shared library is missing, or a call fails, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libzebra_b200.so")

ZB_OK = 0
METRIC_COSINE, METRIC_L2SQ, METRIC_L2 = 0, 1, 2
(METRIC_CHEBYSHEV, METRIC_CANBERRA, METRIC_BRAY_CURTIS, METRIC_MANHATTAN, METRIC_L3, METRIC_L4, METRIC_HAMMING,
 METRIC_MINKOWSKI, METRIC_PNORM) = range(3, 12)
METRIC_MAX_POWER = 64


class ZebraError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"zebra_b200 error {code}: {msg}")
        self.code = code


class Options(C.Structure):
    _fields_ = [
        ("dim", C.c_uint32),
        ("metric", C.c_uint32),
        ("max_node_size", C.c_uint64),
        ("num_trees", C.c_uint32),
        ("device", C.c_int32),
        ("seed", C.c_uint64),
        ("shard_rank", C.c_uint32),
        ("shard_count", C.c_uint32),
        ("metric_power", C.c_int32),
        ("reserved", C.c_uint32 * 3),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("rows", C.c_uint64),
        ("live_rows", C.c_uint64),
        ("total_rows", C.c_uint64),
        ("nodes", C.c_uint64),
        ("planes", C.c_uint64),
        ("leaves", C.c_uint64),
        ("device_bytes", C.c_uint64),
        ("last_queries", C.c_uint64),
        ("last_visits", C.c_uint64),
        ("last_pairs", C.c_uint64),
        ("last_tile_visits", C.c_uint64),
        ("last_tile_pairs", C.c_uint64),
        ("last_moved_bytes", C.c_uint64),
        ("last_ms_plan", C.c_float),
        ("last_ms_scan", C.c_float),
        ("last_ms_select", C.c_float),
        ("last_ms_merge", C.c_float),
        ("last_ms_total", C.c_float),
        ("last_scan_launches", C.c_uint32),
        ("last_total_launches", C.c_uint32),
        ("last_ms_tile_kernel", C.c_float),
        ("last_tiles", C.c_uint32),
        ("last_filter_flagged", C.c_uint32),
        ("last_unique_bytes", C.c_uint64),
        ("last_filter_rows", C.c_uint32),
        ("last_ms_refine", C.c_float),
        ("last_filter_used", C.c_uint32),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if not n.startswith("reserved")}


class ImportReport(C.Structure):
    _fields_ = [
        ("rows_loaded", C.c_uint64),
        ("missing_ids", C.c_uint64),
        ("orphan_rows", C.c_uint64),
        ("nodes", C.c_uint64),
        ("planes", C.c_uint64),
        ("leaves", C.c_uint64),
        ("max_depth", C.c_uint32),
        ("reserved", C.c_uint32 * 3),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if not n.startswith("reserved")}


# every symbol include/zebra_b200.h declares: name -> (restype, argtypes)
_vp, _u64, _u32, _i32, _i64 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_int64
SYMBOLS = {
    "zb_last_error": (C.c_char_p, []),
    "zb_abi_version": (C.c_int, []),
    "zb_device_count": (C.c_int, [_vp]),
    "zb_index_create": (C.c_int, [C.POINTER(Options), C.POINTER(_vp)]),
    "zb_index_destroy": (C.c_int, [_vp]),
    "zb_index_options": (C.c_int, [_vp, C.POINTER(Options)]),
    "zb_index_add": (C.c_int, [_vp, _u64, _vp, _vp, _vp, _vp]),
    "zb_index_add_device": (C.c_int, [_vp, _u64, _vp, _vp, _vp, _vp]),
    "zb_index_add_owned_device": (C.c_int, [_vp, _u64, _vp, _vp, _u64]),
    "zb_index_remove": (C.c_int, [_vp, _u64, _vp, _vp]),
    "zb_index_remove_ordinals": (C.c_int, [_vp, _u64, _vp, _vp]),
    "zb_index_deduplicate": (C.c_int, [_vp, C.POINTER(_u64), _vp, _vp, _u64]),
    "zb_index_clear": (C.c_int, [_vp]),
    "zb_index_no_vectors": (C.c_int, [_vp, _vp]),
    "zb_index_no_trees": (C.c_int, [_vp, _vp]),
    "zb_index_search_batch": (C.c_int, [_vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp]),
    "zb_index_search_batch_device": (C.c_int, [_vp, _u64, _vp, _u64, _vp, _vp, _vp]),
    "zb_index_search_slice": (C.c_int, [_vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp]),
    "zb_index_search_slice_device": (C.c_int, [_vp, _u64, _vp, _u64, _vp, _vp, _vp]),
    "zb_index_search_prefetch": (C.c_int, [_vp, _u64, _vp]),
    "zb_index_search_exact": (C.c_int, [_vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp]),
    "zb_index_search_exact_device": (C.c_int, [_vp, _u64, _vp, _u64, _vp, _vp, _vp]),
    "zb_index_search_probe": (C.c_int, [_vp, _u64, _vp, _u64, C.c_uint32, _vp, _vp, _vp, _vp]),
    "zb_index_search_probe_device": (C.c_int, [_vp, _u64, _vp, _u64, C.c_uint32, _vp, _vp, _vp]),
    "zb_index_search_slice_probe": (C.c_int, [_vp, _u64, _vp, _u64, C.c_uint32, _vp, _vp, _vp, _vp]),
    "zb_index_search_slice_probe_device": (C.c_int, [_vp, _u64, _vp, _u64, C.c_uint32, _vp, _vp, _vp]),
    "zb_index_hash": (C.c_int, [_vp, _u64, _vp, _vp, _vp, _vp]),
    "zb_index_hash_device": (C.c_int, [_vp, _u64, _vp, _vp, _vp, _vp]),
    "zb_index_forest_sizes": (C.c_int, [_vp, _vp]),
    "zb_index_export_forest": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "zb_index_load_forest": (C.c_int, [_vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "zb_tree_blob_decode": (C.c_int, [_u32, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "zb_tree_blob_encode": (C.c_int, [_u32, _i64, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _u64, C.POINTER(_u64)]),
    "zb_zebra_file_encode": (C.c_int, [_vp, _u32, _i32, _u64, _u64, _vp, _u64, C.POINTER(_u64)]),
    "zb_zebra_file_decode": (C.c_int, [_vp, _u64, _u32, _vp, C.POINTER(_i32), C.POINTER(_u64), C.POINTER(_u64)]),
    "zb_store_flatten": (C.c_int, [_u32, _u64, _vp, _u32, _vp, _vp, C.POINTER(_vp), C.POINTER(ImportReport)]),
    "zb_flat_store_view": (C.c_int, [_vp] + [_vp] * 9),
    "zb_flat_store_free": (C.c_int, [_vp]),
    "zb_index_import_store": (C.c_int, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, C.POINTER(ImportReport), _vp, _u64]),
    "zb_index_export_rows": (C.c_int, [_vp, _u64, _u64, _vp, _vp, _vp]),
    "zb_index_export_tree_blob": (C.c_int, [_vp, _u32, _vp, _u64, C.POINTER(_u64)]),
    "zb_index_export_tree_blobs": (C.c_int, [_vp, _vp, _u64, _vp, C.POINTER(_u64)]),
    "zb_index_load_flat": (C.c_int, [_vp, _u64, _vp, _vp, _u32, _vp, _vp]),
    "zb_index_stats": (C.c_int, [_vp, C.POINTER(Stats)]),
    "zb_index_stream": (C.c_int, [_vp, C.POINTER(_vp)]),
    "zb_index_set_param": (C.c_int, [_vp, C.c_char_p, _i64]),
    "zb_comm_unique_id": (C.c_int, [_vp]),
    "zb_index_comm_init": (C.c_int, [_vp, _vp]),
    "zb_metric_distance_batch": (C.c_int, [C.c_int, _u32, _i32, _u64, _u32, _vp, _vp, _vp]),
    "zb_point_is_above_batch": (C.c_int, [C.c_int, _u64, _u32, _vp, _vp, _vp, _vp]),
    "zb_synth_fill_device": (C.c_int, [C.c_int, _vp, _u64, _u64, _u64, _u32, _u64, _u32]),
}

_lib = None


def lib():
    """Load libzebra_b200.so.  Raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C zebra_b200` (or __graft_entry__.build()); "
                "zebra_b200 has no CPU fallback"
            )
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != ZB_OK:
        msg = lib().zb_last_error()
        raise ZebraError(rc, msg.decode("utf-8", "replace") if msg else "?")
