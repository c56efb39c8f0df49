"""ctypes binding of the C-ABI library (include/semadb_b200.h).

This is the same boundary a Go shard binds through cgo (INTEGRATION.md). There is no
CPU fallback: if the CUDA library is missing the import fails loudly, and without a
CUDA device every compute call raises SdbError.
"""
from __future__ import annotations

import ctypes as C
import re
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "libsemadb_b200.so"
HEADER_PATH = _HERE.parent / "include" / "semadb_b200.h"

OK, ERR_INVALID, ERR_CUDA, ERR_OOM, ERR_STATE, ERR_SEARCHSIZE, ERR_RESERVED_ID, ERR_NOTFOUND, ERR_INTERNAL = range(9)

METRICS = {"euclidean": 0, "dot": 1, "cosine": 2, "hamming": 3, "jaccard": 4, "haversine": 5}
QUANTIZERS = {"none": 0, "binary": 1, "product": 2}


class SdbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[sdb error {code}] {msg}")
        self.code = code
        self.msg = msg


class SdbParams(C.Structure):
    _fields_ = [
        ("dim", C.c_uint32), ("metric", C.c_int32), ("search_size", C.c_uint32), ("degree_bound", C.c_uint32),
        ("alpha", C.c_float), ("quantizer", C.c_int32), ("bq_threshold", C.c_float), ("bq_metric", C.c_int32),
        ("bq_trigger", C.c_uint32), ("pq_subvectors", C.c_uint32), ("pq_centroids", C.c_uint32),
        ("pq_trigger", C.c_uint32), ("device", C.c_int32), ("relaxed", C.c_int32),
    ]


MAX_PEERS = 16


class SdbPeerGather(C.Structure):
    """sdb_peer_gather (include/semadb_b200.h): peer-mapped gather buffers of every GPU."""
    _fields_ = [
        ("n_peers", C.c_uint32), ("shard", C.c_uint32), ("per_shard_limit", C.c_uint32), ("reserved", C.c_uint32),
        ("ids", C.c_void_p * MAX_PEERS), ("dists", C.c_void_p * MAX_PEERS), ("counts", C.c_void_p * MAX_PEERS),
    ]


class SdbRequest(C.Structure):
    """sdb_request (include/semadb_b200.h): one request's limit, searchSize, shard limit and filter."""
    _fields_ = [("limit", C.c_uint32), ("search_size", C.c_uint32), ("shard_limit", C.c_uint32), ("filter", C.c_int32)]


f32p = C.POINTER(C.c_float)
u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)
u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
H = C.c_void_p

_SIGS = {
    "sdb_last_error": (C.c_char_p, []),
    "sdb_abi_version": (C.c_int, []),
    "sdb_device_count": (C.c_int, []),
    "sdb_index_create": (C.c_int, [C.POINTER(SdbParams), C.POINTER(H)]),
    "sdb_index_destroy": (None, [H]),
    "sdb_index_size_bytes": (C.c_int64, [H]),
    "sdb_index_reserve": (C.c_int, [H, C.c_uint64]),
    "sdb_index_max_node_id": (C.c_uint64, [H]),
    "sdb_index_count": (C.c_uint64, [H]),
    "sdb_index_set_start": (C.c_int, [H, f32p]),
    "sdb_index_set_vectors": (C.c_int, [H, C.c_uint64, u64p, f32p]),
    "sdb_index_set_edges": (C.c_int, [H, C.c_uint64, u64p, u32p, u64p]),
    "sdb_index_get_edges": (C.c_int, [H, C.c_uint64, u64p, u32p, u64p]),
    "sdb_index_get_vectors": (C.c_int, [H, C.c_uint64, u64p, f32p]),
    "sdb_index_delete": (C.c_int, [H, C.c_uint64, u64p]),
    "sdb_search_batch": (C.c_int, [H, C.c_uint32, f32p, C.c_uint32, C.c_uint32, u64p, C.c_uint64, u64p, f32p, u32p]),
    "sdb_search_batch_filters": (C.c_int, [H, C.c_uint32, f32p, C.c_uint32, C.c_uint32, C.c_uint32, u64p, u64p, i32p, u64p, f32p,
                                           u32p]),
    "sdb_search_batch_device": (C.c_int, [H, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "sdb_search_batch_gather_device": (C.c_int, [H, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.POINTER(SdbPeerGather), C.c_void_p]),
    "sdb_search_batch_filters_device": (C.c_int, [H, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, u64p, u64p,
                                                  i32p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SdbPeerGather),
                                                  C.c_void_p]),
    "sdb_search_batch_requests": (C.c_int, [H, C.c_uint32, f32p, C.POINTER(SdbRequest), C.c_uint32, u64p, u64p,
                                            C.c_uint32, u64p, f32p, u32p]),
    "sdb_search_batch_requests_device": (C.c_int, [H, C.c_uint32, C.c_void_p, C.POINTER(SdbRequest), C.c_uint32, u64p,
                                                   u64p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.POINTER(SdbPeerGather), C.c_void_p]),
    "sdb_flat_search_batch_requests": (C.c_int, [H, C.c_uint32, f32p, C.POINTER(SdbRequest), C.c_uint32, u64p, u64p,
                                                 C.c_uint32, u64p, f32p, u32p]),
    "sdb_flat_search_batch_requests_device": (C.c_int, [H, C.c_uint32, C.c_void_p, C.POINTER(SdbRequest), C.c_uint32,
                                                        u64p, u64p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                        C.POINTER(SdbPeerGather), C.c_void_p]),
    "sdb_merge_topk_requests_device": (C.c_int, [C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p]),
    "sdb_peer_barrier_device": (C.c_int, [C.c_int32, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p), C.c_uint32,
                                          C.c_void_p]),
    "sdb_peer_barrier_check": (C.c_int, [C.c_int32, C.c_int32]),
    "sdb_last_search_stats": (C.c_int, [H, C.c_uint32, u32p, u32p]),
    "sdb_search_profile": (C.c_int, [H, C.c_int32]),
    "sdb_search_profile_read": (C.c_int, [H, C.c_uint32, f32p, u32p]),
    "sdb_launch_count": (C.c_uint64, [H]),
    "sdb_search_visited": (C.c_int, [H, C.c_uint32, f32p, C.c_uint32, C.c_uint32, u64p, f32p, u32p]),
    "sdb_flat_search_batch": (C.c_int, [H, C.c_uint32, f32p, C.c_uint32, u64p, C.c_uint64, u64p, f32p, u32p]),
    "sdb_flat_search_batch_device": (C.c_int, [H, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p]),
    "sdb_flat_search_batch_gather_device": (C.c_int, [H, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                                      C.c_void_p, C.POINTER(SdbPeerGather), C.c_void_p]),
    "sdb_flat_search_batch_filters_device": (C.c_int, [H, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, u64p, u64p, i32p,
                                                       C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SdbPeerGather),
                                                       C.c_void_p]),
    "sdb_flat_last_stats": (C.c_int, [H, i32p, u64p, u32p]),
    "sdb_flat_search_batch_filters": (C.c_int, [H, C.c_uint32, f32p, C.c_uint32, C.c_uint32, u64p, u64p, i32p, u64p, f32p,
                                                u32p]),
    "sdb_flat_last_filter_stats": (C.c_int, [H, u32p, u32p, u64p]),
    "sdb_filter_staging_bytes": (C.c_int, [H, u64p, u64p]),
    "sdb_insert_batch": (C.c_int, [H, C.c_uint64, u64p, f32p]),
    "sdb_insert_batch_device": (C.c_int, [H, C.c_uint64, u64p, C.c_void_p]),
    "sdb_insert_truncated": (C.c_uint64, [H]),
    "sdb_insert_stats": (C.c_int, [H, u64p, C.c_int32]),
    "sdb_insert_config": (C.c_int, [H, C.c_uint32, C.c_uint32, C.c_uint32]),
    "sdb_insert_update_delete": (C.c_int, [H, C.c_uint64, u64p, f32p, u8p]),
    "sdb_edge_scan": (C.c_int, [H, C.c_uint64, u64p, u64p, u64p, u64p, u64p]),
    "sdb_index_get_start_overflow": (C.c_int, [H, C.c_uint64, u64p, u64p]),
    "sdb_index_set_start_overflow": (C.c_int, [H, C.c_uint64, u64p]),
    "sdb_index_fit": (C.c_int, [H, C.c_uint64, i32p]),
    "sdb_index_get_pq": (C.c_int, [H, f32p, f32p]),
    "sdb_index_set_pq": (C.c_int, [H, f32p, f32p]),
    "sdb_index_get_bq_threshold": (C.c_int, [H, f32p]),
    "sdb_index_set_bq_threshold": (C.c_int, [H, f32p]),
    "sdb_index_get_codes": (C.c_int, [H, C.c_uint64, u64p, u8p]),
    "sdb_index_set_codes": (C.c_int, [H, C.c_uint64, u64p, u8p]),
    "sdb_index_dirty_edges": (C.c_int, [H, C.c_uint64, u64p, u64p, C.c_int32]),
    "sdb_distance_float": (C.c_int, [C.c_int32, C.c_int32, C.c_uint64, C.c_uint32, f32p, f32p, f32p]),
    "sdb_distance_bits": (C.c_int, [C.c_int32, C.c_int32, C.c_uint64, C.c_uint32, u64p, u64p, f32p]),
    "sdb_index_query_dists": (C.c_int, [H, f32p, C.c_uint64, u64p, f32p]),
    "sdb_index_point_dists": (C.c_int, [H, C.c_uint64, C.c_uint64, u64p, f32p]),
    "sdb_bq_encode": (C.c_int, [C.c_int32, C.c_uint64, C.c_uint32, f32p, f32p, u64p]),
    "sdb_pq_adc_tables": (C.c_int, [H, C.c_uint32, f32p, f32p]),
    "sdb_merge_topk": (C.c_int, [C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, u64p, f32p, u32p, u64p, f32p, u32p]),
    "sdb_merge_topk_device": (C.c_int, [C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sdb_hybrid_merge": (C.c_int, [C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, u64p, f32p, f32p, u32p, u64p,
                                   f32p, f32p, u32p]),
    "sdb_shard_limit": (C.c_uint32, [C.c_uint32, C.c_uint32, C.c_uint32]),
}

_lib = None


def declared_symbols() -> list[str]:
    """Every function include/semadb_b200.h declares (used by the export test)."""
    text = HEADER_PATH.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sdb_[a-z0-9_]+)\s*\(", text)))


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). semadb_b200 has no CPU fallback.")
    L = C.CDLL(str(LIB_PATH))
    for name, (res, args) in _SIGS.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != OK:
        msg = lib().sdb_last_error()
        raise SdbError(rc, msg.decode() if msg else "unknown error")
