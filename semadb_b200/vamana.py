"""Host-side mirror of the reference's index surfaces for the hot path, over the C ABI.

Mirrors (same names, argument meaning, error behaviour):
  * models.IndexVectorVamanaParameters / Quantizer (models/index.go:275-282,
    models/quantizer.go:5-76)
  * vamana.IndexVamana: NewIndexVamana, SizeInMemory, InsertUpdateDelete, Search
    (shard/index/vamana/vamana.go:54,83,127,278)
  * flat.IndexFlat.Search (shard/index/flat/flat.go:76)
plus the batched entry points the reference lacks (SearchBatch): one C call per batch,
never per distance (SURVEY.md §7.3-⑨).

The reference host language is Go; no Go toolchain exists in this image, so this mirror
is what the parity tests drive. The C++ twin is semadb_b200/host/gpuvamana.hpp and the
cgo stub a maintainer would add is in INTEGRATION.md.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Iterable, Optional, Sequence

import numpy as np

from . import _capi
from ._capi import SdbError, SdbParams, check, f32p, u32p, u64p, u8p

STARTID = 1  # vamana.go:28


@dataclass
class BinaryQuantizerParameters:  # models/quantizer.go:30-39
    threshold: Optional[float] = None
    trigger_threshold: int = 0
    distance_metric: str = "hamming"


@dataclass
class ProductQuantizerParameters:  # models/quantizer.go:52-63
    num_centroids: int = 256
    num_sub_vectors: int = 8
    trigger_threshold: int = 10000


@dataclass
class Quantizer:  # models/quantizer.go:5-9
    type: str = "none"
    binary: Optional[BinaryQuantizerParameters] = None
    product: Optional[ProductQuantizerParameters] = None


@dataclass
class IndexVectorVamanaParameters:  # models/index.go:275-282
    vector_size: int
    distance_metric: str = "euclidean"
    search_size: int = 75
    degree_bound: int = 64
    alpha: float = 1.2
    quantizer: Optional[Quantizer] = None


@dataclass
class IndexVectorFlatParameters:  # models/index.go:255-259
    vector_size: int
    distance_metric: str = "euclidean"
    quantizer: Optional[Quantizer] = None


@dataclass
class SearchVectorVamanaOptions:  # models/search.go:268-275
    vector: Sequence[float]
    search_size: int = 75
    limit: int = 10
    weight: Optional[float] = None


@dataclass
class SearchVectorFlatOptions:  # models/search.go:308-314
    vector: Sequence[float]
    limit: int = 10
    weight: Optional[float] = None


@dataclass
class SearchResult:  # models/search.go:238-252
    node_id: int
    distance: float
    hybrid_score: float


@dataclass
class IndexVectorChange:  # vamana.go:122-125 (vector None = delete)
    id: int
    vector: Optional[Sequence[float]] = None


def _params_struct(p, device: int, relaxed: bool, search_size=75, degree_bound=64, alpha=1.2) -> SdbParams:
    if p.distance_metric not in _capi.METRICS:
        raise SdbError(_capi.ERR_INVALID, f"unknown distance metric {p.distance_metric}")
    s = SdbParams()
    s.dim = int(p.vector_size)
    s.metric = _capi.METRICS[p.distance_metric]
    s.search_size = int(getattr(p, "search_size", search_size))
    s.degree_bound = int(getattr(p, "degree_bound", degree_bound))
    s.alpha = float(getattr(p, "alpha", alpha))
    s.quantizer = 0
    s.bq_threshold = float("nan")
    s.bq_metric = _capi.METRICS["hamming"]
    q = p.quantizer
    if q is not None and q.type != "none":
        if q.type not in _capi.QUANTIZERS:
            raise SdbError(_capi.ERR_INVALID, f"unknown quantizer type {q.type}")
        s.quantizer = _capi.QUANTIZERS[q.type]
        if q.type == "binary":
            if q.binary is None:
                raise SdbError(_capi.ERR_INVALID, "binary quantizer parameters are nil")  # vectorstore.go:83
            if q.binary.distance_metric not in ("hamming", "jaccard"):
                raise SdbError(_capi.ERR_INVALID, "invalid distance metric for binary quantization")
            s.bq_threshold = float("nan") if q.binary.threshold is None else float(q.binary.threshold)
            s.bq_metric = _capi.METRICS[q.binary.distance_metric]
            s.bq_trigger = int(q.binary.trigger_threshold)
        if q.type == "product":
            if q.product is None:
                raise SdbError(_capi.ERR_INVALID, "product quantizer parameters are nil")  # vectorstore.go:88
            s.pq_subvectors = int(q.product.num_sub_vectors)
            s.pq_centroids = int(q.product.num_centroids)
            s.pq_trigger = int(q.product.trigger_threshold)
    s.device = int(device)
    s.relaxed = int(relaxed)
    return s


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64)


def _ptr(a, t):
    return None if a is None else a.ctypes.data_as(t)


class _DeviceIndex:
    """Owns an sdb_index handle; shared by IndexVamana and IndexFlat."""

    def __init__(self, params_struct: SdbParams):
        self._lib = _capi.lib()
        self._h = _capi.H()
        self.dim = int(params_struct.dim)
        self.R = int(params_struct.degree_bound)
        self.L = int(params_struct.search_size)
        self._ps = params_struct
        check(self._lib.sdb_index_create(C.byref(params_struct), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.sdb_index_destroy(self._h)
            self._h = _capi.H()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- cache.Cachable / bookkeeping
    def size_in_memory(self) -> int:
        return int(self._lib.sdb_index_size_bytes(self._h))

    @property
    def max_node_id(self) -> int:
        return int(self._lib.sdb_index_max_node_id(self._h))

    @property
    def count(self) -> int:
        return int(self._lib.sdb_index_count(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._lib.sdb_launch_count(self._h))

    def reserve(self, max_node_id: int):
        check(self._lib.sdb_index_reserve(self._h, int(max_node_id)))

    # ---- hydrate / flush
    def set_start(self, vec):
        v = _f32(vec)
        if v.shape != (self.dim,):
            raise SdbError(_capi.ERR_INVALID, "start vector has the wrong length")
        check(self._lib.sdb_index_set_start(self._h, _ptr(v, f32p)))

    def set_vectors(self, ids, vectors):
        ids, v = _u64(ids), _f32(vectors)
        if v.shape != (len(ids), self.dim):
            raise SdbError(_capi.ERR_INVALID, "vectors must be [n, dim]")
        check(self._lib.sdb_index_set_vectors(self._h, len(ids), _ptr(ids, u64p), _ptr(v, f32p)))

    def get_vectors(self, ids) -> np.ndarray:
        ids = _u64(ids)
        out = np.zeros((len(ids), self.dim), dtype=np.float32)
        check(self._lib.sdb_index_get_vectors(self._h, len(ids), _ptr(ids, u64p), _ptr(out, f32p)))
        return out

    def set_edges(self, ids, degrees, edges_flat):
        ids = _u64(ids)
        deg = np.ascontiguousarray(degrees, dtype=np.uint32)
        e = _u64(edges_flat)
        if len(deg) != len(ids) or int(deg.sum()) != len(e):
            raise SdbError(_capi.ERR_INVALID, "edge lists do not match degrees")
        check(self._lib.sdb_index_set_edges(self._h, len(ids), _ptr(ids, u64p), _ptr(deg, u32p), _ptr(e, u64p)))

    def set_graph_dense(self, adj: np.ndarray, deg: np.ndarray, first_id: int = 1):
        """adj: [n, R] rows for node ids first_id.. (padding ignored), deg: [n]."""
        n = adj.shape[0]
        ids = np.arange(first_id, first_id + n, dtype=np.uint64)
        deg = np.ascontiguousarray(deg, dtype=np.uint32)
        mask = np.arange(adj.shape[1])[None, :] < deg[:, None]
        self.set_edges(ids, deg, adj[mask].astype(np.uint64))

    def get_edges(self, ids):
        ids = _u64(ids)
        deg = np.zeros(len(ids), dtype=np.uint32)
        e = np.zeros((len(ids), self.R), dtype=np.uint64)
        check(self._lib.sdb_index_get_edges(self._h, len(ids), _ptr(ids, u64p), _ptr(deg, u32p), _ptr(e, u64p)))
        return deg, e

    def delete_rows(self, ids):
        ids = _u64(ids)
        check(self._lib.sdb_index_delete(self._h, len(ids), _ptr(ids, u64p)))

    # ---- quantizers
    def fit(self, pq_first_row: int = 0) -> bool:
        f = C.c_int32(0)
        check(self._lib.sdb_index_fit(self._h, int(pq_first_row), C.byref(f)))
        return bool(f.value)

    def get_pq(self):
        M, K = int(self._ps.pq_subvectors), int(self._ps.pq_centroids)
        fc = np.zeros((M, K, self.dim // M), dtype=np.float32)
        cd = np.zeros((M, K, K), dtype=np.float32)
        check(self._lib.sdb_index_get_pq(self._h, _ptr(fc, f32p), _ptr(cd, f32p)))
        return fc, cd

    def set_pq(self, flat_centroids, centroid_dists):
        fc, cd = _f32(flat_centroids), _f32(centroid_dists)
        check(self._lib.sdb_index_set_pq(self._h, _ptr(fc, f32p), _ptr(cd, f32p)))

    def get_bq_threshold(self) -> np.ndarray:
        t = np.zeros(self.dim, dtype=np.float32)
        check(self._lib.sdb_index_get_bq_threshold(self._h, _ptr(t, f32p)))
        return t

    def set_bq_threshold(self, thr):
        t = _f32(thr)
        check(self._lib.sdb_index_set_bq_threshold(self._h, _ptr(t, f32p)))

    def get_codes(self, ids) -> np.ndarray:
        ids = _u64(ids)
        width = int(self._ps.pq_subvectors) if self._ps.quantizer == 2 else 8 * ((self.dim + 63) // 64)
        out = np.zeros((len(ids), width), dtype=np.uint8)
        check(self._lib.sdb_index_get_codes(self._h, len(ids), _ptr(ids, u64p), _ptr(out, u8p)))
        return out

    def adc_tables(self, queries) -> np.ndarray:
        q = _f32(queries).reshape(-1, self.dim)
        M, K = int(self._ps.pq_subvectors), int(self._ps.pq_centroids)
        out = np.zeros((q.shape[0], M, K), dtype=np.float32)
        check(self._lib.sdb_pq_adc_tables(self._h, q.shape[0], _ptr(q, f32p), _ptr(out, f32p)))
        return out

    # ---- store-level distance closures, batched
    def query_dists(self, query, ids) -> np.ndarray:
        q, ids = _f32(query), _u64(ids)
        out = np.zeros(len(ids), dtype=np.float32)
        check(self._lib.sdb_index_query_dists(self._h, _ptr(q, f32p), len(ids), _ptr(ids, u64p), _ptr(out, f32p)))
        return out

    def point_dists(self, x: int, ids) -> np.ndarray:
        ids = _u64(ids)
        out = np.zeros(len(ids), dtype=np.float32)
        check(self._lib.sdb_index_point_dists(self._h, int(x), len(ids), _ptr(ids, u64p), _ptr(out, f32p)))
        return out

    # ---- batched search entry points
    def search_batch(self, queries, k: int = 10, search_size: Optional[int] = None, filter_ids=None):
        q = _f32(queries)
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise SdbError(_capi.ERR_INVALID, "queries must be [B, dim]")
        B = q.shape[0]
        L = self.L if search_size is None else int(search_size)
        ids = np.zeros((B, k), dtype=np.uint64)
        d = np.zeros((B, k), dtype=np.float32)
        cnt = np.zeros(B, dtype=np.uint32)
        filt = None if filter_ids is None else np.unique(_u64(filter_ids))
        check(self._lib.sdb_search_batch(self._h, B, _ptr(q, f32p), k, L, _ptr(filt, u64p),
                                         0 if filt is None else len(filt), _ptr(ids, u64p), _ptr(d, f32p),
                                         _ptr(cnt, u32p)))
        return ids, d, cnt

    def search_batch_filters(self, queries, filters, query_filter=None, k: int = 10, search_size: Optional[int] = None):
        """One filter per request (shard/index/search.go:59-85): `filters` is a list of id
        collections (an empty one filters everything out), query_filter[b] the filter index of
        request b or -1 for none (None: every request uses filters[0])."""
        q = _f32(queries)
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise SdbError(_capi.ERR_INVALID, "queries must be [B, dim]")
        B = q.shape[0]
        L = self.L if search_size is None else int(search_size)
        lists = [np.unique(_u64(f)) for f in filters]
        off = np.zeros(len(lists) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(x) for x in lists])
        flat = np.concatenate(lists) if lists and off[-1] else np.zeros(0, dtype=np.uint64)
        qf = None if query_filter is None else np.ascontiguousarray(query_filter, dtype=np.int32)
        ids = np.zeros((B, k), dtype=np.uint64)
        d = np.zeros((B, k), dtype=np.float32)
        cnt = np.zeros(B, dtype=np.uint32)
        check(self._lib.sdb_search_batch_filters(self._h, B, _ptr(q, f32p), k, L, len(lists),
                                                 _ptr(flat, u64p) if len(flat) else None, _ptr(off, u64p),
                                                 None if qf is None else _ptr(qf, _capi.i32p), _ptr(ids, u64p),
                                                 _ptr(d, f32p), _ptr(cnt, u32p)))
        return ids, d, cnt

    def search_batch_device(self, d_queries, k: int, search_size: int, d_out_ids, d_out_dists, d_out_counts,
                            stream: int = 0):
        """torch CUDA tensors (contiguous): queries f32 [B,dim], out ids int64/uint64 [B,k],
        dists f32 [B,k], counts int32/uint32 [B]. Enqueues on `stream` (raw cudaStream_t)."""
        B = int(d_queries.shape[0])
        check(self._lib.sdb_search_batch_device(self._h, B, d_queries.data_ptr(), k, search_size,
                                                d_out_ids.data_ptr(), d_out_dists.data_ptr(),
                                                d_out_counts.data_ptr(), stream))

    def last_search_stats(self, B: int):
        hops = np.zeros(B, dtype=np.uint32)
        nd = np.zeros(B, dtype=np.uint32)
        check(self._lib.sdb_last_search_stats(self._h, B, _ptr(hops, u32p), _ptr(nd, u32p)))
        return hops, nd

    def search_profile(self, enable: bool):
        """CUDA events around the first-pass beam-search kernel of every following search."""
        check(self._lib.sdb_search_profile(self._h, 1 if enable else 0))

    def search_profile_read(self) -> np.ndarray:
        """Kernel durations (ms) of the searches recorded since search_profile(True)."""
        import ctypes as C
        out = np.zeros(256, dtype=np.float32)
        n = C.c_uint32(0)
        check(self._lib.sdb_search_profile_read(self._h, len(out), _ptr(out, f32p), C.byref(n)))
        return out[:min(n.value, len(out))].copy()

    def search_visited(self, queries, search_size: Optional[int] = None, vis_cap: int = 256):
        q = _f32(queries)
        B = q.shape[0]
        L = self.L if search_size is None else int(search_size)
        ids = np.zeros((B, vis_cap), dtype=np.uint64)
        d = np.zeros((B, vis_cap), dtype=np.float32)
        n = np.zeros(B, dtype=np.uint32)
        check(self._lib.sdb_search_visited(self._h, B, _ptr(q, f32p), L, vis_cap, _ptr(ids, u64p), _ptr(d, f32p),
                                           _ptr(n, u32p)))
        return ids, d, n

    def flat_search_batch(self, queries, k: int = 10, filter_ids=None):
        q = _f32(queries)
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise SdbError(_capi.ERR_INVALID, "queries must be [B, dim]")
        B = q.shape[0]
        ids = np.zeros((B, k), dtype=np.uint64)
        d = np.zeros((B, k), dtype=np.float32)
        cnt = np.zeros(B, dtype=np.uint32)
        filt = None if filter_ids is None else np.unique(_u64(filter_ids))
        check(self._lib.sdb_flat_search_batch(self._h, B, _ptr(q, f32p), k, _ptr(filt, u64p),
                                              0 if filt is None else len(filt), _ptr(ids, u64p), _ptr(d, f32p),
                                              _ptr(cnt, u32p)))
        return ids, d, cnt

    def flat_search_batch_device(self, d_queries, k: int, d_out_ids, d_out_dists, d_out_counts, stream: int = 0):
        """Flat twin of search_batch_device: torch tensors (contiguous) queries f32 [B,dim] on the
        device or page-locked, out ids int64/uint64 [B,k], dists f32 [B,k], counts int32/uint32 [B].
        Enqueues on `stream` (raw cudaStream_t) without synchronising; rows equal flat_search_batch."""
        B = int(d_queries.shape[0])
        check(self._lib.sdb_flat_search_batch_device(self._h, B, d_queries.data_ptr(), k, d_out_ids.data_ptr(),
                                                     d_out_dists.data_ptr(), d_out_counts.data_ptr(), stream))

    def flat_search_batch_filters(self, queries, filters, query_filter=None, k: int = 10):
        """Flat search with one filter per request, shaped like search_batch_filters: `filters` is a
        list of id collections (an empty one filters everything out; ids that are not stored never
        match), query_filter[b] the filter index of request b or -1 for none (None: every request
        uses filters[0]). Row b equals flat_search_batch(queries[b:b+1], k, filters[query_filter[b]])."""
        q = _f32(queries)
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise SdbError(_capi.ERR_INVALID, "queries must be [B, dim]")
        B = q.shape[0]
        lists = [np.unique(_u64(f)) for f in filters]
        off = np.zeros(len(lists) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(x) for x in lists])
        flat = np.concatenate(lists) if lists and off[-1] else np.zeros(0, dtype=np.uint64)
        qf = None if query_filter is None else np.ascontiguousarray(query_filter, dtype=np.int32)
        ids = np.zeros((B, k), dtype=np.uint64)
        d = np.zeros((B, k), dtype=np.float32)
        cnt = np.zeros(B, dtype=np.uint32)
        check(self._lib.sdb_flat_search_batch_filters(self._h, B, _ptr(q, f32p), k, len(lists),
                                                      _ptr(flat, u64p) if len(flat) else None, _ptr(off, u64p),
                                                      None if qf is None else _ptr(qf, _capi.i32p), _ptr(ids, u64p),
                                                      _ptr(d, f32p), _ptr(cnt, u32p)))
        return ids, d, cnt

    def flat_last_filter_stats(self):
        """(gathered_filters, scanned_filters, gathered_pairs) of the last flat search: filters that
        took the gather route and the range-scan route, and the (request, id) pairs gathered."""
        import ctypes as C
        g, s, p = C.c_uint32(0), C.c_uint32(0), C.c_uint64(0)
        check(self._lib.sdb_flat_last_filter_stats(self._h, C.byref(g), C.byref(s), C.byref(p)))
        return g.value, s.value, p.value

    def flat_last_stats(self):
        """(path, candidates, overflowed) of the last flat search: path 0 = exact CUDA-core
        scan, 1 = mma.sync candidate pass, 2 = tcgen05 + TMA candidate pass. After a device-entry
        call, waits for that call to complete."""
        import ctypes as C
        path, cand, ovf = C.c_int32(0), C.c_uint64(0), C.c_uint32(0)
        check(self._lib.sdb_flat_last_stats(self._h, C.byref(path), C.byref(cand), C.byref(ovf)))
        return path.value, cand.value, ovf.value

    def insert_batch(self, ids, vectors):
        ids, v = _u64(ids), _f32(vectors)
        if v.shape != (len(ids), self.dim):
            raise SdbError(_capi.ERR_INVALID, "vectors must be [n, dim]")
        check(self._lib.sdb_insert_batch(self._h, len(ids), _ptr(ids, u64p), _ptr(v, f32p)))

    def insert_batch_device(self, ids, d_vectors):
        """d_vectors: contiguous f32 CUDA tensor [n, dim] on this index's device."""
        ids = _u64(ids)
        assert d_vectors.is_cuda and d_vectors.is_contiguous() and tuple(d_vectors.shape) == (len(ids), self.dim)
        check(self._lib.sdb_insert_batch_device(self._h, len(ids), _ptr(ids, u64p), d_vectors.data_ptr()))

    def insert_stats(self, reset: bool = False) -> dict:
        """Totals of the batched insert (sdb_insert_stats)."""
        out = np.zeros(8, dtype=np.uint64)
        check(self._lib.sdb_insert_stats(self._h, _ptr(out, u64p), 1 if reset else 0))
        keys = ("points", "hops", "ndist", "edges", "targets", "prunes", "prune_candidates")
        return {k: int(v) for k, v in zip(keys, out)}

    def insert_update_delete_batch(self, ids, vectors, has_vector=None):
        """sdb_insert_update_delete: the whole classify / insert / removeInboundEdges / drop /
        re-insert sequence of vamana.go:136-253 for n changes (has_vector[i] == 0 = nil vector)."""
        ids, v = _u64(ids), _f32(vectors)
        if v.shape != (len(ids), self.dim):
            raise SdbError(_capi.ERR_INVALID, "vectors must be [n, dim]")
        hv = None if has_vector is None else np.ascontiguousarray(has_vector, dtype=np.uint8)
        check(self._lib.sdb_insert_update_delete(self._h, len(ids), _ptr(ids, u64p), _ptr(v, f32p), _ptr(hv, u8p)))

    def edge_scan(self, delete_ids):
        """EdgeScan (node.go:142-199): (toPrune, toSave), ascending ids."""
        d = _u64(delete_ids)
        cap = self.max_node_id + 2
        tp, ts = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.uint64)
        n1, n2 = C.c_uint64(0), C.c_uint64(0)
        check(self._lib.sdb_edge_scan(self._h, len(d), _ptr(d, u64p), _ptr(tp, u64p), C.byref(n1), _ptr(ts, u64p),
                                      C.byref(n2)))
        return tp[:n1.value].copy(), ts[:n2.value].copy()

    def get_start_overflow(self) -> np.ndarray:
        n = C.c_uint64(0)
        check(self._lib.sdb_index_get_start_overflow(self._h, 0, None, C.byref(n)))
        out = np.zeros(max(1, n.value), dtype=np.uint64)
        check(self._lib.sdb_index_get_start_overflow(self._h, n.value, _ptr(out, u64p), C.byref(n)))
        return out[:n.value]

    def set_start_overflow(self, ids):
        ids = _u64(ids)
        check(self._lib.sdb_index_set_start_overflow(self._h, len(ids), _ptr(ids, u64p)))

    def insert_config(self, min_batch=0, max_batch=0, growth_div=0):
        check(self._lib.sdb_insert_config(self._h, min_batch, max_batch, growth_div))


class IndexVamana(_DeviceIndex):
    """vamana.IndexVamana on the GPU (shard/index/vamana/vamana.go:36-52)."""

    def __init__(self, name: str, params: IndexVectorVamanaParameters, device: int = 0,
                 start_vector=None, start_seed: Optional[int] = None, relaxed: bool = False):
        """NewIndexVamana (vamana.go:54-81). setupStartNode (vamana.go:93-120) draws node 1's
        vector at random in the reference; pass start_vector (hydrate) or start_seed."""
        self.name = name
        self.parameters = params
        super().__init__(_params_struct(params, device, relaxed))
        if start_vector is None:
            from . import synth
            seed = start_seed if start_seed is not None else int(np.random.SeedSequence().entropy % (1 << 31))
            start_vector = synth.start_vector(self.dim, seed)
        self.set_start(start_vector)

    def insert_update_delete(self, changes: Iterable[IndexVectorChange], pq_first_row: int = 0) -> None:
        """InsertUpdateDelete (vamana.go:127-263): classify against the store, insert, remove
        the inbound edges of updated/deleted points, drop deleted rows, re-insert updated
        points, then Fit (vamana.go:258)."""
        ids, vecs, has = [], [], []
        zero = np.zeros(self.dim, dtype=np.float32)
        for ch in changes:
            ids.append(ch.id)
            has.append(0 if ch.vector is None else 1)
            vecs.append(zero if ch.vector is None else np.asarray(ch.vector, dtype=np.float32))
        if ids:
            self.insert_update_delete_batch(np.asarray(ids, dtype=np.uint64), np.stack(vecs), np.asarray(has, np.uint8))
        self.fit(pq_first_row)  # vamana.go:258

    def search(self, options: SearchVectorVamanaOptions, filter_ids=None):
        """Search (vamana.go:278-310): returns (set of node ids, [SearchResult])."""
        q = _f32(options.vector).reshape(1, -1)
        ids, d, cnt = self.search_batch(q, options.limit, options.search_size, filter_ids)
        w = np.float32(1.0 if options.weight is None else options.weight)
        res = [SearchResult(int(ids[0, i]), float(d[0, i]), float(np.float32(-1) * d[0, i] * w))
               for i in range(int(cnt[0]))]
        return {r.node_id for r in res}, res


class IndexFlat(_DeviceIndex):
    """flat.IndexFlat on the GPU (shard/index/flat/flat.go:17-39)."""

    def __init__(self, params: IndexVectorFlatParameters, device: int = 0, relaxed: bool = True):
        super().__init__(_params_struct(params, device, relaxed))

    def insert_update_delete(self, changes: Iterable[IndexVectorChange], pq_first_row: int = 0) -> None:
        """flat.go:41-74: Set for vectors, Delete for nil vectors, then Fit."""
        set_ids, set_vecs, del_ids = [], [], []
        for ch in changes:
            if ch.vector is None:
                del_ids.append(ch.id)
            else:
                set_ids.append(ch.id)
                set_vecs.append(ch.vector)
        if set_ids:
            self.set_vectors(np.asarray(set_ids, dtype=np.uint64), np.asarray(set_vecs, dtype=np.float32))
        if del_ids:
            self.delete_rows(np.asarray(del_ids, dtype=np.uint64))
        self.fit(pq_first_row)

    def search(self, options: SearchVectorFlatOptions, filter_ids=None):
        q = _f32(options.vector).reshape(1, -1)
        ids, d, cnt = self.flat_search_batch(q, options.limit, filter_ids)
        w = np.float32(1.0 if options.weight is None else options.weight)
        res = [SearchResult(int(ids[0, i]), float(d[0, i]), float(np.float32(-1) * w * d[0, i]))
               for i in range(int(cnt[0]))]
        return {r.node_id for r in res}, res
