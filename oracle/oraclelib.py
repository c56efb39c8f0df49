"""ctypes binding of the CPU oracle (oracle/oracle.cpp).

TEST INFRASTRUCTURE ONLY — importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs. The product package
(semadb_b200/) never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB = None

METRICS = {"euclidean": 0, "dot": 1, "cosine": 2, "hamming": 3, "jaccard": 4, "haversine": 5}
QUANT = {"none": 0, "binary": 1, "product": 2}

f32p = C.POINTER(C.c_float)
u32p = C.POINTER(C.c_uint32)
u16p = C.POINTER(C.c_uint16)
u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)
i64p = C.POINTER(C.c_int64)


def build(force: bool = False) -> Path:
    so = _HERE / "liboracle.so"
    src = _HERE / "oracle.cpp"
    if force or not so.exists() or (src.exists() and so.stat().st_mtime < src.stat().st_mtime):
        subprocess.run(["make", "-C", str(_HERE), "liboracle.so"], check=True, capture_output=True)
    return so


def _p(a, t):
    if a is None:
        return None
    return a.ctypes.data_as(t)


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    L = C.CDLL(str(build()))
    for name in ("orc_sq_l2_avx", "orc_dot_avx", "orc_sq_l2_pure", "orc_dot_pure", "orc_sq_l2_model", "orc_dot_model"):
        fn = getattr(L, name)
        fn.restype = C.c_float
        fn.argtypes = [f32p, f32p, C.c_size_t]
    L.orc_float_dist.restype = C.c_float
    L.orc_float_dist.argtypes = [C.c_int, f32p, f32p, C.c_size_t]
    L.orc_bit_dist.restype = C.c_float
    L.orc_bit_dist.argtypes = [C.c_int, u64p, u64p, C.c_size_t]
    L.orc_bq_encode.argtypes = [f32p, f32p, C.c_int, u64p]
    L.orc_bq_fit_threshold.argtypes = [f32p, C.c_size_t, C.c_int, f32p]
    L.orc_distset_new.restype = C.c_void_p
    L.orc_distset_new.argtypes = [C.c_int, f32p, C.c_int]
    L.orc_distset_op.argtypes = [C.c_void_p, C.c_int, u32p, C.c_int]
    L.orc_distset_items.restype = C.c_int
    L.orc_distset_items.argtypes = [C.c_void_p, u32p, f32p, C.c_int]
    L.orc_distset_free.argtypes = [C.c_void_p]
    L.orc_kmeans_fit.restype = C.c_int
    L.orc_kmeans_fit.argtypes = [f32p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_size_t,
                                 C.c_int, f32p, u8p, i64p]
    L.orc_index_new.restype = C.c_void_p
    L.orc_index_new.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_float, C.c_int, C.c_int,
                                C.c_int, C.c_int, C.c_int]
    L.orc_index_free.argtypes = [C.c_void_p]
    L.orc_index_set_start.argtypes = [C.c_void_p, f32p]
    L.orc_index_set_vectors.argtypes = [C.c_void_p, u32p, f32p, C.c_size_t]
    L.orc_index_insert.restype = C.c_int
    L.orc_index_insert.argtypes = [C.c_void_p, u32p, f32p, C.c_size_t, C.c_int]
    L.orc_index_insert_rounds.restype = C.c_int
    L.orc_index_insert_rounds.argtypes = [C.c_void_p, u32p, f32p, C.c_size_t, C.c_int, C.c_size_t]
    L.orc_index_fit.restype = C.c_int
    L.orc_index_fit.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int]
    L.orc_index_update_delete.argtypes = [C.c_void_p, u32p, f32p, u8p, C.c_size_t, C.c_int]
    L.orc_index_update_delete.restype = C.c_int
    L.orc_edge_scan.argtypes = [C.c_void_p, u32p, C.c_size_t, u32p, C.POINTER(C.c_size_t), u32p,
                                C.POINTER(C.c_size_t)]
    L.orc_edge_scan.restype = None
    L.orc_index_start_extra.argtypes = [C.c_void_p, u32p, C.c_size_t]
    L.orc_index_start_extra.restype = C.c_size_t
    L.orc_index_set_pq.restype = C.c_int
    L.orc_index_set_pq.argtypes = [C.c_void_p, f32p, f32p, C.c_int]
    L.orc_index_get_pq.restype = C.c_int
    L.orc_index_get_pq.argtypes = [C.c_void_p, f32p, f32p]
    L.orc_index_get_bq_threshold.restype = C.c_int
    L.orc_index_get_bq_threshold.argtypes = [C.c_void_p, f32p]
    L.orc_index_get_codes.restype = C.c_int
    L.orc_index_get_codes.argtypes = [C.c_void_p, u32p, C.c_size_t, u8p]
    L.orc_index_set_codes.restype = C.c_int
    L.orc_index_set_codes.argtypes = [C.c_void_p, u32p, u8p, C.c_size_t]
    L.orc_index_get_vectors.restype = C.c_int
    L.orc_index_get_vectors.argtypes = [C.c_void_p, u32p, C.c_size_t, f32p]
    L.orc_index_capacity.restype = C.c_uint64
    L.orc_index_capacity.argtypes = [C.c_void_p]
    L.orc_index_count.restype = C.c_uint64
    L.orc_index_count.argtypes = [C.c_void_p]
    L.orc_index_max_node_id.restype = C.c_uint32
    L.orc_index_max_node_id.argtypes = [C.c_void_p]
    L.orc_index_get_graph.argtypes = [C.c_void_p, C.c_size_t, u32p, u16p]
    L.orc_index_set_graph.argtypes = [C.c_void_p, C.c_size_t, u32p, u16p]
    L.orc_index_search.restype = C.c_int
    L.orc_index_search.argtypes = [C.c_void_p, f32p, C.c_size_t, C.c_int, C.c_int, u32p, C.c_size_t, u32p, f32p, u32p,
                                   u32p, u32p, u32p, f32p, u32p, u32p, f32p, u32p, C.c_int, C.c_int]
    L.orc_robust_prune.restype = C.c_int
    L.orc_robust_prune.argtypes = [C.c_void_p, C.c_uint32, u32p, f32p, C.c_int, u32p]
    L.orc_index_point_dist.restype = C.c_float
    L.orc_index_point_dist.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
    L.orc_index_query_dists.argtypes = [C.c_void_p, f32p, u32p, C.c_size_t, f32p]
    L.orc_index_adc_table.restype = C.c_int
    L.orc_index_adc_table.argtypes = [C.c_void_p, f32p, f32p]
    L.orc_flat_search.restype = C.c_int
    L.orc_flat_search.argtypes = [C.c_void_p, f32p, C.c_size_t, C.c_int, C.c_uint32, u32p, C.c_size_t, u32p, f32p,
                                  u32p, C.c_int]
    L.orc_merge_topk.argtypes = [u64p, f32p, u32p, C.c_int, C.c_size_t, C.c_int, u64p, f32p, u32p]
    L.orc_hybrid_merge.argtypes = [u64p, f32p, f32p, u32p, C.c_int, C.c_size_t, C.c_int, C.c_int, u64p, f32p, f32p, u32p]
    L.orc_hybrid_merge.restype = None
    L.orc_shard_limit.restype = C.c_int
    L.orc_shard_limit.argtypes = [C.c_int, C.c_int, C.c_int]
    L.orc_hw_threads.restype = C.c_int
    _LIB = L
    return L


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def float_dist(metric: str, x, y, impl: str = "avx") -> float:
    x, y = _f32(x), _f32(y)
    L = lib()
    if impl == "avx":
        return float(L.orc_float_dist(METRICS[metric], _p(x, f32p), _p(y, f32p), len(x)))
    fn = {("euclidean", "pure"): L.orc_sq_l2_pure, ("dot", "pure"): L.orc_dot_pure,
          ("euclidean", "model"): L.orc_sq_l2_model, ("dot", "model"): L.orc_dot_model,
          ("euclidean", "raw"): L.orc_sq_l2_avx, ("dot", "raw"): L.orc_dot_avx}[(metric, impl)]
    return float(fn(_p(x, f32p), _p(y, f32p), len(x)))


def bit_dist(metric: str, x, y) -> float:
    x = np.ascontiguousarray(x, dtype=np.uint64)
    y = np.ascontiguousarray(y, dtype=np.uint64)
    return float(lib().orc_bit_dist(METRICS[metric], _p(x, u64p), _p(y, u64p), len(x)))


def bq_encode(v, thr) -> np.ndarray:
    v, thr = _f32(v), _f32(thr)
    out = np.zeros((len(v) + 63) // 64, dtype=np.uint64)
    lib().orc_bq_encode(_p(v, f32p), _p(thr, f32p), len(v), _p(out, u64p))
    return out


def bq_fit_threshold(X) -> np.ndarray:
    X = _f32(X)
    out = np.zeros(X.shape[1], dtype=np.float32)
    lib().orc_bq_fit_threshold(_p(X, f32p), X.shape[0], X.shape[1], _p(out, f32p))
    return out


class DistSet:
    """distset_test.go harness (ids index into a distance table)."""

    def __init__(self, capacity: int, dists):
        self._d = _f32(dists)
        self._h = lib().orc_distset_new(capacity, _p(self._d, f32p), len(self._d))

    def _op(self, op, ids):
        ids = _u32(ids)
        lib().orc_distset_op(self._h, op, _p(ids, u32p), len(ids))

    def add_with_limit(self, *ids):
        self._op(0, ids)

    def add(self, *ids):
        self._op(1, ids)

    def sort(self):
        self._op(2, [])

    def items(self):
        ids = np.zeros(4096, dtype=np.uint32)
        d = np.zeros(4096, dtype=np.float32)
        n = lib().orc_distset_items(self._h, _p(ids, u32p), _p(d, f32p), 4096)
        return ids[:n].tolist(), d[:n].tolist()

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_distset_free(self._h)
            self._h = None


def kmeans_fit(X, K, max_iter=100, offset=0, length=None, first=0, alias=False):
    """utils.KMeans.Fit. Returns (centroids[K,len], labels[n], iters, init_rows[K]); with
    alias=True X is modified in place exactly as the reference does (kmeans.go:63,82,144)."""
    assert X.dtype == np.float32 and X.flags.c_contiguous
    n, stride = X.shape
    length = stride - offset if length is None else length
    cent = np.zeros((K, length), dtype=np.float32)
    labels = np.zeros(n, dtype=np.uint8)
    rows = np.zeros(K, dtype=np.int64)
    it = lib().orc_kmeans_fit(_p(X, f32p), n, stride, offset, length, K, max_iter, first, int(alias), _p(cent, f32p),
                              _p(labels, u8p), _p(rows, i64p))
    return cent, labels, it, rows


class OracleIndex:
    """The reference's IndexVamana + VectorStore, restated (dense u32 node ids)."""

    def __init__(self, dim, metric="euclidean", search_size=75, degree_bound=64, alpha=1.2, quantizer="none",
                 bq_threshold=None, bq_metric="hamming", bq_trigger=0, pq_m=0, pq_k=0, pq_trigger=0):
        self.dim, self.metric, self.L, self.R = dim, metric, search_size, degree_bound
        self.quant = quantizer
        self.pq_m, self.pq_k = pq_m, pq_k
        thr = float("nan") if bq_threshold is None else float(bq_threshold)
        self._h = lib().orc_index_new(dim, METRICS[metric], search_size, degree_bound, alpha, QUANT[quantizer], thr,
                                      METRICS[bq_metric], bq_trigger, pq_m, pq_k, pq_trigger)
        if not self._h:
            raise ValueError("invalid index parameters")
        if metric in ("hamming", "jaccard"):
            self.quant = "binary"

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_index_free(self._h)
            self._h = None

    def set_start(self, v):
        v = _f32(v)
        assert v.shape == (self.dim,)
        lib().orc_index_set_start(self._h, _p(v, f32p))

    def set_vectors(self, ids, vecs):
        ids, vecs = _u32(ids), _f32(vecs)
        lib().orc_index_set_vectors(self._h, _p(ids, u32p), _p(vecs, f32p), len(ids))

    def insert(self, ids, vecs, threads=1, max_round=0):
        """max_round 0: the reference's schedule (sequential, or concurrent workers when threads > 1);
        max_round > 0: rounds of at most that many points, a graph independent of threads and timing."""
        ids, vecs = _u32(ids), _f32(vecs)
        assert vecs.shape == (len(ids), self.dim)
        if max_round:
            rc = lib().orc_index_insert_rounds(self._h, _p(ids, u32p), _p(vecs, f32p), len(ids), threads, max_round)
        else:
            rc = lib().orc_index_insert(self._h, _p(ids, u32p), _p(vecs, f32p), len(ids), threads)
        if rc:
            raise RuntimeError(f"oracle insert failed rc={rc}")

    def update_delete(self, ids, vecs, has_vec, threads=1):
        """insertUpdateDelete (vamana.go:136-263) minus Fit: has_vec[i] == 0 is a nil vector."""
        ids, vecs = _u32(ids), _f32(vecs)
        hv = np.ascontiguousarray(has_vec, dtype=np.uint8)
        assert vecs.shape == (len(ids), self.dim) and hv.shape == (len(ids),)
        rc = lib().orc_index_update_delete(self._h, _p(ids, u32p), _p(vecs, f32p), _p(hv, u8p), len(ids), threads)
        if rc:
            raise RuntimeError(f"oracle update_delete failed rc={rc}")

    def edge_scan(self, delete_ids):
        """EdgeScan (node.go:142-199): (toPrune, toSave) in ascending id order."""
        d = _u32(delete_ids)
        cap = self.capacity
        tp, ts = np.zeros(cap, dtype=np.uint32), np.zeros(cap, dtype=np.uint32)
        n1, n2 = C.c_size_t(0), C.c_size_t(0)
        lib().orc_edge_scan(self._h, _p(d, u32p), len(d), _p(tp, u32p), C.byref(n1), _p(ts, u32p), C.byref(n2))
        return tp[:n1.value].copy(), ts[:n2.value].copy()

    def start_extra(self):
        n = int(lib().orc_index_start_extra(self._h, None, 0))
        out = np.zeros(max(n, 1), dtype=np.uint32)
        lib().orc_index_start_extra(self._h, _p(out, u32p), n)
        return out[:n]

    def fit(self, pq_first=0, pq_alias=False, threads=1):
        return lib().orc_index_fit(self._h, pq_first, int(pq_alias), threads)

    def set_pq(self, flat_centroids, centroid_dists, reencode=True):
        fc, cd = _f32(flat_centroids), _f32(centroid_dists)
        rc = lib().orc_index_set_pq(self._h, _p(fc, f32p), _p(cd, f32p), int(reencode))
        assert rc == 0

    def get_pq(self):
        sub = self.dim // self.pq_m
        fc = np.zeros((self.pq_m, self.pq_k, sub), dtype=np.float32)
        cd = np.zeros((self.pq_m, self.pq_k, self.pq_k), dtype=np.float32)
        rc = lib().orc_index_get_pq(self._h, _p(fc, f32p), _p(cd, f32p))
        return (fc, cd) if rc == 0 else None

    def get_bq_threshold(self):
        t = np.zeros(self.dim, dtype=np.float32)
        rc = lib().orc_index_get_bq_threshold(self._h, _p(t, f32p))
        return t if rc == 0 else None

    def get_codes(self, ids):
        ids = _u32(ids)
        width = self.pq_m if self.quant == "product" else 8 * ((self.dim + 63) // 64)
        out = np.zeros((len(ids), width), dtype=np.uint8)
        rc = lib().orc_index_get_codes(self._h, _p(ids, u32p), len(ids), _p(out, u8p))
        assert rc == 0
        return out

    def set_codes(self, ids, codes):
        """Hydrate from quantised codes alone (binary.go:275-296, product.go:349-371)."""
        ids = _u32(ids)
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        rc = lib().orc_index_set_codes(self._h, _p(ids, u32p), _p(codes, u8p), len(ids))
        if rc:
            raise RuntimeError(f"oracle set_codes failed rc={rc}")

    def get_vectors(self, ids):
        ids = _u32(ids)
        out = np.zeros((len(ids), self.dim), dtype=np.float32)
        lib().orc_index_get_vectors(self._h, _p(ids, u32p), len(ids), _p(out, f32p))
        return out

    @property
    def capacity(self):
        return int(lib().orc_index_capacity(self._h))

    @property
    def count(self):
        return int(lib().orc_index_count(self._h))

    @property
    def max_node_id(self):
        return int(lib().orc_index_max_node_id(self._h))

    def get_graph(self, n=None):
        n = self.max_node_id + 1 if n is None else n
        n = max(n, 2)
        adj = np.zeros((n, self.R), dtype=np.uint32)
        deg = np.zeros(n, dtype=np.uint16)
        lib().orc_index_get_graph(self._h, n, _p(adj, u32p), _p(deg, u16p))
        return adj, deg

    def set_graph(self, adj, deg):
        adj = _u32(adj)
        deg = np.ascontiguousarray(deg, dtype=np.uint16)
        lib().orc_index_set_graph(self._h, adj.shape[0], _p(adj, u32p), _p(deg, u16p))

    def search(self, queries, k=10, search_size=None, filter_ids=None, threads=1, diagnostics=False, vis_cap=0):
        q = _f32(queries)
        B = q.shape[0]
        L = self.L if search_size is None else search_size
        ids = np.zeros((B, k), dtype=np.uint32)
        d = np.zeros((B, k), dtype=np.float32)
        cnt = np.zeros(B, dtype=np.uint32)
        filt = None if filter_ids is None else np.sort(_u32(filter_ids))
        hops = ndist = lids = ldist = llen = vids = vd = vlen = None
        if diagnostics:
            hops = np.zeros(B, dtype=np.uint32)
            ndist = np.zeros(B, dtype=np.uint32)
            lids = np.zeros((B, L), dtype=np.uint32)
            ldist = np.zeros((B, L), dtype=np.float32)
            llen = np.zeros(B, dtype=np.uint32)
        if vis_cap:
            vids = np.zeros((B, vis_cap), dtype=np.uint32)
            vd = np.zeros((B, vis_cap), dtype=np.float32)
            vlen = np.zeros(B, dtype=np.uint32)
        rc = lib().orc_index_search(self._h, _p(q, f32p), B, k, L, _p(filt, u32p), 0 if filt is None else len(filt),
                                    _p(ids, u32p), _p(d, f32p), _p(cnt, u32p), _p(hops, u32p), _p(ndist, u32p),
                                    _p(lids, u32p), _p(ldist, f32p), _p(llen, u32p), _p(vids, u32p), _p(vd, f32p),
                                    _p(vlen, u32p), vis_cap, threads)
        if rc == 1:
            raise ValueError(f"searchSize ({L}) must be greater than k ({k})")
        if rc:
            raise RuntimeError(f"oracle search failed rc={rc}")
        out = {"ids": ids, "dists": d, "counts": cnt}
        if diagnostics:
            out.update(hops=hops, ndist=ndist, list_ids=lids, list_dists=ldist, list_len=llen)
        if vis_cap:
            out.update(vis_ids=vids, vis_dists=vd, vis_len=vlen)
        return out

    def robust_prune(self, node, cand_ids, cand_dists):
        ci, cd = _u32(cand_ids), _f32(cand_dists)
        out = np.zeros(self.R, dtype=np.uint32)
        n = lib().orc_robust_prune(self._h, node, _p(ci, u32p), _p(cd, f32p), len(ci), _p(out, u32p))
        return out[:n]

    def point_dist(self, x, y):
        return float(lib().orc_index_point_dist(self._h, x, y))

    def query_dists(self, query, ids):
        q, ids = _f32(query), _u32(ids)
        out = np.zeros(len(ids), dtype=np.float32)
        lib().orc_index_query_dists(self._h, _p(q, f32p), _p(ids, u32p), len(ids), _p(out, f32p))
        return out

    def adc_table(self, query):
        q = _f32(query)
        out = np.zeros((self.pq_m, self.pq_k), dtype=np.float32)
        rc = lib().orc_index_adc_table(self._h, _p(q, f32p), _p(out, f32p))
        return out if rc == 0 else None

    def flat_search(self, queries, k=10, first_id=2, filter_ids=None, threads=1):
        q = _f32(queries)
        B = q.shape[0]
        ids = np.zeros((B, k), dtype=np.uint32)
        d = np.zeros((B, k), dtype=np.float32)
        cnt = np.zeros(B, dtype=np.uint32)
        filt = None if filter_ids is None else np.sort(_u32(filter_ids))
        lib().orc_flat_search(self._h, _p(q, f32p), B, k, first_id, _p(filt, u32p), 0 if filt is None else len(filt),
                              _p(ids, u32p), _p(d, f32p), _p(cnt, u32p), threads)
        return {"ids": ids, "dists": d, "counts": cnt}


def merge_topk(ids, dists, counts, k):
    """cluster/actions.go:357-376. ids/dists: [S,B,k]; counts: [S,B]."""
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    dists = _f32(dists)
    counts = _u32(counts)
    S, B, kk = ids.shape
    assert kk == k
    oi = np.zeros((B, k), dtype=np.uint64)
    od = np.zeros((B, k), dtype=np.float32)
    oc = np.zeros(B, dtype=np.uint32)
    lib().orc_merge_topk(_p(ids, u64p), _p(dists, f32p), _p(counts, u32p), S, B, k, _p(oi, u64p), _p(od, f32p),
                         _p(oc, u32p))
    return oi, od, oc


def hybrid_merge(ids, hybrid, dists, counts, disjunction):
    """shard/index/search.go:259-298. ids/hybrid/dists: [S,B,k]; counts: [S,B] -> [B,S*k] lists."""
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    hybrid, dists, counts = _f32(hybrid), _f32(dists), _u32(counts)
    S, B, k = ids.shape
    oi = np.zeros((B, S * k), dtype=np.uint64)
    oh = np.zeros((B, S * k), dtype=np.float32)
    od = np.zeros((B, S * k), dtype=np.float32)
    oc = np.zeros(B, dtype=np.uint32)
    lib().orc_hybrid_merge(_p(ids, u64p), _p(hybrid, f32p), _p(dists, f32p), _p(counts, u32p), S, B, k,
                           1 if disjunction else 0, _p(oi, u64p), _p(oh, f32p), _p(od, f32p), _p(oc, u32p))
    return oi, oh, od, oc


def shard_limit(limit, nshards, max_search_limit=75):
    return int(lib().orc_shard_limit(limit, nshards, max_search_limit))


def hw_threads():
    return int(lib().orc_hw_threads())


def random_unit_vector(dim, seed):
    """setupStartNode (vamana.go:100-110) with a seeded generator: U(-1,1) normalised."""
    rng = np.random.Generator(np.random.PCG64(seed))
    v = (rng.random(dim, dtype=np.float32) * np.float32(2) - np.float32(1)).astype(np.float32)
    s = np.float32(0)
    for x in v:
        s = np.float32(s + x * x)
    norm = np.float32(1) / np.float32(np.sqrt(np.float64(s)))
    return (v * norm).astype(np.float32)
