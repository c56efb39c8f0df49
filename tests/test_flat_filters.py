"""Flat search with one filter per request (sdb_flat_search_batch_filters): every store the flat
scan serves against the oracle, both routes (gathered rows, range scan with a bitmap) against each
other, chunked filters, the per-request contract, the old single-filter entry and the errors."""
import numpy as np
import pytest

from oracle import oraclelib as O
from semadb_b200 import _capi, synth
from semadb_b200._capi import SdbError
from semadb_b200.vamana import (IndexFlat, IndexVamana, IndexVectorFlatParameters, IndexVectorVamanaParameters,
                                ProductQuantizerParameters, Quantizer)

pytestmark = pytest.mark.gpu

u64p, f32p, u32p, i32p = _capi.u64p, _capi.f32p, _capi.u32p, _capi.i32p


def _store(n, dim, metric, seed):
    if metric == "haversine":
        rng = np.random.Generator(np.random.PCG64(seed))
        X = np.stack([rng.uniform(-80, 80, n), rng.uniform(-179, 179, n)], axis=1).astype(np.float32)
    elif metric in ("hamming", "jaccard"):
        X = synth.planted_bits(n, dim, seed=seed, n_proto=32)
    else:
        X = synth.latent_gaussian(n, dim, seed=seed, latent=8)
    return X


def _filters(rng, ids, k, deleted, rows_hint):
    """Sizes 0, 1, k-1, k, k+1, 1 000 and all ids, and lists naming deleted ids, ids beyond the store
    and ids 0 and 1 (never matched)."""
    pick = lambda m: np.sort(rng.choice(ids, size=min(m, len(ids)), replace=False))
    fs = [np.zeros(0, np.uint64), pick(1), pick(max(k - 1, 0)), pick(k), pick(k + 1), pick(1000), ids.copy()]
    fs.append(np.union1d(pick(30), deleted))
    fs.append(np.union1d(pick(20), [rows_hint + 7, rows_hint * 4 + 3, 1 << 40]))
    fs.append(np.union1d(pick(k), [0, 1]))
    return [np.asarray(f, dtype=np.uint64) for f in fs]


def _assign(B, n_filters, seed):
    """Every filter at least once, plus unfiltered requests (-1)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    qf = np.array([(b % (n_filters + 1)) - 1 for b in range(B)], dtype=np.int32)
    rng.shuffle(qf)
    return qf


def _check_oracle(g, oix, Q, filters, qf, k, exact=True):
    fi, fd, fc = g.flat_search_batch_filters(Q, filters, qf, k)
    plain = oix.flat_search(Q, k=k, threads=8)
    for b in range(len(Q)):
        if qf[b] < 0:
            ref = {key: v[b] for key, v in plain.items()}
        else:
            f = filters[qf[b]]
            f = f[(f >= 2) & (f < np.uint64(1 << 32))].astype(np.uint32)  # ids below 2 never match
            if len(f):
                r = oix.flat_search(Q[b:b + 1], k=k, filter_ids=f, threads=1)
                ref = {key: v[0] for key, v in r.items()}
            else:
                ref = {"counts": 0, "ids": np.zeros(k, np.uint32), "dists": np.full(k, np.inf, np.float32)}
        assert fc[b] == ref["counts"], (b, qf[b])
        assert (fi[b] == ref["ids"].astype(np.uint64)).all(), (b, qf[b])
        if exact:
            assert fd[b].tobytes() == ref["dists"].tobytes(), (b, qf[b])
        else:
            n = int(fc[b])
            assert np.allclose(fd[b, :n], ref["dists"][:n], rtol=1e-5, atol=1.0), (b, qf[b])
    return fi, fd, fc


def _both_routes(g, Q, filters, qf, k, monkeypatch):
    monkeypatch.delenv("SDB_FLAT_EXACT", raising=False)
    a = g.flat_search_batch_filters(Q, filters, qf, k)
    sa = g.flat_last_filter_stats()
    monkeypatch.setenv("SDB_FLAT_EXACT", "1")
    b = g.flat_search_batch_filters(Q, filters, qf, k)
    sb = g.flat_last_filter_stats()
    monkeypatch.delenv("SDB_FLAT_EXACT")
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    assert sb[0] == 0 and sb[1] == sa[0] + sa[1] and sb[2] == 0
    return a, sa


# ---------------------------------------------------------------- oracle parity, every store

@pytest.mark.parametrize("dim,metric", [(128, "euclidean"), (128, "dot"), (128, "cosine"), (100, "euclidean"),
                                        (100, "dot"), (768, "cosine"), (768, "euclidean"), (2, "haversine")])
def test_f32_stores_match_oracle(dim, metric, monkeypatch):
    n = 3000
    X = _store(n, dim, metric, seed=dim + 3)
    X[2500:2550] = X[:50]  # exact duplicates: ties by ascending id
    Q = np.concatenate([_store(40, dim, metric, seed=dim + 4), X[:8]])
    ids = np.arange(2, n + 2, dtype=np.uint64)
    deleted = ids[::97]
    g = IndexFlat(IndexVectorFlatParameters(dim, metric))
    g.set_vectors(ids, X)
    g.delete_rows(deleted)
    live = np.setdiff1d(ids, deleted)
    oix = O.OracleIndex(dim, metric)
    oix.set_vectors(live.astype(np.uint32), X[live.astype(np.int64) - 2])
    rng = np.random.Generator(np.random.PCG64(dim))
    for k in (1, 10, 75):
        filters = _filters(rng, live, k, deleted, n + 2)
        qf = _assign(len(Q), len(filters), k)
        exact = metric != "haversine"  # float64 sin/cos/asin: CUDA's libm vs glibc
        a = _check_oracle(g, oix, Q, filters, qf, k, exact=exact)
        b, _ = _both_routes(g, Q, filters, qf, k, monkeypatch)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))  # haversine: bit-identical to the scan


@pytest.mark.parametrize("metric", ["hamming", "jaccard"])
def test_binary_store_matches_oracle(metric, monkeypatch):
    n, dim = 3000, 256
    X = _store(n, dim, metric, seed=7)
    X[2500:2550] = X[:50]
    Q = _store(40, dim, metric, seed=8)
    ids = np.arange(2, n + 2, dtype=np.uint64)
    g = IndexVamana("bq", IndexVectorVamanaParameters(dim, metric), start_vector=synth.start_vector(dim, 5))
    g.set_vectors(ids, X)
    deleted = ids[::89]
    g.delete_rows(deleted)
    live = np.setdiff1d(ids, deleted)
    oix = O.OracleIndex(dim, metric)
    oix.set_vectors(live.astype(np.uint32), X[live.astype(np.int64) - 2])
    rng = np.random.Generator(np.random.PCG64(3))
    for k in (1, 10, 75):
        filters = _filters(rng, live, k, deleted, n + 2)
        qf = _assign(len(Q), len(filters), k + 1)
        _check_oracle(g, oix, Q, filters, qf, k)
        _both_routes(g, Q, filters, qf, k, monkeypatch)


def test_pq_store_matches_oracle(monkeypatch):
    n, dim, M, K = 3000, 64, 16, 64
    X = _store(n, dim, "euclidean", seed=21)
    X[2500:2550] = X[:50]
    Q = _store(40, dim, "euclidean", seed=22)
    ids = np.arange(2, n + 2, dtype=np.uint64)
    start = synth.start_vector(dim, 5)
    oix = O.OracleIndex(dim, "euclidean", quantizer="product", pq_m=M, pq_k=K, pq_trigger=1000)
    oix.set_start(start)
    g = IndexVamana("pq", IndexVectorVamanaParameters(dim, "euclidean", quantizer=Quantizer(
        "product", product=ProductQuantizerParameters(K, M, 1000))), start_vector=start)
    oix.set_vectors(ids.astype(np.uint32), X)
    g.set_vectors(ids, X)
    assert oix.fit(pq_first=3, pq_alias=True, threads=8) == 1
    assert g.fit(3) is True
    assert g.get_codes(ids[:200]).tobytes() == oix.get_codes(ids[:200].astype(np.uint32)).tobytes()
    rng = np.random.Generator(np.random.PCG64(4))
    for k in (1, 10, 75):
        filters = _filters(rng, ids, k, np.zeros(0, np.uint64), n + 2)
        qf = _assign(len(Q), len(filters), k + 2)
        _check_oracle(g, oix, Q, filters, qf, k)
        _both_routes(g, Q, filters, qf, k, monkeypatch)


# ---------------------------------------------------------------- routes, chunks, contract

def _tc_store(n=20_000, dim=128):
    X = synth.latent_gaussian(n, dim, seed=5, latent=8)
    ids = np.arange(2, n + 2, dtype=np.uint64)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(ids, X)
    return g, X, ids


def test_route_ab_both_routes_taken(monkeypatch):
    """A dense filter shared by 600 requests takes the range scan, sparse per-request filters the
    gather route; forcing the scan for every filter gives the same bytes."""
    g, X, ids = _tc_store()
    rng = np.random.Generator(np.random.PCG64(9))
    Q = synth.latent_gaussian(1000, 128, seed=6, latent=8)
    dense = np.sort(rng.choice(ids, size=len(ids) // 2, replace=False))
    filters = [dense] + [np.sort(rng.choice(ids, size=50, replace=False)) for _ in range(300)]
    qf = np.concatenate([np.zeros(600, np.int32), np.arange(1, 301, dtype=np.int32), -np.ones(100, np.int32)])
    for k in (10, 75):
        (fi, fd, fc), (gathered, scanned, pairs) = _both_routes(g, Q, filters, qf, k, monkeypatch)
        assert scanned == 1 and gathered == 300 and pairs == 300 * 50, (gathered, scanned, pairs)
        for b in (0, 599, 600, 899, 950):
            one = g.flat_search_batch(Q[b:b + 1], k, None if qf[b] < 0 else filters[qf[b]])
            assert fi[b].tobytes() == one[0][0].tobytes() and fd[b].tobytes() == one[1][0].tobytes() and fc[b] == one[2][0]


def test_chunking_duplicates_across_chunks(monkeypatch):
    """One filter of 5 000 ids (five work items) whose rows repeat across chunks: ties by ascending id
    across the chunk merge."""
    n, dim = 20_000, 128
    X = synth.latent_gaussian(n, dim, seed=12, latent=8)
    filt = np.arange(2, 5002, dtype=np.uint64)
    for c in range(1, 5):  # rows of chunk 0 repeated at the start of chunks 1..4 (ids 2+1024c ..)
        X[1024 * c:1024 * c + 100] = X[:100]
    ids = np.arange(2, n + 2, dtype=np.uint64)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(ids, X)
    oix = O.OracleIndex(dim, "euclidean")
    oix.set_vectors(ids.astype(np.uint32), X)
    Q = np.concatenate([X[:40], synth.latent_gaussian(10, dim, seed=13, latent=8)])
    for k in (5, 75):
        fi, fd, fc = g.flat_search_batch_filters(Q, [filt], None, k)
        assert g.flat_last_filter_stats() == (1, 0, len(Q) * len(filt))
        ref = oix.flat_search(Q, k=k, filter_ids=filt.astype(np.uint32), threads=8)
        assert (fi == ref["ids"].astype(np.uint64)).all() and fd.tobytes() == ref["dists"].tobytes()
        assert (fi[:40, 0] == np.arange(2, 42)).all() and (fi[:40, 1] == np.arange(1026, 1066)).all()
        _both_routes(g, Q, [filt], None, k, monkeypatch)


def test_contract_rows_equal_single_calls(monkeypatch):
    """Each row equals flat_search_batch of that query alone with its filter; the unfiltered rows of
    a mixed batch on a store served by the tensor-core pass equal the unfiltered batch call."""
    monkeypatch.delenv("SDB_FLAT_EXACT", raising=False)
    g, X, ids = _tc_store()
    rng = np.random.Generator(np.random.PCG64(14))
    Q = synth.latent_gaussian(300, 128, seed=15, latent=8)
    filters = [np.sort(rng.choice(ids, size=m, replace=False)) for m in (0, 3, 10, 11, 700, 5000)]
    qf = _assign(len(Q), len(filters), 16)
    k = 10
    fi, fd, fc = g.flat_search_batch_filters(Q, filters, qf, k)
    plain = qf < 0
    assert g.flat_last_stats()[0] == 2  # the unfiltered subset took the tensor-core pass
    ui, ud, uc = g.flat_search_batch(Q, k)
    assert fi[plain].tobytes() == ui[plain].tobytes() and fd[plain].tobytes() == ud[plain].tobytes()
    assert (fc[plain] == uc[plain]).all()
    for b in range(0, len(Q), 7):
        one = g.flat_search_batch(Q[b:b + 1], k, None if qf[b] < 0 else filters[qf[b]])
        assert fi[b].tobytes() == one[0][0].tobytes() and fd[b].tobytes() == one[1][0].tobytes() and fc[b] == one[2][0], b
    # the whole batch unfiltered through the filtered entry, and n_filters == 0
    a = g.flat_search_batch_filters(Q, filters, -np.ones(len(Q), np.int32), k)
    b = g.flat_search_batch_filters(Q, [], None, k)
    for x, y, z in zip(a, b, (ui, ud, uc)):
        assert x.tobytes() == z.tobytes() and y.tobytes() == z.tobytes()


def _raw_flat(g, Q, k, filt):
    B = len(Q)
    ids, d, c = np.zeros((B, k), np.uint64), np.zeros((B, k), np.float32), np.zeros(B, np.uint32)
    _capi.check(g._lib.sdb_flat_search_batch(g._h, B, Q.ctypes.data_as(f32p), k, filt.ctypes.data_as(u64p), len(filt),
                                             ids.ctypes.data_as(u64p), d.ctypes.data_as(f32p), c.ctypes.data_as(u32p)))
    return ids, d, c


def test_old_entry_unsorted_duplicated_filter():
    g, X, ids = _tc_store(n=5000)
    rng = np.random.Generator(np.random.PCG64(17))
    Q = np.ascontiguousarray(synth.latent_gaussian(20, 128, seed=18, latent=8))
    base = rng.choice(ids, size=300, replace=False)
    messy = np.ascontiguousarray(np.concatenate([base, base[:50], [3, 3]])[rng.permutation(352)], dtype=np.uint64)
    clean = np.unique(messy)
    for k in (10, 75):
        a = _raw_flat(g, Q, k, messy)
        b = _raw_flat(g, Q, k, clean)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
        assert g.flat_last_filter_stats()[0] + g.flat_last_filter_stats()[1] == 1


def test_errors_leave_the_handle_usable():
    g, X, ids = _tc_store(n=5000)
    Q = np.ascontiguousarray(X[:4])
    B, k = len(Q), 10
    out = np.zeros((B, k), np.uint64), np.zeros((B, k), np.float32), np.zeros(B, np.uint32)
    outp = [out[0].ctypes.data_as(u64p), out[1].ctypes.data_as(f32p), out[2].ctypes.data_as(u32p)]

    def raw(filt, offs, qf):
        f = np.ascontiguousarray(filt, dtype=np.uint64)
        o = np.ascontiguousarray(offs, dtype=np.uint64)
        q = None if qf is None else np.ascontiguousarray(qf, dtype=np.int32)
        return g._lib.sdb_flat_search_batch_filters(g._h, B, Q.ctypes.data_as(f32p), k, len(o) - 1, f.ctypes.data_as(u64p),
                                                    o.ctypes.data_as(u64p), None if q is None else q.ctypes.data_as(i32p),
                                                    *outp)

    assert raw([5, 4, 9], [0, 3], None) == _capi.ERR_INVALID  # descending
    assert raw([5, 5, 9], [0, 3], None) == _capi.ERR_INVALID  # duplicate
    assert raw([4, 5, 9], [0, 3], [0, 1, 0, -1]) == _capi.ERR_INVALID  # query_filter index out of range
    for bad_k in (0, 76):
        with pytest.raises(SdbError) as e:
            g.flat_search_batch_filters(Q, [[4, 5]], None, bad_k)
        assert e.value.code == _capi.ERR_INVALID
    assert raw([4, 5, 9], [0, 3], [0, -1, 0, 0]) == _capi.OK
    assert (out[2] == np.array([3, 10, 3, 3])).all()
    ref = g.flat_search_batch(Q, k, [4, 5, 9])
    assert out[0][0].tobytes() == ref[0][0].tobytes() and out[1][0].tobytes() == ref[1][0].tobytes()
