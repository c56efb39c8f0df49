"""Every dimension-specialised f32 and PQ kernel variant against the oracle and a float64 reference.

The hot kernels are compiled per dimension class, so each class runs different code:
- beam search (K1, search_launch.cuh launch_float): FIXED 4 / 8 / 12 / 24 trips of 32 floats
  (dim 128 / 256 / 384 / 768), GENERIC otherwise, each with a RETRY form (exact visited bitmap)
  and a FILTER form;
- batched insert (K8): how many candidate rows robustPrune stages in shared memory shrinks with
  the row width (64 at dim 128, a handful at 4096), the rest is read from global memory;
- flat exact scan (K5, flat.cu): the query tile in shared memory up to dim ~403, streamed through
  L1 above; the point tile shrinks once 16 rows of it no longer fit (dim > ~3 632);
- flat tensor-core path (flat_tc.cu): tcgen05 for padded dims up to 384, the mma.sync level
  scheme above, and an exact re-score whose query rows pass 48 KB of shared memory above 3 072;
- PQ search: on-the-fly evaluators for sub-vectors of 4, 8 and 16 floats, the per-query table in
  shared memory (chunks of up to 8 x 16 sub-vectors) or through L1/L2.

Results must equal the oracle bit for bit. The oracle restates the reference in f32, so returned
distances are also held to a float64 reference within the f32 summation bound
(tests/helpers.f64_dists): a tail both forgot would agree with itself, not with float64."""
import functools

import numpy as np
import pytest

from oracle import oraclelib as O
from semadb_b200 import synth
from semadb_b200.vamana import (IndexFlat, IndexVamana, IndexVectorFlatParameters, IndexVectorVamanaParameters,
                                ProductQuantizerParameters, Quantizer)
from tests.helpers import check_graph_equal, check_search, f64_dists, mirror_to_gpu, oracle_graph

METRICS = ("euclidean", "dot", "cosine")


def _data(n, dim, seed, metric, w_seed=None):
    return synth.latent_gaussian(n, dim, seed=seed, w_seed=w_seed, latent=8, normalize=(metric == "cosine"))


# ---------------------------------------------------------------- float64 reference (CPU only)

@pytest.mark.parametrize("dim", [1, 2, 7, 31, 32, 33, 100, 128, 384, 768, 1000, 1536, 4096])
def test_f64_bound_contains_oracle_distances(dim):
    """The bound holds for the oracle's f32 distances (the reference's summation order), and it
    is tight enough to see one 32-float trip of squared L2 left out."""
    rng = np.random.Generator(np.random.PCG64(dim))
    X = rng.standard_normal((64, dim)).astype(np.float32)
    Y = rng.standard_normal((64, dim)).astype(np.float32)
    for metric in METRICS:
        f32 = np.array([O.float_dist(metric, X[i], Y[i]) for i in range(64)], np.float64)
        d, b = f64_dists(metric, X, Y)
        d, b = np.diag(d), np.diag(b)
        assert (np.abs(f32 - d) <= b).all(), metric
    if dim >= 64:
        d, b = f64_dists("euclidean", X, Y)
        short, _ = f64_dists("euclidean", X[:, :dim - 32], Y[:, :dim - 32])
        assert (np.abs(np.diag(short) - np.diag(d)) > np.diag(b)).all()


def _check_f64_rows(metric, Q, X, ids, d, cnt):
    """Every returned distance lies within the f32 bound of its float64 value (ids start at 2)."""
    for b in range(len(Q)):
        n = int(cnt[b])
        rows = X[ids[b, :n].astype(np.int64) - 2]
        ref, bound = f64_dists(metric, Q[b:b + 1], rows)
        assert (np.abs(d[b, :n].astype(np.float64) - ref[0]) <= bound[0]).all(), b


def _check_f64_flat(metric, Q, X, ids, d, cnt, k, chunk=4096):
    """Flat search against float64 brute force: each returned distance within the bound of its
    float64 value, and no returned point farther (in float64) than the float64 k-th nearest plus
    the two bounds that separate them — ties and near-ties may resolve either way, nothing else."""
    parts = [f64_dists(metric, Q, X[s:s + chunk]) for s in range(0, len(X), chunk)]
    D = np.concatenate([p[0] for p in parts], axis=1)
    Bd = np.concatenate([p[1] for p in parts], axis=1)
    assert (cnt == min(k, len(X))).all()
    for b in range(len(Q)):
        rows = ids[b, :k].astype(np.int64) - 2
        assert (np.abs(d[b, :k].astype(np.float64) - D[b, rows]) <= Bd[b, rows]).all(), b
        top = np.argpartition(D[b], k - 1)[:k]
        kth = D[b, top].max()
        assert (D[b, rows] <= kth + Bd[b, rows] + Bd[b, top].max()).all(), b


# ---------------------------------------------------------------- beam search (K1)

@functools.lru_cache(maxsize=None)
def _graph(dim, metric):
    """Oracle-built graph mirrored onto the GPU, shared by the search tests of one (dim, metric)."""
    n = 1000 if dim >= 4096 else 2000
    X = _data(n, dim, dim, metric)
    Q = _data(200, dim, dim + 1, metric, w_seed=dim)
    oix, ids, start = oracle_graph(X, metric)
    g = mirror_to_gpu(oix, X, ids, start, metric)
    return oix, g, X, Q, ids


def _search_all(dim, metric):
    oix, g, X, Q, _ = _graph(dim, metric)
    for B, k, L in ((200, 10, 75), (50, 1, 25), (50, 75, 75)):
        check_search(oix, g, Q[:B], k=k, L=L)
        ids, d, cnt = g.search_batch(Q[:B], k, L)
        _check_f64_rows(metric, Q[:B], X, ids, d, cnt)


@pytest.mark.gpu
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("dim", [256, 768])
def test_search_fixed_trips(dim, metric):
    """FIXED 8 and 24 trips; each metric is its own translation unit."""
    _search_all(dim, metric)


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", [(385, "euclidean"), (1024, "dot"), (1536, "cosine"), (4096, "euclidean")])
def test_search_generic_wide(dim, metric):
    """GENERIC above 128: a tail past the last 32-float trip (385), multiples of 32 with no FIXED
    case (1024, 1536) and the widest rows an index accepts."""
    _search_all(dim, metric)


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", [(256, "euclidean"), (768, "dot"), (1024, "dot")])
def test_search_retry_wide(dim, metric, monkeypatch):
    """A visited table far too small for any query sends every query to the RETRY instantiation
    of its evaluator; results, hops and evaluations still equal the oracle's, and so does the
    visited list the insert path reads."""
    oix, g, X, Q, _ = _graph(dim, metric)
    monkeypatch.setenv("SDB_VT_SLOTS", "64")
    check_search(oix, g, Q[:100])
    vi, vd, vn = g.search_visited(Q[:50], 75, 256)
    ref = oix.search(Q[:50], k=1, vis_cap=256, threads=8)
    assert (vn == ref["vis_len"]).all()
    for b in range(50):
        assert (vi[b, :vn[b]] == ref["vis_ids"][b, :vn[b]]).all()
        assert vd[b, :vn[b]].tobytes() == ref["vis_dists"][b, :vn[b]].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", [(768, "cosine"), (4096, "euclidean")])
def test_search_filters_wide(dim, metric):
    """FILTER variant: filtered and unfiltered requests in one batch, each equal to the oracle's
    answer for that request alone."""
    oix, g, X, Q, pid = _graph(dim, metric)
    rng = np.random.Generator(np.random.PCG64(dim))
    filters = [np.sort(rng.choice(pid, size=nf, replace=False)) for nf in (1, 40, 75, 76, 500)]
    B = 48
    qf = np.array([(b % (len(filters) + 1)) - 1 for b in range(B)], dtype=np.int32)  # -1 = unfiltered
    ids, d, cnt = g.search_batch_filters(Q[:B], filters, qf, 10, 75)
    plain = oix.search(Q[:B], k=10, threads=8)
    for b in range(B):
        if qf[b] < 0:
            ref = {key: v[b] for key, v in plain.items()}
        else:
            r = oix.search(Q[b:b + 1], k=10, filter_ids=filters[qf[b]], threads=1)
            ref = {key: v[0] for key, v in r.items()}
        assert cnt[b] == ref["counts"], b
        assert (ids[b] == ref["ids"].astype(np.uint64)).all(), b
        assert d[b].tobytes() == ref["dists"].tobytes(), b
    _check_f64_rows(metric, Q[:B], X, ids, d, cnt)


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", [(768, "euclidean"), (4096, "dot")])
def test_search_visited_wide(dim, metric):
    """greedySearch's visited list (the robustPrune candidates of the insert path)."""
    oix, g, X, Q, _ = _graph(dim, metric)
    ref = oix.search(Q[:100], k=1, vis_cap=256, threads=8)
    vi, vd, vn = g.search_visited(Q[:100], 75, 256)
    assert (vn == ref["vis_len"]).all()
    for b in range(100):
        n = vn[b]
        assert (vi[b, :n] == ref["vis_ids"][b, :n]).all()
        assert vd[b, :n].tobytes() == ref["vis_dists"][b, :n].tobytes()


# ---------------------------------------------------------------- batched insert (K8)

@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric,n", [(256, "euclidean", 1000), (768, "cosine", 800), (1536, "dot", 500),
                                          (4096, "euclidean", 300)])
def test_sequential_insert_wide_rows(dim, metric, n):
    """One point per mini-batch (the reference's sequential schedule) reproduces the oracle's graph
    edge for edge while robustPrune stages only part of each candidate list in shared memory;
    the store's distance closures equal the oracle's bit for bit."""
    X = _data(n, dim, dim + 5, metric)
    oix, ids, start = oracle_graph(X, metric, threads=1)
    g = IndexVamana("wide", IndexVectorVamanaParameters(dim, metric), start_vector=start)
    g.insert_config(1, 1, 16)
    g.insert_batch(ids.astype(np.uint64), X)
    check_graph_equal(oix, g, n)
    q = _data(1, dim, dim + 6, metric, w_seed=dim + 5)[0]
    assert g.query_dists(q, ids.astype(np.uint64)).tobytes() == oix.query_dists(q, ids).tobytes()
    want = np.array([oix.point_dist(7, int(i)) for i in ids[:200]], dtype=np.float32)
    assert g.point_dists(7, ids[:200].astype(np.uint64)).tobytes() == want.tobytes()


# ---------------------------------------------------------------- flat exact scan (K5)

@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric", [(400, "euclidean"), (410, "dot"), (3600, "cosine"), (3700, "euclidean"),
                                        (4096, "dot")])
def test_flat_exact_scan_wide(dim, metric):
    """Fewer than 4 096 points, so the exact scan serves every call. Dims on both sides of each
    shared-memory switch: query tile in shared memory (400) or streamed (410); 16-row point tile
    (3 600) or fewer rows (3 700, 4 096)."""
    n = 3000
    X = _data(n, dim, dim, metric)
    Q = _data(40, dim, dim + 1, metric, w_seed=dim)
    X[2000:2050] = X[:50]  # exact duplicates: ties by ascending id
    ids = np.arange(2, n + 2, dtype=np.uint32)
    oix = O.OracleIndex(dim, metric)
    oix.set_vectors(ids, X)
    g = IndexFlat(IndexVectorFlatParameters(dim, metric))
    g.set_vectors(ids.astype(np.uint64), X)
    gt = oix.flat_search(Q, k=75, threads=8)
    for k in (1, 10, 75):
        fi, fd, fc = g.flat_search_batch(Q, k)
        assert g.flat_last_stats()[0] == 0
        assert (fc == gt["counts"].clip(max=k)).all()
        assert (fi == gt["ids"][:, :k].astype(np.uint64)).all() and fd.tobytes() == gt["dists"][:, :k].tobytes()
    _check_f64_flat(metric, Q, X, fi, fd, fc, 75)
    filt = np.sort(np.random.Generator(np.random.PCG64(dim)).choice(ids, size=400, replace=False))
    fi, fd, fc = g.flat_search_batch(X[:40], 10, filter_ids=filt)
    ref = oix.flat_search(X[:40], k=10, filter_ids=filt, threads=8)
    assert (fc == ref["counts"]).all()
    assert (fi == ref["ids"].astype(np.uint64)).all() and fd.tobytes() == ref["dists"].tobytes()


# ---------------------------------------------------------------- flat tensor-core path (K5)

def _flat_tc_store(dim, metric, n=20_000, B=None):
    X = _data(n, dim, dim, metric)
    X[10_000:10_100] = X[:100]  # exact duplicates: ties by ascending id
    B = B or (200 if dim <= 768 else 64)
    Q = _data(B, dim, dim + 1, metric, w_seed=dim)
    Q[:8] = X[:8]  # queries that are stored (duplicated) points
    return X, Q


def _flat_tc_search(g, Q, k, monkeypatch):
    """Tensor-core path and the exact scan (SDB_FLAT_EXACT=1): returns both results and the stats."""
    monkeypatch.delenv("SDB_FLAT_EXACT", raising=False)
    a = g.flat_search_batch(Q, k)
    stats = g.flat_last_stats()
    monkeypatch.setenv("SDB_FLAT_EXACT", "1")
    b = g.flat_search_batch(Q, k)
    assert g.flat_last_stats()[0] == 0
    monkeypatch.delenv("SDB_FLAT_EXACT")
    return a, b, stats


@pytest.mark.gpu
@pytest.mark.parametrize("dim,metric,path", [
    (320, "euclidean", 2), (384, "dot", 2),
    (385, "euclidean", 1), (385, "dot", 1), (385, "cosine", 1),
    (768, "euclidean", 1), (768, "dot", 1), (768, "cosine", 1),
    (1000, "dot", 1), (1536, "cosine", 1), (3072, "euclidean", 1), (3073, "dot", 1), (4096, "cosine", 1)])
def test_flat_tc_wide(dim, metric, path, monkeypatch):
    """tcgen05 up to a padded dim of 384, the mma.sync level scheme above (kp 448 from dim 385):
    no overflow into the exact scan, at least k candidates per query, lists equal to the oracle's
    and to the exact scan's bit for bit, distances within the f32 bound of float64."""
    X, Q = _flat_tc_store(dim, metric)
    n = len(X)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    g = IndexFlat(IndexVectorFlatParameters(dim, metric))
    g.set_vectors(ids.astype(np.uint64), X)
    oix = O.OracleIndex(dim, metric)
    oix.set_vectors(ids, X)
    gt = oix.flat_search(Q, k=75, threads=8)
    for k in (1, 10, 75):
        (ti, td, tc), (ei, ed, ec), (p, cand, ovf) = _flat_tc_search(g, Q, k, monkeypatch)
        assert p == path and ovf == 0 and cand >= k * len(Q), (k, p, cand, ovf)
        assert (tc == k).all() and (ec == k).all()
        assert (ti == gt["ids"][:, :k].astype(np.uint64)).all() and td.tobytes() == gt["dists"][:, :k].tobytes(), k
        assert (ti == ei).all() and td.tobytes() == ed.tobytes(), k
    _check_f64_flat(metric, Q, X, ti, td, tc, 75)
    if metric == "euclidean":  # a stored point is its own nearest, then its duplicate
        assert (ti[:8, 0] == ids[:8]).all() and (ti[:8, 1] == ids[10_000:10_008]).all() and (td[:8, :2] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["euclidean", "dot"])
@pytest.mark.parametrize("dim,path", [(384, 2), (768, 1)])
def test_flat_tc_power_of_two_scaling(dim, path, metric, monkeypatch):
    """f32 arithmetic is exact under power-of-two scaling while nothing under- or overflows, so
    scaling store and queries by 2^s must keep every id and scale every distance by exactly 4^s,
    at the scale edges of the candidate bound too."""
    X, Q = _flat_tc_store(dim, metric, B=100)
    ids = np.arange(2, len(X) + 2, dtype=np.uint64)
    base = {}
    for s in (0, -30, 30):
        f = np.float32(2.0 ** s)
        g = IndexFlat(IndexVectorFlatParameters(dim, metric))
        g.set_vectors(ids, X * f)
        for k in (10, 75):
            (ti, td, tc), (ei, ed, ec), (p, cand, ovf) = _flat_tc_search(g, Q * f, k, monkeypatch)
            assert p == path and ovf == 0 and cand >= k * len(Q), (s, k, p, cand, ovf)
            assert (ti == ei).all() and td.tobytes() == ed.tobytes(), (s, k)
            if s == 0:
                base[k] = (ti, td)
            else:
                assert (ti == base[k][0]).all(), (s, k)
                assert td.tobytes() == (base[k][1] * np.float32(4.0 ** s)).tobytes(), (s, k)


@pytest.mark.gpu
@pytest.mark.parametrize("dim,path", [(384, 2), (768, 1)])
def test_flat_tc_common_offset(dim, path, monkeypatch):
    """Squared L2 over a store far from the origin (X + 1000): centring keeps the bf16 bound tight,
    so nothing overflows into the exact scan and the lists are the exact scan's and the oracle's."""
    X, Q = _flat_tc_store(dim, "euclidean", B=100)
    X, Q = X + np.float32(1000), Q + np.float32(1000)
    ids = np.arange(2, len(X) + 2, dtype=np.uint32)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(ids.astype(np.uint64), X)
    oix = O.OracleIndex(dim, "euclidean")
    oix.set_vectors(ids, X)
    gt = oix.flat_search(Q, k=75, threads=8)
    for k in (10, 75):
        (ti, td, tc), (ei, ed, ec), (p, cand, ovf) = _flat_tc_search(g, Q, k, monkeypatch)
        assert p == path and ovf == 0 and cand >= k * len(Q), (k, p, cand, ovf)
        assert (ti == ei).all() and td.tobytes() == ed.tobytes(), k
        assert (ti == gt["ids"][:, :k].astype(np.uint64)).all() and td.tobytes() == gt["dists"][:, :k].tobytes(), k
    _check_f64_flat("euclidean", Q, X, ti, td, tc, 75)


# ---------------------------------------------------------------- PQ evaluators

@pytest.mark.gpu
@pytest.mark.parametrize("metric,dim,M,K", [
    ("euclidean", 64, 16, 64),  # sub-vectors of 4 floats: AdcEvalFly<., 4>
    ("dot", 128, 8, 64),  # sub-vectors of 16 floats: AdcEvalFly<., 16>
    ("euclidean", 96, 6, 32),  # M % 4 != 0: the per-query table in shared memory
    ("cosine", 1024, 256, 16),  # 256 sub-vectors: the table loop of AdcEvalSmem::chains runs twice
])
def test_pq_evaluators(metric, dim, M, K, monkeypatch):
    """The flow of the reference: raw inserts until the trigger, Fit (centroids, centroidDists,
    codes, written-through rows and ADC tables equal to the oracle's), then ADC search and SDC
    prune: the graph edge for edge, searches with ids, distances, hops and evaluations equal,
    and one batch of per-request filters."""
    n, n0 = 2000, 1400
    X = _data(n, dim, dim + 11, metric)
    Q = _data(100, dim, dim + 12, metric, w_seed=dim + 11)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    oix = O.OracleIndex(dim, metric, quantizer="product", pq_m=M, pq_k=K, pq_trigger=1000)
    start = synth.start_vector(dim, 5)
    oix.set_start(start)
    g = IndexVamana("pq", IndexVectorVamanaParameters(dim, metric, quantizer=Quantizer(
        "product", product=ProductQuantizerParameters(K, M, 1000))), start_vector=start)
    g.insert_config(1, 1, 16)
    oix.insert(ids[:n0], X[:n0], threads=1)
    g.insert_batch(ids[:n0].astype(np.uint64), X[:n0])
    assert oix.fit(pq_first=3, pq_alias=True, threads=8) == 1
    assert g.fit(3) is True
    ofc, ocd = oix.get_pq()
    gfc, gcd = g.get_pq()
    assert gfc.tobytes() == ofc.tobytes() and gcd.tobytes() == ocd.tobytes()
    all_ids = np.concatenate([[1], ids[:n0]]).astype(np.uint32)
    assert g.get_codes(all_ids.astype(np.uint64)).tobytes() == oix.get_codes(all_ids).tobytes()
    assert g.get_vectors(all_ids.astype(np.uint64)).tobytes() == oix.get_vectors(all_ids).tobytes()
    tabs = g.adc_tables(Q[:4])
    for b in range(4):
        assert tabs[b].tobytes() == oix.adc_table(Q[b]).tobytes()
    oix.insert(ids[n0:], X[n0:], threads=1)
    g.insert_batch(ids[n0:].astype(np.uint64), X[n0:])
    check_graph_equal(oix, g, n)
    check_search(oix, g, Q)
    check_search(oix, g, Q[:50], k=75, L=75)
    rng = np.random.Generator(np.random.PCG64(M))
    filters = [np.sort(rng.choice(ids, size=nf, replace=False)) for nf in (40, 76, 500)]
    qf = np.array([(b % (len(filters) + 1)) - 1 for b in range(48)], dtype=np.int32)
    fi, fd, fc = g.search_batch_filters(Q[:48], filters, qf, 10, 75)
    plain = oix.search(Q[:48], k=10, threads=8)
    for b in range(48):
        if qf[b] < 0:
            ref = {key: v[b] for key, v in plain.items()}
        else:
            r = oix.search(Q[b:b + 1], k=10, filter_ids=filters[qf[b]], threads=1)
            ref = {key: v[0] for key, v in r.items()}
        assert fc[b] == ref["counts"], b
        assert (fi[b] == ref["ids"].astype(np.uint64)).all() and fd[b].tobytes() == ref["dists"].tobytes(), b
    monkeypatch.setenv("SDB_ADC_GLOBAL", "1")  # the table through L1/L2: the same answers
    check_search(oix, g, Q)
