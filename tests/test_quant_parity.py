"""K2/K3/K4/K7/K9 parity: binary and product quantizers on the GPU vs the oracle.
Integer/byte results (thresholded bits, PQ codes, hamming/jaccard distances, ids) are
bit-exact; f32 values (thresholds, centroids, tables, distances) are bit-identical too
because the kernels keep the reference's summation order."""
import numpy as np
import pytest

from oracle import oraclelib as O
from semadb_b200 import synth
from semadb_b200.vamana import (BinaryQuantizerParameters, IndexVamana, IndexVectorVamanaParameters,
                                ProductQuantizerParameters, Quantizer)
from tests.helpers import check_graph_equal as _check_graph_equal
from tests.helpers import check_search as _check_search

pytestmark = pytest.mark.gpu


def _same(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


def _mirror(oix, X, ids, start, params, relaxed=True):
    g = IndexVamana("q", params, start_vector=start, relaxed=relaxed)
    g.set_vectors(ids.astype(np.uint64), X)
    adj, deg = oix.get_graph()
    g.set_graph_dense(adj[1:], deg[1:], first_id=1)
    return g


@pytest.mark.parametrize("metric", ["hamming", "jaccard"])
@pytest.mark.parametrize("dim", [1024, 100, 64, 2048, 4000, 256, 768])
def test_bit_metric_search_matches_oracle(metric, dim):
    """C5b-shaped: 0/1 floats, binary store forced on with threshold 0.5 (vectorstore.go:56-66);
    integer distances make boundary ties ubiquitous (SURVEY.md §7.3-②)."""
    n = 6000
    X = synth.planted_bits(n, dim, seed=7, n_proto=64)
    Q = synth.planted_bits(200, dim, seed=10, n_proto=64, proto_seed=7)
    oix = O.OracleIndex(dim, metric)
    start = synth.start_vector(dim, 5)
    oix.set_start(start)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    oix.insert(ids, X, threads=1)
    g = _mirror(oix, X, ids, start, IndexVectorVamanaParameters(dim, metric))
    assert _same(g.get_codes(ids[:50].astype(np.uint64)), oix.get_codes(ids[:50]))
    _check_search(oix, g, Q)
    # flat scan over the same store
    gt = oix.flat_search(Q[:50], k=10, threads=4)
    fi, fd, fc = g.flat_search_batch(Q[:50], 10)
    assert (fi == gt["ids"].astype(np.uint64)).all() and _same(fd, gt["dists"])
    # store-level closures
    assert _same(g.query_dists(Q[0], ids[:100].astype(np.uint64)), oix.query_dists(Q[0], ids[:100]))
    assert _same(g.point_dists(2, ids[:100].astype(np.uint64)),
                 np.array([oix.point_dist(2, int(i)) for i in ids[:100]], dtype=np.float32))


def test_bit_metric_sequential_insert_reproduces_oracle_graph():
    n, dim = 1200, 256
    X = synth.planted_bits(n, dim, seed=7, n_proto=32)
    oix = O.OracleIndex(dim, "hamming")
    start = synth.start_vector(dim, 5)
    oix.set_start(start)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    oix.insert(ids, X, threads=1)
    g = IndexVamana("h", IndexVectorVamanaParameters(dim, "hamming"), start_vector=start)
    g.insert_config(1, 1, 16)
    g.insert_batch(ids.astype(np.uint64), X)
    _check_graph_equal(oix, g, n)


def test_binary_quantizer_fit_and_search():
    """binaryQuantizer.Fit (binary.go:145-185): threshold = per-dimension mean once
    Count() >= TriggerThreshold; until then distances use the raw floats."""
    n, dim = 3000, 96
    X = synth.latent_gaussian(n, dim, seed=21, latent=8)
    Q = synth.latent_gaussian(100, dim, seed=22, w_seed=21, latent=8)
    oix = O.OracleIndex(dim, "euclidean", quantizer="binary", bq_metric="hamming", bq_trigger=2000)
    start = synth.start_vector(dim, 5)
    oix.set_start(start)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    params = IndexVectorVamanaParameters(dim, "euclidean", quantizer=Quantizer(
        "binary", binary=BinaryQuantizerParameters(None, 2000, "hamming")))
    g = IndexVamana("bq", params, start_vector=start)
    g.insert_config(1, 1, 16)
    # first batch: below the trigger => float distances, no fit
    oix.insert(ids[:1500], X[:1500], threads=1)
    assert oix.fit() == 0
    g.insert_batch(ids[:1500].astype(np.uint64), X[:1500])
    assert g.fit() is False
    _check_search(oix, g, Q)
    # second batch crosses the trigger => fit, re-encode
    oix.insert(ids[1500:2500], X[1500:2500], threads=1)
    assert oix.fit() == 1
    g.insert_batch(ids[1500:2500].astype(np.uint64), X[1500:2500])
    assert g.fit() is True
    assert _same(g.get_bq_threshold(), oix.get_bq_threshold())
    assert _same(g.get_codes(ids[:2500].astype(np.uint64)), oix.get_codes(ids[:2500]))
    _check_search(oix, g, Q)
    # third batch inserts through hamming search + prune
    oix.insert(ids[2500:], X[2500:], threads=1)
    g.insert_batch(ids[2500:].astype(np.uint64), X[2500:])
    _check_graph_equal(oix, g, n)
    _check_search(oix, g, Q)


@pytest.mark.parametrize("metric,M,K,dim", [("euclidean", 8, 32, 64), ("dot", 12, 256, 96), ("cosine", 4, 16, 128)])
def test_product_quantizer_fit_matches_oracle(metric, M, K, dim):
    """productQuantizer.Fit (product.go:175-236) + utils.KMeans.Fit (kmeans.go:34-150),
    aliasing quirk included: centroids, codes, centroidDists and the written-through rows."""
    n = 1200
    X = synth.latent_gaussian(n, dim, seed=31, latent=8, normalize=(metric == "cosine"))
    ids = np.arange(2, n + 2, dtype=np.uint32)
    oix = O.OracleIndex(dim, metric, quantizer="product", pq_m=M, pq_k=K, pq_trigger=1000)
    start = synth.start_vector(dim, 5)
    oix.set_start(start)
    oix.set_vectors(ids, X)
    params = IndexVectorVamanaParameters(dim, metric, quantizer=Quantizer(
        "product", product=ProductQuantizerParameters(K, M, 1000)))
    g = IndexVamana("pq", params, start_vector=start)
    g.set_vectors(ids.astype(np.uint64), X)
    assert oix.fit(pq_first=7, pq_alias=True, threads=8) == 1
    assert g.fit(pq_first_row=7) is True
    ofc, ocd = oix.get_pq()
    gfc, gcd = g.get_pq()
    assert _same(gfc, ofc)
    assert _same(gcd, ocd)
    all_ids = np.concatenate([[1], ids]).astype(np.uint32)
    assert _same(g.get_codes(all_ids.astype(np.uint64)), oix.get_codes(all_ids))
    assert _same(g.get_vectors(all_ids.astype(np.uint64)), oix.get_vectors(all_ids))  # kmeans.go:144 write-through
    # K4: ADC tables (product.go:255-263)
    Q = synth.latent_gaussian(16, dim, seed=32, w_seed=31, latent=8, normalize=(metric == "cosine"))
    tabs = g.adc_tables(Q)
    for b in range(len(Q)):
        assert _same(tabs[b], oix.adc_table(Q[b]))
    assert _same(g.query_dists(Q[0], ids[:200].astype(np.uint64)), oix.query_dists(Q[0], ids[:200]))
    assert _same(g.point_dists(5, ids[:200].astype(np.uint64)),
                 np.array([oix.point_dist(5, int(i)) for i in ids[:200]], dtype=np.float32))
    # points set after the fit are encoded with the index metric (product.go:136-159)
    X2 = synth.latent_gaussian(64, dim, seed=33, w_seed=31, latent=8, normalize=(metric == "cosine"))
    ids2 = np.arange(n + 2, n + 66, dtype=np.uint32)
    oix.set_vectors(ids2, X2)
    g.set_vectors(ids2.astype(np.uint64), X2)
    assert _same(g.get_codes(ids2.astype(np.uint64)), oix.get_codes(ids2))


def test_product_quantizer_insert_and_search():
    """Reference flow: insert with raw floats until the trigger, Fit, then ADC search
    (product.go:238-277) and SDC prune (product.go:279-305) for later inserts."""
    n, dim, M, K = 2400, 64, 8, 64
    X = synth.latent_gaussian(n, dim, seed=41, latent=8)
    Q = synth.latent_gaussian(100, dim, seed=42, w_seed=41, latent=8)
    oix = O.OracleIndex(dim, "euclidean", quantizer="product", pq_m=M, pq_k=K, pq_trigger=1000)
    start = synth.start_vector(dim, 5)
    oix.set_start(start)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    params = IndexVectorVamanaParameters(dim, "euclidean", quantizer=Quantizer(
        "product", product=ProductQuantizerParameters(K, M, 1000)))
    g = IndexVamana("pq", params, start_vector=start)
    g.insert_config(1, 1, 16)
    oix.insert(ids[:1600], X[:1600], threads=1)
    assert oix.fit(pq_first=0, pq_alias=True, threads=8) == 1
    g.insert_batch(ids[:1600].astype(np.uint64), X[:1600])
    assert g.fit(0) is True
    _check_search(oix, g, Q)
    oix.insert(ids[1600:], X[1600:], threads=1)
    g.insert_batch(ids[1600:].astype(np.uint64), X[1600:])
    _check_graph_equal(oix, g, n)
    _check_search(oix, g, Q)
    gt = oix.flat_search(Q[:20], k=10, threads=4)
    fi, fd, fc = g.flat_search_batch(Q[:20], 10)
    assert (fi == gt["ids"].astype(np.uint64)).all() and _same(fd, gt["dists"])


def test_c4_shape_fit_tables_and_search(monkeypatch):
    """The C4 shape of BASELINE.json — 768-d dot product, PQ with 96 sub-vectors of 8 floats and
    256 centroids — against the oracle: k-means centroids, centroidDists, codes and the
    written-through rows (product.go:175-236, kmeans.go:34-150), the per-query ADC tables
    (product.go:255-263), and the search itself (product.go:238-277) by each of the three PQ
    evaluators: entries computed on the fly from the codebook (default), table in shared memory,
    table through L1/L2 — ids, distances, hop and evaluation counts all equal."""
    n, dim, M, K = 3000, 768, 96, 256
    X = synth.latent_gaussian(n, dim, seed=8, latent=16, normalize=True)
    Q = synth.latent_gaussian(64, dim, seed=9, w_seed=8, latent=16, normalize=True)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    oix = O.OracleIndex(dim, "dot", quantizer="product", pq_m=M, pq_k=K, pq_trigger=1000)
    start = synth.start_vector(dim, 5)
    oix.set_start(start)
    params = IndexVectorVamanaParameters(dim, "dot", quantizer=Quantizer(
        "product", product=ProductQuantizerParameters(K, M, 1000)))
    g = IndexVamana("c4", params, start_vector=start)
    g.insert_config(1, 1, 16)  # the reference's sequential schedule: the graph must come out edge for edge
    oix.insert(ids[:2000], X[:2000], threads=1)
    g.insert_batch(ids[:2000].astype(np.uint64), X[:2000])
    assert oix.fit(pq_first=3, pq_alias=True, threads=8) == 1
    assert g.fit(3) is True
    ofc, ocd = oix.get_pq()
    gfc, gcd = g.get_pq()
    assert _same(gfc, ofc) and _same(gcd, ocd)
    all_ids = np.concatenate([[1], ids[:2000]]).astype(np.uint32)
    assert _same(g.get_codes(all_ids.astype(np.uint64)), oix.get_codes(all_ids))
    assert _same(g.get_vectors(all_ids.astype(np.uint64)), oix.get_vectors(all_ids))
    tabs = g.adc_tables(Q[:4])
    for b in range(4):
        assert _same(tabs[b], oix.adc_table(Q[b]))
    oix.insert(ids[2000:], X[2000:], threads=1)  # ADC search + SDC prune
    g.insert_batch(ids[2000:].astype(np.uint64), X[2000:])
    _check_graph_equal(oix, g, n)
    _check_search(oix, g, Q)  # on the fly
    monkeypatch.setenv("SDB_ADC_TABLE", "1")
    _check_search(oix, g, Q)  # table in shared memory
    monkeypatch.setenv("SDB_ADC_GLOBAL", "1")
    _check_search(oix, g, Q)  # table through L1/L2
