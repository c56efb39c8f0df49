"""Pins the CPU oracle against every exact known-answer test and property test the
reference holds for the hot path (SURVEY.md §8c). Runs on CPU."""
import numpy as np
import pytest

from oracle import oraclelib as O

# distance/distance_test.go:9-21
VECTOR_TABLE = [
    ("Zero", [0, 0, 0], [0, 0, 0], 0, 0),
    ("One", [1, 1], [1, 1], 2, 0),
    ("Two", [1, 2, 3], [4, 5, 6], 32, 27),
    ("Negative", [-1, -2, -3], [-4, -5, -6], 32, 27),
    ("Mixed", [-1, 2, 3], [4, -5, 6], 4, 83),
]


@pytest.mark.parametrize("name,x,y,want_dot,want_l2", VECTOR_TABLE)
@pytest.mark.parametrize("impl", ["pure", "raw", "model"])
def test_distance_table(name, x, y, want_dot, want_l2, impl):
    # distance_test.go:23-39 (pure) and distance_amd64_test.go:12-28 (asm): require.Equal
    assert O.float_dist("dot", x, y, impl) == np.float32(want_dot)
    assert O.float_dist("euclidean", x, y, impl) == np.float32(want_l2)


def test_metric_wrappers():
    # distance.go:19-25: dot distance = -dot, cosine = 1 - dot (no normalisation)
    x, y = [1, 2, 3], [4, 5, 6]
    assert O.float_dist("dot", x, y) == np.float32(-32)
    assert O.float_dist("cosine", x, y) == np.float32(1 - 32)
    assert O.float_dist("euclidean", x, y) == np.float32(27)


def test_hamming_jaccard_kat():
    # distance_test.go:41-57
    x = [0b1001, 0b1]
    y = [0b1101, 0b0]
    assert O.bit_dist("hamming", x, y) == 2.0
    assert O.bit_dist("jaccard", x, y) == 0.5
    assert O.bit_dist("jaccard", [0, 0], [0, 0]) == 0.0


def test_haversine_kat():
    # distance_test.go:59-67
    d = O.float_dist("haversine", [-34.83333, -58.5166646], [49.0083899664, 2.53844117956]) / 1000
    assert abs(d - 11099.54) < 0.01


@pytest.mark.parametrize("n", [1, 2, 7, 8, 31, 32, 33, 63, 64, 100, 128, 129, 384, 768, 1000, 1536, 4096])
def test_avx_equals_order_model(n):
    # SURVEY.md §7.3-①: the scalar order model (what the CUDA kernels implement) must be
    # bit-identical to the AVX2/FMA restatement of dot.s / euclidean.s.
    rng = np.random.Generator(np.random.PCG64(n))
    for _ in range(20):
        x = rng.standard_normal(n).astype(np.float32)
        y = rng.standard_normal(n).astype(np.float32)
        for m in ("euclidean", "dot"):
            a = np.float32(O.float_dist(m, x, y, "raw"))
            b = np.float32(O.float_dist(m, x, y, "model"))
            assert a.tobytes() == b.tobytes()


def test_binary_encode_kat():
    # binary_test.go:11-23
    enc = O.bq_encode([1.0, 0.1, 0.6, 0.7, 0.4], [0.5] * 5)
    assert len(enc) == 1 and int(enc[0]) == 0b01101


def test_binary_encode_word_boundaries():
    v = np.zeros(130, dtype=np.float32)
    v[[0, 63, 64, 129]] = 1.0
    enc = O.bq_encode(v, np.full(130, 0.5, np.float32))
    assert len(enc) == 3
    assert int(enc[0]) == (1 | (1 << 63)) and int(enc[1]) == 1 and int(enc[2]) == 2
    # strictly greater (binary.go:124)
    assert int(O.bq_encode([0.5], [0.5])[0]) == 0


def test_binary_fit_kat():
    # binary_test.go:25-39
    thr = O.bq_fit_threshold(np.array([[1.0, 2.0], [3.0, 4.0]], dtype=np.float32))
    assert thr.tolist() == [2.0, 3.0]
    ix = O.OracleIndex(2, "euclidean", quantizer="binary", bq_trigger=2)
    ix.set_vectors([2, 3], [[1.0, 2.0], [3.0, 4.0]])
    assert ix.fit() == 1
    assert ix.get_bq_threshold().tolist() == [2.0, 3.0]


# ---- distset_test.go:41-74 ------------------------------------------------

def test_distset_add():
    ds = O.DistSet(2, [0.5, 1.0, 0.2])
    ds.add(0, 1, 2)
    assert ds.items()[0] == [0, 1, 2]
    ds.sort()
    assert ds.items()[0] == [2, 0, 1]


def test_distset_add_dedupe():
    ds = O.DistSet(2, [0.5, 1.0, 0.2])
    ds.add(0, 1, 2, 0)
    assert ds.items()[0] == [0, 1, 2]
    ds.sort()
    assert ds.items()[0] == [2, 0, 1]


def test_distset_add_duplicate():
    ds = O.DistSet(3, [0.5, 1.0, 0.1])
    ds.add(0, 1, 2)
    ds.add(0)
    assert len(ds.items()[0]) == 3
    ds.sort()
    assert ds.items()[0] == [2, 0, 1]


def test_distset_add_with_limit():
    ds = O.DistSet(2, [0.5, 1.0, 0.1, 1.2])
    ds.add_with_limit(0, 1, 2)
    assert ds.items()[0] == [2, 0]
    ds.add_with_limit(3, 3)
    assert ds.items()[0] == [2, 0]


def test_distset_boundary_tie_newest_wins():
    # distset.go:184 rejects only d > worst; an equal newcomer overwrites the last slot.
    ds = O.DistSet(2, [0.1, 0.5, 0.5, 0.5])
    ds.add_with_limit(0, 1, 2)
    assert ds.items()[0] == [0, 2]
    ds.add_with_limit(3)
    assert ds.items()[0] == [0, 3]


# ---- vamana_test.go property tests ---------------------------------------

def _rand_index(n, dim=2, seed=0, threads=1, **kw):
    rng = np.random.Generator(np.random.PCG64(seed))
    ix = O.OracleIndex(dim, kw.pop("metric", "euclidean"), 75, 64, 1.2, **kw)
    ix.set_start(O.random_unit_vector(dim, seed + 1000))
    vecs = rng.random((n, dim), dtype=np.float32)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    ix.insert(ids, vecs, threads=threads)
    return ix, ids, vecs


def _bfs_reach(adj, deg, start=1):
    seen = {start}
    q = [start]
    while q:
        u = q.pop()
        for v in adj[u, :deg[u]]:
            v = int(v)
            if v not in seen:
                seen.add(v)
                q.append(v)
    return seen


@pytest.mark.parametrize("n", [1, 100, 4242])
@pytest.mark.parametrize("threads", [1, 4])
def test_insert_connectivity(n, threads):
    # vamana_test.go:29-46,63-75: BFS from the start node reaches every point
    ix, ids, _ = _rand_index(n, threads=threads)
    adj, deg = ix.get_graph()
    assert deg.max() <= 64
    seen = _bfs_reach(adj, deg)
    assert len(seen) == n + 1
    # no self edges, no duplicates
    for u in range(1, n + 2):
        row = adj[u, :deg[u]].tolist()
        assert u not in row and len(set(row)) == len(row)


def test_insert_rejects_reserved_ids():
    # vamana_test.go:77-90
    ix = O.OracleIndex(2)
    ix.set_start(O.random_unit_vector(2, 1))
    for bad in (0, 1):
        with pytest.raises(RuntimeError):
            ix.insert([bad], [[0.1, 0.2]])


def test_search_empty():
    # vamana_test.go:213-228
    ix = O.OracleIndex(2)
    ix.set_start(O.random_unit_vector(2, 1))
    r = ix.search([[0.5, 0.5]], k=10)
    assert r["counts"][0] == 0


def test_search_self_recall():
    # vamana_test.go:230-252: 200 random 2-d points, each queried; top-1 is itself, 10 results
    ix, ids, vecs = _rand_index(200, seed=3)
    r = ix.search(vecs, k=10)
    assert (r["counts"] == 10).all()
    assert (r["ids"][:, 0] == ids).all()
    assert (r["dists"][:, 0] == 0).all()


def test_search_size_lt_k_is_error():
    # search.go:23-25
    ix, _, vecs = _rand_index(50)
    with pytest.raises(ValueError):
        ix.search(vecs[:1], k=30, search_size=25)


def test_search_filter():
    # vamana_test.go:254-276: filter search returns exactly the filtered ids, self first
    ix, ids, vecs = _rand_index(200, seed=5)
    filt = [ids[10], ids[20], ids[30]]
    r = ix.search(vecs[10:11], k=10, filter_ids=filt)
    assert r["counts"][0] == 3
    assert r["ids"][0, 0] == ids[10]
    assert sorted(r["ids"][0, :3].tolist()) == sorted(int(x) for x in filt)


def test_search_counters_and_lists():
    ix, ids, vecs = _rand_index(3000, dim=8, seed=7)
    r = ix.search(vecs[:50], k=10, diagnostics=True, vis_cap=256)
    assert (r["hops"] >= 75).all() and (r["hops"] < 200).all()
    assert (r["ndist"] >= r["hops"]).all()
    assert (r["list_len"] == 75).all()
    d = r["list_dists"]
    assert (np.diff(d, axis=1) >= 0).all()
    assert (r["vis_len"] == r["hops"]).all()
    for b in range(50):
        n = r["vis_len"][b]
        assert (np.diff(r["vis_dists"][b, :n]) >= 0).all()


# ---- vectorestore_test.go:112-154 ----------------------------------------

# triggerFit fixture (vectorestore_test.go:37-50)
FIT_IDS = [1, 2, 3, 4, 5]
FIT_VECS = np.array([[1, 2, 3, 4], [4, 5, 6, 7], [7, 8, 9, 10], [-10, -11, -12, -13], [-13, 14, -15, 16]],
                    dtype=np.float32)


@pytest.mark.parametrize("quant,kw", [("none", {}), ("binary", dict(bq_trigger=5)),
                                       ("product", dict(pq_m=2, pq_k=256, pq_trigger=5))])
@pytest.mark.parametrize("fitted", [False, True])
def test_vectorstore_distance_contract(quant, kw, fitted):
    # Test_DistanceFromFloat / Test_DistanceFromPoint (vectorestore_test.go:112-154)
    ix = O.OracleIndex(4, "euclidean", quantizer=quant, **kw)
    if fitted:
        ix.set_vectors(FIT_IDS, FIT_VECS)
        assert ix.fit() == (0 if quant == "none" else 1)
    ix.set_vectors([7, 8], [[1, 2, 3, 4], [4, 5, 6, 7]])
    d = ix.query_dists([1, 2, 3, 4], [7, 8])
    assert d[0] == 0
    assert d[0] < d[1]
    assert ix.point_dist(7, 7) == 0
    assert ix.point_dist(7, 7) < ix.point_dist(7, 8)


# ---- flat_test.go:134-191 -------------------------------------------------

@pytest.mark.parametrize("metric", ["euclidean", "cosine", "dot"])
def test_flat_matches_bruteforce(metric):
    rng = np.random.Generator(np.random.PCG64(11))
    X = rng.random((2000, 2), dtype=np.float32)
    ix = O.OracleIndex(2, metric)
    ids = np.arange(2, 2002, dtype=np.uint32)
    ix.set_vectors(ids, X)
    Q = X[:20]
    r = ix.flat_search(Q, k=10)
    for b in range(20):
        all_d = np.array([O.float_dist(metric, Q[b], X[j]) for j in range(2000)], dtype=np.float32)
        order = np.lexsort((ids, all_d))[:10]
        assert r["dists"][b].tolist() == all_d[order].tolist()
        assert r["ids"][b].tolist() == ids[order].tolist()


# ---- kmeans_test.go -------------------------------------------------------

def test_kmeans_pairs():
    # kmeans_test.go:15-68: three well separated pairs; pair-mates share labels
    rng = np.random.Generator(np.random.PCG64(2))
    base = np.array([[0, 0], [0, 0], [10, 10], [10, 10], [-10, -10], [-10, -10]], dtype=np.float32)
    for offset in (0, 2):
        X = np.zeros((6, 4), dtype=np.float32)
        X[:, offset:offset + 2] = base + rng.random((6, 2), dtype=np.float32)
        for alias in (False, True):
            _, labels, _, _ = O.kmeans_fit(X.copy(), 3, 100, offset, 2, first=0, alias=alias)
            assert labels[0] == labels[1] and labels[2] == labels[3] and labels[4] == labels[5]
            assert len({labels[0], labels[2], labels[4]}) == 3


def test_kmeans_256():
    # kmeans_test.go:70-91
    rng = np.random.Generator(np.random.PCG64(4))
    X = rng.random((10000, 16), dtype=np.float32)
    cent, labels, iters, rows = O.kmeans_fit(X, 256, 100, 0, 16, first=17)
    assert cent.shape == (256, 16) and len(labels) == 10000 and 1 <= iters <= 100
    assert rows[0] == 17 and len(set(rows.tolist())) == 256


def test_kmeans_alias_writes_through():
    # kmeans.go:63,82,144: centroids alias input rows, update overwrites caller data
    rng = np.random.Generator(np.random.PCG64(6))
    X = rng.random((500, 4), dtype=np.float32)
    X0 = X.copy()
    cent, _, _, rows = O.kmeans_fit(X, 8, 100, 0, 4, first=3, alias=True)
    assert not np.array_equal(X, X0)
    for i, r in enumerate(rows):
        assert np.array_equal(X[r], cent[i])
    Xc = X0.copy()
    O.kmeans_fit(Xc, 8, 100, 0, 4, first=3, alias=False)
    assert np.array_equal(Xc, X0)


# ---- product quantiser ----------------------------------------------------

def test_pq_adc_and_sdc_consistency():
    rng = np.random.Generator(np.random.PCG64(8))
    n, dim, M, K = 1200, 32, 4, 16
    X = rng.standard_normal((n, dim)).astype(np.float32)
    ix = O.OracleIndex(dim, "euclidean", quantizer="product", pq_m=M, pq_k=K, pq_trigger=1000)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    ix.set_vectors(ids, X)
    assert ix.fit(pq_first=0) == 1
    fc, cd = ix.get_pq()
    codes = ix.get_codes(ids)
    assert codes.max() < K
    q = X[5]
    tab = ix.adc_table(q)
    sub = dim // M
    for i in range(M):
        for j in range(K):
            assert tab[i, j] == np.float32(O.float_dist("euclidean", q[i * sub:(i + 1) * sub], fc[i, j]))
    d = ix.query_dists(q, ids[:50])
    for t in range(50):
        s = np.float32(0)
        for i in range(M):
            s = np.float32(s + tab[i, codes[t, i]])
        assert d[t] == s
    s = np.float32(0)
    for i in range(M):
        s = np.float32(s + cd[i, codes[0, i], codes[1, i]])
    assert ix.point_dist(2, 3) == s


def test_pq_cosine_becomes_euclidean_and_validation():
    # product.go:44-65
    with pytest.raises(ValueError):
        O.OracleIndex(10, "euclidean", quantizer="product", pq_m=3, pq_k=4)
    with pytest.raises(ValueError):
        O.OracleIndex(8, "euclidean", quantizer="product", pq_m=2, pq_k=300)
    a = O.OracleIndex(4, "cosine", quantizer="product", pq_m=2, pq_k=2)
    a.set_vectors([2, 3], [[1, 0, 0, 0], [0, 1, 0, 0]])
    # unfitted: falls back to the (replaced) float metric = squared L2 (product.go:239-249)
    assert a.point_dist(2, 3) == 2.0


# ---- cluster merge --------------------------------------------------------

def test_shard_limit_formula():
    # cluster/actions.go:291-299
    assert O.shard_limit(10, 8) == 10
    assert O.shard_limit(100, 5) == 38
    assert O.shard_limit(75, 1) == 75


def test_merge_topk():
    ids = np.array([[[1, 2, 3]], [[4, 5, 6]]], dtype=np.uint64)
    d = np.array([[[0.1, 0.4, 0.9]], [[0.2, 0.4, 0.5]]], dtype=np.float32)
    c = np.array([[3], [2]], dtype=np.uint32)
    oi, od, oc = O.merge_topk(ids, d, c, 3)
    assert oi[0].tolist() == [1, 4, 2] and oc[0] == 3
    assert od[0].tolist() == [np.float32(0.1), np.float32(0.2), np.float32(0.4)]


# ---- update / delete path (vamana.go:223-253, prune.go, node.go:142-199) ----------------

def _graph_invariants(ix, alive_ids):
    """shard_vector_test.go:198-225 (no dangling or self edges) + vamana_test.go:63-75 (every
    point reachable from the start node)."""
    adj, deg = ix.get_graph()
    alive = set(int(i) for i in alive_ids) | {1}
    extra = [int(x) for x in ix.start_extra()]
    seen, todo = {1}, [1]
    while todo:
        v = todo.pop()
        nb = [int(x) for x in adj[v, :deg[v]]] + (extra if v == 1 else [])
        for u in nb:
            assert u in alive, f"edge {v}->{u} points at a deleted node"
            assert u != v, f"self edge at {v}"
            if u not in seen:
                seen.add(u)
                todo.append(u)
    assert seen == alive, f"{len(alive - seen)} points unreachable from the start node"


def test_edge_scan_kat():
    """vamana_test.go:142-175: graph 2->{3,6} 3->{2,4} 4->{3,5} 5->{4} 6->{2}; deleting {3,4}
    gives toPrune [2,5] and toSave [5]."""
    ix = O.OracleIndex(2, "euclidean", 75, 64, 1.2)
    ix.set_start(np.array([1, 0], np.float32))
    ix.set_vectors(np.arange(2, 7, dtype=np.uint32), np.zeros((5, 2), np.float32))
    adj = np.full((7, 64), 0xFFFFFFFF, dtype=np.uint32)
    deg = np.zeros(7, np.uint16)
    for nid, e in {2: [3, 6], 3: [2, 4], 4: [3, 5], 5: [4], 6: [2]}.items():
        adj[nid, :len(e)] = e
        deg[nid] = len(e)
    ix.set_graph(adj, deg)
    tp, ts = ix.edge_scan([3, 4])
    assert tp.tolist() == [2, 5] and ts.tolist() == [5]


@pytest.mark.parametrize("threads", [1, 4])
def test_update_delete_invariants(threads):
    """Test_ConcurrentCUD (vamana_test.go:92-140) + shard_vector_test.go:198-225,408-420."""
    rng = np.random.Generator(np.random.PCG64(5))
    n = 1500
    X = rng.random((n, 8), dtype=np.float32)
    ix = O.OracleIndex(8, "euclidean", 75, 64, 1.2)
    ix.set_start(O.random_unit_vector(8, 3))
    ids = np.arange(2, n + 2, dtype=np.uint32)
    ix.insert(ids, X, threads=threads)
    # one call: 200 new points, 150 updates, 250 deletes, 5 deletes of absent ids (skipped)
    new_ids = np.arange(n + 2, n + 202, dtype=np.uint32)
    upd_ids = ids[100:250]
    del_ids = ids[300:550]
    ghost = np.arange(5000, 5005, dtype=np.uint32)
    ch_ids = np.concatenate([new_ids, upd_ids, del_ids, ghost])
    vec = rng.random((len(ch_ids), 8), dtype=np.float32)
    has = np.concatenate([np.ones(350, np.uint8), np.zeros(255, np.uint8)])
    ix.update_delete(ch_ids, vec, has, threads=threads)
    alive = np.concatenate([np.setdiff1d(ids, del_ids), new_ids])
    assert ix.count == len(alive) + 1
    _graph_invariants(ix, alive)
    # updated points are found at their new position, deleted ones never come back
    got = ix.search(vec[200:350], k=10)
    assert (got["ids"][:, 0] == upd_ids).all() and (got["dists"][:, 0] == 0).all()
    assert not np.isin(got["ids"], del_ids).any()
    assert (ix.get_vectors(upd_ids) == vec[200:350]).all()


def test_delete_orphan_goes_to_start_overflow():
    """removeInboundEdges re-attaches nodes that lost every inbound edge to the start node with
    AddNeighbourIfNotExists (prune.go:137-151), which ignores the degree bound: with the start
    node already at R edges the orphan lands in the overflow list and stays searchable; a
    later pruneDeleteNeighbour of the start node folds the overflow back under R."""
    R = 4
    ix = O.OracleIndex(2, "euclidean", 25, R, 1.2)
    ix.set_start(np.array([1, 0], np.float32))
    pts = np.array([[i, 0.5 * i] for i in range(2, 11)], np.float32)
    ix.set_vectors(np.arange(2, 11, dtype=np.uint32), pts)
    adj = np.full((11, R), 0xFFFFFFFF, dtype=np.uint32)
    deg = np.zeros(11, np.uint16)
    g = {1: [2, 3, 4, 5], 2: [6, 3], 3: [2, 4], 4: [3, 5], 5: [4, 8], 6: [7], 7: [6], 8: [9, 10], 9: [8], 10: [8]}
    for nid, e in g.items():
        adj[nid, :len(e)] = e
        deg[nid] = len(e)
    ix.set_graph(adj, deg)
    tp, ts = ix.edge_scan([6])
    assert tp.tolist() == [2, 7] and ts.tolist() == [7]
    ix.update_delete(np.array([6], np.uint32), np.zeros((1, 2), np.float32), np.zeros(1, np.uint8))
    assert ix.start_extra().tolist() == [7]
    _graph_invariants(ix, [2, 3, 4, 5, 7, 8, 9, 10])
    got = ix.search(pts[5:6], k=3, search_size=25)  # node 7's own vector
    assert got["ids"][0, 0] == 7 and got["dists"][0, 0] == 0
    # deleting node 2 prunes the start node: candidates = {3,4,5,7} + N(2)\{deleted} -> <= R edges
    ix.update_delete(np.array([2], np.uint32), np.zeros((1, 2), np.float32), np.zeros(1, np.uint8))
    assert ix.start_extra().tolist() == []
    _graph_invariants(ix, [3, 4, 5, 7, 8, 9, 10])


def test_hybrid_merge_semantics():
    """indexManager.searchParallel (shard/index/search.go:259-298), shaped after the reference's
    TestSearch_Or / TestSearch_And / TestSearch_OrVector (shard/index/search_test.go:289-457):
    union vs intersection of the result-id sets, duplicate hits add their HybridScore, the first
    non-nil distance is kept, output sorted by HybridScore descending."""
    nan = np.float32(np.nan)
    # request 0: two sub-searches overlapping in ids 42 and 43
    ids = np.zeros((2, 1, 4), np.uint64)
    h = np.zeros((2, 1, 4), np.float32)
    d = np.full((2, 1, 4), nan, np.float32)
    ids[0, 0] = [42, 43, 44, 45]
    h[0, 0] = [-0.0, -0.5, -1.0, -1.5]      # vector search, weight 0.5: HybridScore = -d * w
    d[0, 0] = [0.0, 1.0, 2.0, 3.0]
    ids[1, 0, :3] = [43, 42, 7]
    h[1, 0, :3] = [2.0, 1.0, 0.5]           # text search: score * weight, no distance
    c = np.array([[4], [3]], np.uint32)
    oi, oh, od, oc = O.hybrid_merge(ids, h, d, c, disjunction=True)
    assert oc[0] == 5
    assert oi[0, :5].tolist() == [43, 42, 7, 44, 45]
    assert oh[0, :5].tolist() == [1.5, 1.0, 0.5, -1.0, -1.5]
    assert od[0, 0] == 1.0 and od[0, 1] == 0.0 and np.isnan(od[0, 2])
    assert (np.diff(oh[0, :5]) <= 0).all()
    oi, oh, od, oc = O.hybrid_merge(ids, h, d, c, disjunction=False)
    assert oc[0] == 2 and oi[0, :2].tolist() == [43, 42] and oh[0, :2].tolist() == [1.5, 1.0]
    # TestSearch_OrVector: the same five results from two searches with weight 0.5 each:
    # HybridScore adds up to -distance
    ids2 = np.tile(np.array([42, 43, 41, 44, 40], np.uint64), (2, 1, 1))
    d2 = np.tile(np.array([0.0, 2.0, 2.0, 8.0, 8.0], np.float32), (2, 1, 1))
    h2 = (np.float32(-1) * d2 * np.float32(0.5)).astype(np.float32)
    c2 = np.full((2, 1), 5, np.uint32)
    oi, oh, od, oc = O.hybrid_merge(ids2, h2, d2, c2, disjunction=True)
    assert oc[0] == 5 and oi[0, 0] == 42 and (oh[0, :5] == -od[0, :5]).all()
    assert oi[0, :5].tolist() == [42, 43, 41, 44, 40]  # ties keep first-appearance order
    # a single sub-search is returned as is (search.go:246-249)
    oi, oh, od, oc = O.hybrid_merge(ids[:1], h[:1], d[:1], c[:1], disjunction=False)
    assert oc[0] == 4 and oi[0].tolist() == [42, 43, 44, 45]


def test_round_insert_depends_on_the_input_only():
    """OracleIndex.insert(max_round=...): the same graph for any thread count, and rounds of one
    point are the reference's 1-worker schedule, edge for edge."""
    from semadb_b200 import synth
    X = synth.sift_shaped(3000, 32, 11)

    def graph(threads, max_round):
        ix = O.OracleIndex(32, "euclidean", 75, 64, 1.2)
        ix.set_start(synth.start_vector(32, 5))
        ix.insert(np.arange(2, len(X) + 2, dtype=np.uint32), X, threads=threads, max_round=max_round)
        return ix.get_graph()

    for want, got in ((graph(1, 64), graph(7, 64)), (graph(1, 0), graph(4, 1))):
        assert (want[1] == got[1]).all() and (want[0] == got[0]).all()
