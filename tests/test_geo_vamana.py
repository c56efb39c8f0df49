"""Haversine (geo) Vamana indexes: the GeoEval beam search, build, update/delete and the Python
surface on (latitude, longitude) rows, against the CPU oracle.

Parity bar. The device and the oracle compute float64 sin / cos / asin with different libraries
(CUDA's and glibc's), so a distance can differ by one float ulp in rare cases and a flipped
comparison can change a traversal. So:
  * bit for bit: every distance a search returns equals sdb_index_query_dists of the same
    (query, id) — the same device function;
  * against the oracle: distances within one float ulp (a row at exactly the query's coordinates:
    0 on the device, the oracle's FMA-contracted rounding residue, see _check_parity); ids, counts,
    hops and evaluations identical
    on >= 99.9 % of the rows. Each check prints how many rows differ (0 expected), and every
    differing row must contain a pair whose device and oracle distances differ."""
import numpy as np
import pytest

from semadb_b200 import synth
from semadb_b200.vamana import IndexVamana, IndexVectorChange, IndexVectorVamanaParameters, SearchVectorVamanaOptions

gpu = pytest.mark.gpu


def _bfs(n_rows, deg, adj_row):
    seen = {1}
    stack = [1]
    while stack:
        u = stack.pop()
        for v in adj_row(u)[:deg[u]]:
            v = int(v)
            if v not in seen:
                seen.add(v)
                stack.append(v)
    return seen


def _geo_mix(n_clustered, n_uniform, seed):
    """Clustered cities plus points uniform on the sphere (background=1)."""
    return np.concatenate([synth.geo_points(n_clustered, seed), synth.geo_points(n_uniform, seed + 1, background=1.0)])


def _edge_queries(n, seed):
    """Queries at the poles and on both sides of the antimeridian."""
    rng = np.random.Generator(np.random.PCG64(seed))
    m = n // 4
    north = np.stack([rng.uniform(89.0, 90.0, m), rng.uniform(-180, 180, m)], 1)
    south = np.stack([rng.uniform(-90.0, -89.0, m), rng.uniform(-180, 180, m)], 1)
    east = np.stack([rng.uniform(-60, 60, m), rng.uniform(179.0, 180.0, m)], 1)
    west = np.stack([rng.uniform(-60, 60, m), rng.uniform(-180.0, -179.0, m)], 1)
    q = np.concatenate([north, south, east, west]).astype(np.float32)
    q[q[:, 1] >= 180.0, 1] = -180.0
    return q


def test_oracle_geo_graph_cpu():
    """The oracle's haversine graph (vamana_test.go:63-75 property): BFS-connected from the start
    node, every point finds itself (or an exact duplicate) at rank 0, recall@10 >= 0.99."""
    from tests.helpers import oracle_graph, recall_at_k
    X = synth.geo_points(20_000, 11)
    oix, ids, _ = oracle_graph(X, "haversine", threads=1)
    adj, deg = oix.get_graph()
    assert len(_bfs(len(deg), deg, lambda u: adj[u])) == len(X) + 1
    self_hit = oix.search(X, k=10, threads=8)
    top = self_hit["ids"][:, 0].astype(np.int64) - 2
    # itself, an exact copy, or a point at the same place: at a pole every longitude is one point
    same_place = (X[top] == X).all(1) | (self_hit["dists"][:, 0] <= 1e-3)
    assert same_place.all(), ("a point did not find itself at rank 0", np.nonzero(~same_place)[0][:5])
    Q = synth.geo_queries(1000, 11)
    r = recall_at_k(oix.search(Q, k=10, threads=8)["ids"], oix.flat_search(Q, k=10, threads=8)["ids"])
    assert r >= 0.99, r


# ---- GPU ----------------------------------------------------------------------------------

def _ulp_close(a, b):
    return (a == b) | (a == np.nextafter(b, np.float32(np.inf))) | (a == np.nextafter(b, np.float32(-np.inf)))


def _check_parity(tag, oix, g, Q, gi, gd, gc, ref, hops=None, ndist=None, L=75, filters=None):
    """Parity bar of the module docstring. ref: oracle search of the same rows (diagnostics on when
    hops / ndist are given). filters[b]: the row's filter (None = unfiltered) for the evidence search."""
    B = len(Q)
    for b in range(B):  # bit for bit against the device's own distance function
        n = int(gc[b])
        if n:
            assert g.query_dists(Q[b], gi[b, :n]).tobytes() == gd[b, :n].tobytes(), (tag, b)
    same = (gc == ref["counts"]) & (gi == ref["ids"].astype(np.uint64)).all(1)
    if hops is not None:
        same &= (hops == ref["hops"]) & (ndist == ref["ndist"])
    # The oracle's compiler fuses lon_x*degToRad - lon_y and sdlat*sdlat + ... into FMAs (vfmsub /
    # vfmadd in liboracle.so), so for a row at exactly the query's coordinates it returns the
    # rounding error of lon_y (~1e-10 m) where the unfused formula, the device's, gives 0. Such a
    # pair is accepted only when the device says 0, the oracle less than a micrometre, and the row
    # equals the query.
    rd = ref["dists"]
    zero = (gd == 0) & (rd != 0) & (rd < 1e-6)
    for b in np.nonzero(zero.any(1))[0]:
        assert (g.get_vectors(gi[b][zero[b]]) == Q[b]).all(), (tag, b)
    close = (_ulp_close(gd, rd) | zero).all(1)
    far = np.nonzero(same & ~close)[0]
    assert len(far) == 0, (tag, "distances beyond one ulp", far[:5], [(gi[b], gd[b], ref["dists"][b]) for b in far[:2]])
    bad = np.nonzero(~same)[0]
    print(f"{tag}: {len(bad)} of {B} rows differ from the oracle")
    assert len(bad) <= B // 1000, (tag, bad[:10])
    for b in bad:
        # a differing row must start at a pair whose device and oracle distances differ
        f = None if filters is None else filters[b]
        vis = oix.search(Q[b:b + 1], k=1, search_size=L, filter_ids=f, vis_cap=512)
        cand = np.unique(np.concatenate([gi[b, :gc[b]], ref["ids"][b, :ref["counts"][b]], vis["vis_ids"][0, :vis["vis_len"][0]]]))
        cand = cand[cand >= 2]
        assert (g.query_dists(Q[b], cand) != oix.query_dists(Q[b], cand)).any(), (tag, b)


def _search_and_check(tag, oix, g, Q, k, L):
    gi, gd, gc = g.search_batch(Q, k, L)
    hops, nd = g.last_search_stats(len(Q))
    ref = oix.search(Q, k=k, search_size=L, threads=8, diagnostics=True)
    _check_parity(tag, oix, g, Q, gi, gd, gc, ref, hops, nd, L)
    assert (gc <= k).all()
    return gi, gd, gc, hops, nd


@pytest.fixture(scope="module")
def geo40k():
    """20 k clustered + 20 k uniform-sphere points, oracle-built graph mirrored onto the GPU."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    X = _geo_mix(20_000, 20_000, 21)
    oix, ids, start = oracle_graph(X, "haversine")
    g = mirror_to_gpu(oix, X, ids, start, "haversine")
    Q = np.concatenate([synth.geo_queries(600, 21), _edge_queries(400, 22)])
    return oix, g, X, ids, Q


@gpu
@pytest.mark.parametrize("k,L", [(10, 75), (1, 25), (75, 75)])
def test_geo_search_on_oracle_graph(geo40k, k, L):
    oix, g, X, ids, Q = geo40k
    _search_and_check(f"geo search k={k} L={L}", oix, g, Q, k, L)


@gpu
def test_geo_search_exact_duplicates():
    """30 % of the points are exact copies of others (POIs at one address): equal inputs give equal
    distances on both sides, so ties are real, and the newest-equal-wins rule of AddWithLimit
    (distset.go:184-194) decides which copy keeps the last slot of the list."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    rng = np.random.Generator(np.random.PCG64(31))
    base = synth.geo_points(7_000, 31, centres=50, spread_deg=0.05)
    X = np.concatenate([base, base[rng.integers(0, len(base), 3_000)]])
    X = X[rng.permutation(len(X))]
    oix, ids, start = oracle_graph(X, "haversine")
    g = mirror_to_gpu(oix, X, ids, start, "haversine")
    Q = np.concatenate([X[rng.integers(0, len(X), 300)], synth.geo_queries(300, 31, centres=50, spread_deg=0.05)])
    for k, L in ((10, 75), (1, 25), (75, 75)):
        _search_and_check(f"duplicates k={k} L={L}", oix, g, Q, k, L)


@gpu
def test_geo_per_request_filters(geo40k):
    """Filtered, unfiltered and empty-filter requests in one batch (search_batch_filters)."""
    oix, g, X, ids, Q = geo40k
    rng = np.random.Generator(np.random.PCG64(41))
    B = 120
    Qb = Q[:B]
    filters = [np.sort(rng.choice(ids, size=nf, replace=False)) for nf in (1, 40, 75, 76, 500, 5000)] + [np.zeros(0, np.uint64)]
    qf = np.array([(b % (len(filters) + 1)) - 1 for b in range(B)], dtype=np.int32)  # -1 = unfiltered
    gi, gd, gc = g.search_batch_filters(Qb, filters, qf, 10, 75)
    rows = {"ids": np.zeros((B, 10), np.uint32), "dists": np.zeros((B, 10), np.float32), "counts": np.zeros(B, np.uint32)}
    plain = oix.search(Qb, k=10, threads=8)
    row_filter = []
    for b in range(B):
        f = qf[b]
        row_filter.append(None if f < 0 else filters[f])
        if f >= 0 and len(filters[f]) == 0:  # a non-nil empty filter seeds nothing: no result
            assert gc[b] == 0 and (gi[b] == 0).all()
            rows["dists"][b] = np.inf
            continue
        r = plain if f < 0 else oix.search(Qb[b:b + 1], k=10, filter_ids=filters[f])
        i = b if f < 0 else 0
        for key in rows:
            rows[key][b] = r[key][i]
    _check_parity("filters", oix, g, Qb, gi, gd, gc, rows, filters=row_filter)


@gpu
def test_geo_retry_path(geo40k, monkeypatch):
    """A visited table far too small (64 slots) sends every query through the RETRY launch
    (VisitedBitmap, same evaluator): results equal the normal run's, and the insert path, whose
    searches then all retry, still builds the same graph."""
    oix, g, X, ids, Q = geo40k
    want = g.search_batch(Q, 10, 75)
    whops = g.last_search_stats(len(Q))
    monkeypatch.setenv("SDB_VT_SLOTS", "64")
    got = g.search_batch(Q, 10, 75)
    ghops = g.last_search_stats(len(Q))
    for a, b in zip(want + whops, got + ghops):
        assert a.tobytes() == b.tobytes()
    Xs = synth.geo_points(1_500, 43)
    start = synth.start_vector(2, 99)
    graphs = []
    for slots in ("64", None):
        if slots:
            monkeypatch.setenv("SDB_VT_SLOTS", slots)
        else:
            monkeypatch.delenv("SDB_VT_SLOTS")
        b = IndexVamana("retry", IndexVectorVamanaParameters(2, "haversine"), start_vector=start)
        b.insert_config(1, 1, 1)
        b.insert_batch(np.arange(2, len(Xs) + 2, dtype=np.uint64), Xs)
        graphs.append(b.get_edges(np.arange(1, len(Xs) + 2, dtype=np.uint64)))
    assert (graphs[0][0] == graphs[1][0]).all() and (graphs[0][1] == graphs[1][1]).all()


def _graph_diff(oix, g, n_rows):
    adj, odeg = oix.get_graph(n_rows)
    deg, e = g.get_edges(np.arange(1, n_rows, dtype=np.uint64))
    return [i + 1 for i in range(n_rows - 1) if deg[i] != odeg[i + 1] or (e[i, :deg[i]] != adj[i + 1, :deg[i]]).any()]


@gpu
def test_geo_sequential_build_matches_oracle():
    """insert_config(1, 1, 1): the reference's sequential schedule, the oracle's graph edge for edge
    (this runs the haversine branch of the prune kernels: robustPrune of the new point and of its
    saturated back-edge targets)."""
    from tests.helpers import oracle_graph
    X = synth.geo_points(3_000, 51)
    oix, ids, start = oracle_graph(X, "haversine", threads=1)
    g = IndexVamana("seq", IndexVectorVamanaParameters(2, "haversine"), start_vector=start)
    g.insert_config(1, 1, 1)
    g.insert_batch(ids.astype(np.uint64), X)
    diff = _graph_diff(oix, g, len(X) + 2)
    print(f"sequential geo build: {len(diff)} of {len(X) + 1} nodes differ from the oracle")
    assert not diff, diff[:10]


@gpu
def test_geo_batched_build_quality():
    """Default mini-batch schedule on 100 k geo points: recall@10 of the GPU graph within 0.005 of
    the oracle graph's on the same queries, BFS-connected, no truncated visited list."""
    from semadb_b200 import _capi
    from tests.helpers import oracle_graph, recall_at_k
    n = 100_000
    X = synth.geo_points(n, 61)
    Q = synth.geo_queries(1000, 61)
    oix, ids, start = oracle_graph(X, "haversine")
    g = IndexVamana("build", IndexVectorVamanaParameters(2, "haversine"), start_vector=start)
    g.insert_batch(ids.astype(np.uint64), X)
    gt = oix.flat_search(Q, k=10, threads=8)
    r_ref = recall_at_k(oix.search(Q, k=10, threads=8)["ids"], gt["ids"])
    r_gpu = recall_at_k(g.search_batch(Q, 10, 75)[0], gt["ids"].astype(np.uint64))
    print(f"geo 100k build: recall@10 gpu graph {r_gpu:.4f}, oracle graph {r_ref:.4f}")
    assert r_gpu >= r_ref - 0.005, (r_gpu, r_ref)
    deg, e = g.get_edges(np.arange(1, n + 2, dtype=np.uint64))
    assert len(_bfs(n + 2, np.concatenate([[0], deg]), lambda u: e[u - 1])) == n + 1
    assert _capi.lib().sdb_insert_truncated(g._h) == 0


@gpu
def test_geo_update_delete_matches_oracle():
    """One insert_update_delete call (5 % deleted, 5 % moved, new points inserted) gives the oracle's
    update_delete graph edge for edge (pruneDeleteNeighbour's haversine branch), and no search
    afterwards returns a deleted id."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    n = 3_000
    rng = np.random.Generator(np.random.PCG64(71))
    X = synth.geo_points(n, 71)
    fresh = synth.geo_queries(400, 71, query_seed=2)
    oix, ids, start = oracle_graph(X, "haversine", threads=1)
    g = mirror_to_gpu(oix, X, ids, start, "haversine")
    g.insert_config(1, 1, 1)
    perm = rng.permutation(ids)
    del_ids, mov_ids = perm[:150], perm[150:300]
    new_ids = np.arange(n + 2, n + 202, dtype=np.uint32)
    ch = np.concatenate([new_ids, mov_ids, del_ids]).astype(np.uint32)
    vec = np.concatenate([fresh[:350], np.zeros((150, 2), np.float32)])
    has = np.concatenate([np.ones(350, np.uint8), np.zeros(150, np.uint8)])
    oix.update_delete(ch, vec, has, threads=1)
    g.insert_update_delete_batch(ch.astype(np.uint64), vec, has)
    assert g.count == oix.count
    diff = _graph_diff(oix, g, n + 202)
    print(f"geo update/delete: {len(diff)} nodes differ from the oracle")
    assert not diff, diff[:10]
    assert g.get_start_overflow().tolist() == oix.start_extra().tolist()
    Q = np.concatenate([fresh[350:], X[del_ids - 2][:50]])
    gi, gd, gc, _, _ = _search_and_check("after update/delete", oix, g, Q, 10, 75)
    assert not np.isin(gi, del_ids.astype(np.uint64)).any()


@gpu
def test_geo_python_surface_kat():
    """IndexVamana with a haversine index through insert_update_delete / search: the reference's
    KAT (Buenos Aires -> Paris, 11 099.54 km) through a graph search, hybrid_score = -distance*weight."""
    X = synth.geo_points(60, 81)  # fewer points than the limit: the search returns every one
    paris = np.array([49.0083899664, 2.53844117956], np.float32)
    buenos_aires = [-34.83333, -58.5166646]
    g = IndexVamana("geo", IndexVectorVamanaParameters(2, "haversine"), start_seed=5)
    g.insert_update_delete([IndexVectorChange(2, paris)] + [IndexVectorChange(i + 3, X[i]) for i in range(len(X))])
    w = 0.5
    found, res = g.search(SearchVectorVamanaOptions(buenos_aires, search_size=75, limit=75, weight=w))
    assert len(res) == len(X) + 1 and len(found) == len(X) + 1
    d = [r.distance for r in res]
    assert d == sorted(d)
    for r in res:
        assert r.hybrid_score == float(np.float32(-1) * np.float32(r.distance) * np.float32(w))
    _, near = g.search(SearchVectorVamanaOptions(paris.tolist(), search_size=75, limit=1))
    assert near[0].node_id == 2 and near[0].distance == 0.0
    ba = g.query_dists(np.array(buenos_aires, np.float32), [2])[0]
    assert abs(float(ba) - 11_099_540.0) <= 10.0, ba
    assert [r.distance for r in res if r.node_id == 2] == [float(ba)]


@gpu
def test_geo_gather_epilogue(geo40k):
    """sdb_search_batch_gather_device with one peer: the gather buffer holds the lists of
    sdb_search_batch_device, ids tagged shard << 40."""
    import ctypes as C

    import torch
    from semadb_b200 import _capi
    oix, g, X, ids, Q = geo40k
    B, k, shard = len(Q), 10, 3
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_q = torch.from_numpy(Q).to(dev)
    u_ids = torch.zeros((B, k), dtype=torch.int64, device=dev)
    u_d = torch.zeros((B, k), dtype=torch.float32, device=dev)
    u_c = torch.zeros((B,), dtype=torch.int32, device=dev)
    g.search_batch_device(d_q, k, 75, u_ids, u_d, u_c, st)
    S = shard + 1
    f_ids = torch.full((S, B, k), -1, dtype=torch.int64, device=dev)
    f_d = torch.full((S, B, k), -1.0, dtype=torch.float32, device=dev)
    f_c = torch.full((S, B), -1, dtype=torch.int32, device=dev)
    l_ids = torch.zeros((B, k), dtype=torch.int64, device=dev)
    l_d = torch.zeros((B, k), dtype=torch.float32, device=dev)
    l_c = torch.zeros((B,), dtype=torch.int32, device=dev)
    pg = _capi.SdbPeerGather()
    pg.n_peers, pg.shard, pg.per_shard_limit = 1, shard, 0
    pg.ids[0], pg.dists[0], pg.counts[0] = f_ids.data_ptr(), f_d.data_ptr(), f_c.data_ptr()
    _capi.check(_capi.lib().sdb_search_batch_gather_device(g._h, B, d_q.data_ptr(), k, 75, l_ids.data_ptr(),
                                                           l_d.data_ptr(), l_c.data_ptr(), C.byref(pg), st))
    torch.cuda.synchronize()
    ui, ud, uc = u_ids.cpu().numpy(), u_d.cpu().numpy(), u_c.cpu().numpy()
    assert (l_ids.cpu().numpy() == ui).all() and l_d.cpu().numpy().tobytes() == ud.tobytes() and (l_c.cpu().numpy() == uc).all()
    assert (f_c[shard].cpu().numpy() == uc).all()
    tag = np.int64(shard) << np.int64(40)
    fi = f_ids[shard].cpu().numpy()
    for b in range(B):
        n = int(uc[b])
        assert (fi[b, :n] == (ui[b, :n] | tag)).all(), b
    assert f_d[shard].cpu().numpy().tobytes() == ud.tobytes()
    # the host-buffer entry point returns the same lists
    hi, hd, hc = g.search_batch(Q, k, 75)
    assert (hi == ui.astype(np.uint64)).all() and hd.tobytes() == ud.tobytes()
