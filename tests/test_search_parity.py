"""K1 parity: CUDA beam search vs the oracle on the oracle-built graph, through the C ABI.
Bit-exact ids, distances, hop and distance-evaluation counts (SURVEY.md §7.3-①/②)."""
import numpy as np
import pytest

from semadb_b200 import synth
from tests.helpers import check_search as _check_search

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("metric", ["euclidean", "dot", "cosine"])
@pytest.mark.parametrize("dim", [128, 2, 100, 384])
def test_search_matches_oracle(metric, dim):
    from tests.helpers import mirror_to_gpu, oracle_graph
    n = 4000 if dim > 128 else 8000
    X = synth.latent_gaussian(n, dim, seed=dim, latent=min(8, dim), normalize=(metric == "cosine"))
    Q = synth.latent_gaussian(300, dim, seed=dim + 1, w_seed=dim, latent=min(8, dim), normalize=(metric == "cosine"))
    oix, ids, start = oracle_graph(X, metric)
    g = mirror_to_gpu(oix, X, ids, start, metric)
    _check_search(oix, g, Q)
    _check_search(oix, g, Q[:50], k=1, L=25)
    _check_search(oix, g, Q[:50], k=75, L=75)


def test_search_c1_shape_small():
    """C1-shaped (uniform 128-d, saturated degrees) at 20k points."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    X = synth.uniform(20000, 128, 1)
    Q = synth.uniform(1000, 128, 2)
    oix, ids, start = oracle_graph(X)
    g = mirror_to_gpu(oix, X, ids, start)
    _check_search(oix, g, Q)


@pytest.mark.parametrize("dim", [128, 96])
def test_search_boundary_ties(dim):
    """0/1-valued coordinates: squared-L2 distances are small integers, so ties at the cut of
    the candidate list are everywhere — the newest-equal-wins rule (distset.go:184-194) must
    hold in the batch form of the list update too."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    rng = np.random.Generator(np.random.PCG64(11))
    X = (rng.random((6000, dim)) < 0.3).astype(np.float32)
    X[1000:1200] = X[:200]  # exact duplicates
    Q = (rng.random((400, dim)) < 0.3).astype(np.float32)
    oix, ids, start = oracle_graph(X)
    g = mirror_to_gpu(oix, X, ids, start)
    _check_search(oix, g, Q)
    _check_search(oix, g, X[:300], k=75, L=75)
    _check_search(oix, g, Q[:100], k=5, L=25)


def test_search_sift_shaped_100k():
    from tests.helpers import mirror_to_gpu, oracle_graph, recall_at_k
    X = synth.sift_shaped(100_000, 128, 3)
    Q = synth.sift_shaped(2000, 128, 4, w_seed=3)
    oix, ids, start = oracle_graph(X)
    g = mirror_to_gpu(oix, X, ids, start)
    ref = _check_search(oix, g, Q)
    gt = oix.flat_search(Q[:500], k=10, threads=8)
    assert recall_at_k(ref["ids"][:500], gt["ids"]) >= 0.95
    # GPU flat (K5) must agree bit-exactly with the oracle's brute force
    fi, fd, fc = g.flat_search_batch(Q[:500], 10)
    assert (fi == gt["ids"].astype(np.uint64)).all()
    assert fd.tobytes() == gt["dists"].tobytes()


def test_search_empty_and_tiny():
    """vamana_test.go:213-228 (empty) and graphs smaller than k."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    from semadb_b200.vamana import IndexVamana, IndexVectorVamanaParameters
    g = IndexVamana("empty", IndexVectorVamanaParameters(2), start_seed=1)
    ids, d, cnt = g.search_batch(np.array([[0.5, 0.5]], dtype=np.float32), 10, 75)
    assert cnt[0] == 0 and (ids == 0).all() and np.isinf(d).all()
    X = synth.uniform(5, 2, 3)
    oix, pid, start = oracle_graph(X, threads=1)
    g2 = mirror_to_gpu(oix, X, pid, start)
    _check_search(oix, g2, X)


def test_search_self_recall_200():
    """vamana_test.go:230-252."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    X = synth.uniform(200, 2, 5)
    oix, pid, start = oracle_graph(X, threads=1)
    g = mirror_to_gpu(oix, X, pid, start)
    ids, d, cnt = g.search_batch(X, 10, 75)
    assert (cnt == 10).all() and (ids[:, 0] == pid).all() and (d[:, 0] == 0).all()


def test_search_size_lt_k_is_error():
    """search.go:23-25."""
    from semadb_b200._capi import ERR_SEARCHSIZE, SdbError
    from semadb_b200.vamana import IndexVamana, IndexVectorVamanaParameters
    g = IndexVamana("e", IndexVectorVamanaParameters(2), start_seed=1)
    with pytest.raises(SdbError) as ei:
        g.search_batch(np.zeros((1, 2), np.float32), 30, 25)
    assert ei.value.code == ERR_SEARCHSIZE


def test_search_filter():
    """vamana_test.go:254-276 + oracle parity with a larger filter."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    X = synth.uniform(3000, 8, 7)
    oix, pid, start = oracle_graph(X, threads=1)
    g = mirror_to_gpu(oix, X, pid, start)
    filt = [int(pid[10]), int(pid[20]), int(pid[30])]
    ids, d, cnt = g.search_batch(X[10:11], 10, 75, filter_ids=filt)
    assert cnt[0] == 3 and ids[0, 0] == pid[10] and sorted(ids[0, :3].tolist()) == sorted(filt)
    rng = np.random.Generator(np.random.PCG64(3))
    for nf in (1, 40, 75, 76, 500):
        f = np.sort(rng.choice(pid, size=nf, replace=False))
        ref = oix.search(X[:64], k=10, filter_ids=f, threads=4)
        ids, d, cnt = g.search_batch(X[:64], 10, 75, filter_ids=f)
        assert (cnt == ref["counts"]).all()
        assert (ids == ref["ids"].astype(np.uint64)).all()
        assert d.tobytes() == ref["dists"].tobytes()


def test_visited_list_matches_oracle():
    """greedySearch's second return value (search.go:100), the robustPrune candidate list."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    X = synth.sift_shaped(20000, 128, 3)
    oix, pid, start = oracle_graph(X)
    g = mirror_to_gpu(oix, X, pid, start)
    Q = synth.sift_shaped(200, 128, 4, w_seed=3)
    ref = oix.search(Q, k=1, vis_cap=256, threads=8)
    vi, vd, vn = g.search_visited(Q, 75, 256)
    assert (vn == ref["vis_len"]).all()
    for b in range(len(Q)):
        n = vn[b]
        assert (vi[b, :n] == ref["vis_ids"][b, :n]).all()
        assert vd[b, :n].tobytes() == ref["vis_dists"][b, :n].tobytes()


def test_search_batch_pinned_buffers_zero_copy():
    """sdb_search_batch with page-locked caller buffers (the kernel reads queries from and writes
    results to mapped host memory) must return exactly what the staged-copy path returns for
    pageable buffers, and what the oracle returns."""
    import ctypes as C

    import torch
    from semadb_b200 import _capi
    from tests.helpers import mirror_to_gpu, oracle_graph
    n, dim, B, k = 6000, 128, 500, 10
    X = synth.sift_shaped(n, dim, 3)
    Q = synth.sift_shaped(B, dim, 4, w_seed=3)
    oix, ids, start = oracle_graph(X)
    g = mirror_to_gpu(oix, X, ids, start)
    ref = oix.search(Q, k=k, threads=8)
    pi, pd, pc = g.search_batch(Q, k, 75)  # numpy (pageable) buffers: staging copies
    h_q = torch.from_numpy(Q).pin_memory()
    h_ids = torch.zeros((B, k), dtype=torch.int64).pin_memory()
    h_d = torch.zeros((B, k), dtype=torch.float32).pin_memory()
    h_c = torch.zeros((B,), dtype=torch.int32).pin_memory()
    _capi.check(_capi.lib().sdb_search_batch(g._h, B, C.cast(h_q.data_ptr(), _capi.f32p), k, 75, None, 0,
                                             C.cast(h_ids.data_ptr(), _capi.u64p), C.cast(h_d.data_ptr(), _capi.f32p),
                                             C.cast(h_c.data_ptr(), _capi.u32p)))
    assert (h_ids.numpy().astype(np.uint64) == pi).all() and h_d.numpy().tobytes() == pd.tobytes()
    assert (h_c.numpy().astype(np.uint32) == pc).all()
    assert (pi == ref["ids"].astype(np.uint64)).all() and pd.tobytes() == ref["dists"].tobytes()


def test_search_per_request_filters_and_empty_filter():
    """One filter per request in one batch (shard/index/search.go:59-85 -> vamana/search.go:33-51,
    93-95): filtered, unfiltered and empty-filter requests mixed; every row must equal the oracle's
    answer for that request alone. An empty (non-nil) filter returns nothing."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    X = synth.uniform(4000, 16, 7)
    oix, pid, start = oracle_graph(X, threads=1)
    g = mirror_to_gpu(oix, X, pid, start)
    rng = np.random.Generator(np.random.PCG64(5))
    B = 96
    Q = X[:B]
    filters = [np.sort(rng.choice(pid, size=nf, replace=False)) for nf in (1, 40, 75, 76, 500, 2500)] + [np.zeros(0, np.uint64)]
    qf = np.array([(b % (len(filters) + 1)) - 1 for b in range(B)], dtype=np.int32)  # -1 = unfiltered
    ids, d, cnt = g.search_batch_filters(Q, filters, qf, 10, 75)
    plain = oix.search(Q, k=10, threads=4)
    for b in range(B):
        f = qf[b]
        if f < 0:
            ref = {k_: v[b] for k_, v in plain.items()}
        elif len(filters[f]) == 0:
            assert cnt[b] == 0 and (ids[b] == 0).all()
            continue
        else:
            r = oix.search(Q[b:b + 1], k=10, filter_ids=filters[f], threads=1)
            ref = {k_: v[0] for k_, v in r.items()}
        assert cnt[b] == ref["counts"], (b, f)
        assert (ids[b] == ref["ids"].astype(np.uint64)).all(), (b, f)
        assert d[b].tobytes() == ref["dists"].tobytes(), (b, f)
    # the shared-filter entry point treats a non-NULL empty list the same way
    ids, d, cnt = g.search_batch(Q[:4], 10, 75, filter_ids=np.zeros(0, np.uint64))
    assert (cnt == 0).all()
    # everybody shares filter 0 (query_filter = None)
    ids, d, cnt = g.search_batch_filters(Q[:8], [filters[3]], None, 10, 75)
    ref = oix.search(Q[:8], k=10, filter_ids=filters[3], threads=2)
    assert (ids == ref["ids"].astype(np.uint64)).all() and d.tobytes() == ref["dists"].tobytes()


def test_search_retry_bitmap_is_exact(monkeypatch):
    """A query that overflows the compact shared-memory visited table is re-run against an exact
    global-memory bitmap (the reference's visited bitset never fills up, distset.go:41,140-155):
    with a table far too small for any query, every query takes that path and must still equal
    the oracle — ids, distances, hop and distance counts — and no overflow marker may escape."""
    from tests.helpers import mirror_to_gpu, oracle_graph
    X = synth.sift_shaped(20000, 128, 3)
    oix, pid, start = oracle_graph(X)
    g = mirror_to_gpu(oix, X, pid, start)
    Q = synth.sift_shaped(300, 128, 4, w_seed=3)
    monkeypatch.setenv("SDB_VT_SLOTS", "64")
    ref = _check_search(oix, g, Q)
    assert (ref["counts"] <= 10).all()
    # insert path: the visited list of a re-run query reaches the prune kernel intact
    vi, vd, vn = g.search_visited(Q[:50], 75, 256)
    r2 = oix.search(Q[:50], k=1, vis_cap=256, threads=8)
    assert (vn == r2["vis_len"]).all()
    for b in range(50):
        assert (vi[b, :vn[b]] == r2["vis_ids"][b, :vn[b]]).all()
