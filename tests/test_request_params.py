"""Search batches in which every request has its own limit and searchSize (sdb_search_batch_requests,
sdb_flat_search_batch_requests and their _device twins, sdb_merge_topk_requests_device): every row
against the existing filter entries run on the requests that share its (limit, searchSize), on every
store, with ties across the cut of a filtered result list, on the RETRY launch, through the fused
exchange, and the argument errors."""
import ctypes as C

import numpy as np
import pytest

from oracle import oraclelib as O
from semadb_b200 import _capi, sharded, synth
from semadb_b200._capi import SdbError
from semadb_b200.vamana import (IndexFlat, IndexVectorFlatParameters, PackedRequests, ProductQuantizerParameters,
                                Quantizer)
from tests.helpers import mirror_to_gpu, oracle_graph
from tests.test_sharded_filters import _batches, _flat

pytestmark = pytest.mark.gpu

LIMITS = (1, 5, 10, 37, 75)
INF = np.float32(np.inf)


def _mix(B, rng, tiny=True):
    """limits from LIMITS with searchSizes from {limit, 25, 50, 75} (never below the limit), and a few
    tiny searchSizes (a relaxed index accepts 1..75)."""
    lim = np.array(LIMITS)[rng.integers(0, len(LIMITS), B)]
    L = np.array([rng.choice([x for x in (int(l), 25, 50, 75) if x >= l]) for l in lim])
    if tiny:
        for b in range(0, B, 11):
            lim[b] = 1 + b % 3
            L[b] = lim[b] + b % 2
    return lim.astype(np.int64), L.astype(np.int64)


def _pad(row, k_stride):
    i, d, c = row
    out_i = np.zeros((len(c), k_stride), np.uint64)
    out_d = np.full((len(c), k_stride), INF, np.float32)
    out_i[:, :i.shape[1]], out_d[:, :i.shape[1]] = i, d
    return out_i, out_d, c


def _expect(g, flat, Q, lim, L, filters, qf, k_stride):
    """Row b from the existing entries, run on the requests sharing b's (limit, searchSize)."""
    B = len(Q)
    ei, ed, ec = np.zeros((B, k_stride), np.uint64), np.full((B, k_stride), INF, np.float32), np.zeros(B, np.uint32)
    keys = sorted(set(zip(lim.tolist(), (L if not flat else np.zeros(B, np.int64)).tolist())))
    for k, l in keys:
        idx = np.nonzero((lim == k) & ((L == l) if not flat else True))[0]
        q = Q[idx]
        if filters is None:
            r = g.flat_search_batch(q, k) if flat else g.search_batch(q, k, l)
        else:
            sub = None if qf is None else qf[idx]
            r = g.flat_search_batch_filters(q, filters, sub, k) if flat else g.search_batch_filters(q, filters, sub, k, l)
        ei[idx], ed[idx], ec[idx] = _pad(r, k_stride)
    return ei, ed, ec


def _same(a, b):
    return all(np.asarray(x).tobytes() == np.asarray(y).tobytes() for x, y in zip(a, b))


def _device(g, flat, Q, rq, k_stride, peers=None):
    import torch
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(np.ascontiguousarray(Q)).to(dev)
    o = (torch.full((len(Q), k_stride), -1, dtype=torch.int64, device=dev),
         torch.full((len(Q), k_stride), -1.0, dtype=torch.float32, device=dev),
         torch.full((len(Q),), -1, dtype=torch.int32, device=dev))
    entry = g.flat_search_batch_requests_device if flat else g.search_batch_requests_device
    entry(d_q, rq, k_stride, *o, torch.cuda.current_stream().cuda_stream, peers)
    torch.cuda.synchronize()
    i, d, c = (t.cpu().numpy() for t in o)
    return i.view(np.uint64), d, c.view(np.uint32)


def _check(g, flat, Q, lim, L, filters=None, qf=None):
    k_stride = int(lim.max())
    want = _expect(g, flat, Q, lim, L, filters, qf, k_stride)
    if flat:
        got = g.flat_search_batch_requests(Q, lim, filters, qf)
    else:
        got = g.search_batch_requests(Q, lim, L, filters, qf)
    assert _same(want, got)
    rq = PackedRequests(len(Q), lim, L, filters, qf, default_L=g.L)
    assert _same(want, _device(g, flat, Q, rq, k_stride))
    return want


# ---------------------------------------------------------------- 1. beam search, every store

def _vamana(kind, n=3000, B=96):
    if kind in ("l2_128", "l2_100"):
        dim = 128 if kind == "l2_128" else 100
        X, Q = synth.sift_shaped(n, dim, 3), synth.sift_shaped(B, dim, 4, w_seed=3)
        metric, quant = "euclidean", None
    elif kind in ("dot", "cosine"):
        X = synth.latent_gaussian(n, 64, seed=11, latent=8, normalize=(kind == "cosine"))
        Q = synth.latent_gaussian(B, 64, seed=12, w_seed=11, latent=8, normalize=(kind == "cosine"))
        metric, quant = kind, None
    elif kind == "haversine":
        X, Q = synth.geo_points(n, 5), synth.geo_points(B, 6, background=1.0)
        metric, quant = "haversine", None
    elif kind in ("hamming", "jaccard"):
        X = synth.planted_bits(n, 256, seed=7, n_proto=64)
        Q = synth.planted_bits(B, 256, seed=10, n_proto=64, proto_seed=7)
        metric, quant = kind, None
    else:  # pq_fly / pq_table
        X = synth.latent_gaussian(n, 64, seed=41, latent=8)
        Q = synth.latent_gaussian(B, 64, seed=42, w_seed=41, latent=8)
        metric, quant = "euclidean", Quantizer("product", product=ProductQuantizerParameters(64, 8, 1000))
    X, Q = np.ascontiguousarray(X, np.float32), np.ascontiguousarray(Q, np.float32)
    oix, pid, start = oracle_graph(X, metric)
    g = mirror_to_gpu(oix, X, pid, start, metric, quantizer=quant, relaxed=True)
    if quant is not None:
        assert g.fit(0) is True
    return g, oix, pid, Q


@pytest.mark.parametrize("kind", ["l2_128", "l2_100", "dot", "cosine", "haversine", "hamming", "jaccard", "pq_fly",
                                  "pq_table"])
def test_beam_search_rows_equal_the_existing_entries(kind, monkeypatch):
    if kind == "pq_table":
        monkeypatch.setenv("SDB_ADC_TABLE", "1")
    g, oix, pid, Q = _vamana(kind)
    rng = np.random.default_rng(1)
    lim, L = _mix(len(Q), rng)
    want = _check(g, False, Q, lim, L)
    if kind in ("l2_128", "l2_100", "dot", "cosine", "haversine"):  # an oracle-built graph over raw rows
        for b in range(len(Q)):
            r = oix.search(Q[b:b + 1], k=int(lim[b]), search_size=int(L[b]), threads=1)
            c = int(r["counts"][0])
            assert want[2][b] == c
            assert (want[0][b, :c] == r["ids"][0, :c].astype(np.uint64)).all()
            assert want[1][b, :c].tobytes() == r["dists"][0, :c].tobytes()
    for name, filters, qf in _batches(rng, pid, len(Q), False):
        _check(g, False, Q, lim, L, filters, qf)


# ---------------------------------------------------------------- 2. ties across the cut of a filtered list

def test_filtered_ties_are_not_a_truncated_max_k_search():
    """Integer-valued rows copied to several ids: a filtered result list bounded at k keeps the last
    equal-distance node it met in its last slot, so it is not the first k of the list bounded at 75."""
    rng = np.random.default_rng(7)
    base = synth.sift_shaped(1500, 128, 3)
    dup = np.repeat(base[:60], 12, axis=0)  # 60 vectors, 12 copies each
    X = np.ascontiguousarray(np.concatenate([base, dup]), np.float32)
    Q = np.ascontiguousarray(base[:60] + rng.integers(-2, 3, size=(60, 128)), np.float32)
    oix, pid, start = oracle_graph(X)
    g = mirror_to_gpu(oix, X, pid, start, relaxed=True)
    copies = lambda v: np.concatenate([[pid[v]], pid[1500 + 12 * v:1500 + 12 * (v + 1)]])
    filters = [np.sort(np.concatenate([copies(v) for v in range(j, 60, 3)] + [rng.choice(pid, 40, replace=False)]))
               for j in range(3)]
    filters = [np.unique(f).astype(np.uint64) for f in filters]
    assert all(len(f) > 75 for f in filters)
    B = len(Q)
    qf = (np.arange(B) % 3).astype(np.int32)
    lim = np.array([(3, 5, 7, 10)[b % 4] for b in range(B)], np.int64)
    L = np.array([(25, 40, 60, 75)[(b // 4) % 4] for b in range(B)], np.int64)  # shared filters, other seeds
    want = _check(g, False, Q, lim, L, filters, qf)
    differs = 0  # rows where the search at the batch's largest limit, cut to the row's, differs
    for l in set(L.tolist()):
        idx = np.nonzero(L == l)[0]
        trunc = g.search_batch_filters(Q[idx], filters, qf[idx], int(lim.max()), l)
        differs += sum(not (want[0][b, :lim[b]] == trunc[0][j, :lim[b]]).all() for j, b in enumerate(idx))
    assert differs > 0, "no row separates a k-bounded result list from a truncated 75-bounded one"


# ---------------------------------------------------------------- 3. RETRY launch

def test_retry_launch_mixed_filtered_and_unfiltered(monkeypatch):
    g, _, pid, Q = _vamana("l2_128")
    monkeypatch.setenv("SDB_VT_SLOTS", "64")  # every query overflows its visited table: RETRY launch
    rng = np.random.default_rng(2)
    lim, L = _mix(len(Q), rng)
    filters = [np.sort(rng.choice(pid, size=m, replace=False)).astype(np.uint64) for m in (30, 500)] + [np.zeros(0, np.uint64)]
    qf = (np.arange(len(Q), dtype=np.int32) % 5) - 2  # -2, -1: unfiltered; 2: the empty filter
    qf[qf < 0] = -1
    _check(g, False, Q, lim, L, filters, qf)


# ---------------------------------------------------------------- 4. flat search, every store, both routes

@pytest.mark.parametrize("scan", [False, True])
@pytest.mark.parametrize("kind", ["f32_tc", "f32", "haversine", "binary", "pq"])
def test_flat_rows_equal_the_existing_entries(kind, scan, monkeypatch):
    g, ids, Q, deleted = _flat(kind)
    if scan:
        monkeypatch.setenv("SDB_FLAT_EXACT", "1")
    rng = np.random.default_rng(3)
    lim, _ = _mix(len(Q), rng, tiny=False)
    _check(g, True, Q, lim, None)
    for name, filters, qf in _batches(rng, ids, len(Q), True, rows=len(ids) + 2, deleted=deleted):
        _check(g, True, Q, lim, None, filters, qf)


# ---------------------------------------------------------------- 5. uniform requests, errors

@pytest.mark.parametrize("flat", [False, True])
def test_uniform_requests_give_the_filter_entry_bytes(flat):
    if flat:
        g, ids, Q, deleted = _flat("f32")
    else:
        g, _, ids, Q = _vamana("l2_128")
    rng = np.random.default_rng(4)
    for name, filters, qf in _batches(rng, ids, len(Q), flat):
        want = g.flat_search_batch_filters(Q, filters, qf, 10) if flat else g.search_batch_filters(Q, filters, qf, 10, 50)
        rq = PackedRequests(len(Q), 10, 50, filters, qf)
        assert _same(want, _device(g, flat, Q, rq, 10)), name
        got = g.flat_search_batch_requests(Q, 10, filters, qf) if flat else g.search_batch_requests(Q, 10, 50, filters, qf)
        assert _same(want, got), name


@pytest.mark.parametrize("flat", [False, True])
def test_errors_leave_the_outputs_untouched(flat):
    import torch
    if flat:
        g, ids, Q, _ = _flat("f32")
    else:
        g, _, ids, Q = _vamana("l2_128", n=2000, B=8)
    Q = Q[:8]
    B = len(Q)
    good = np.sort(ids[:200]).astype(np.uint64)
    # a seed missing within request 1's searchSize (40) but beyond request 0's (25)
    seedy = np.concatenate([ids[:30], ids.max() + 100 + np.arange(50)]).astype(np.uint64)
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(np.ascontiguousarray(Q)).to(dev)

    def call(lim, L, filters=None, qf=None, k_stride=10, raw_filter=None):
        o = (torch.full((B, 10), 7, dtype=torch.int64, device=dev), torch.full((B, 10), 7.0, device=dev),
             torch.full((B,), 7, dtype=torch.int32, device=dev))
        rq = PackedRequests(B, lim, L, filters, qf, default_L=75)
        if raw_filter is not None:
            rq.req["filter"] = raw_filter
        entry = g.flat_search_batch_requests_device if flat else g.search_batch_requests_device
        with pytest.raises(SdbError) as e:
            entry(d_q, rq, k_stride, *o, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert all(bool((t == 7).all().item()) for t in o)  # nothing enqueued
        if raw_filter is not None:  # the host methods pack query_filter themselves
            return e.value.code
        with pytest.raises(SdbError) as e2:  # the host entry refuses the same call
            if flat:
                g.flat_search_batch_requests(Q, lim, filters, qf, k_stride)
            else:
                g.search_batch_requests(Q, lim, L, filters, qf, k_stride)
        assert e2.value.code == e.value.code
        return e.value.code

    lim = np.full(B, 10)
    bad0 = lim.copy()
    bad0[3] = 0
    assert call(bad0, 75) == _capi.ERR_INVALID
    bad76 = lim.copy()
    bad76[2] = 76
    assert call(bad76, 75, k_stride=75) == _capi.ERR_INVALID
    assert call(lim, 75, k_stride=76) == _capi.ERR_INVALID
    big = lim.copy()
    big[5] = 11
    assert call(big, 75) == _capi.ERR_INVALID  # limit > k_stride
    assert call(lim, 75, [good], np.full(B, 1, np.int32)) == _capi.ERR_INVALID  # filter index out of range
    assert call(lim, 75, [good], raw_filter=np.full(B, -5, np.int32)) == _capi.ERR_INVALID  # only -1 means unfiltered
    if not flat:
        L = np.full(B, 75)
        L[4] = 76
        assert call(lim, L) == _capi.ERR_INVALID
        L[4] = 0
        assert call(lim, L) == _capi.ERR_INVALID
        L[4] = 9
        assert call(lim, L) == _capi.ERR_SEARCHSIZE
        L = np.full(B, 25)
        L[1] = 40
        qf = np.zeros(B, np.int32)
        assert call(lim, L, [seedy], qf) == _capi.ERR_NOTFOUND
        L[1] = 25  # every request's seeds exist: the same filter is served
        g.search_batch_requests(Q, lim, L, [seedy], qf)
    # the handle still serves
    _check(g, flat, Q, lim, np.full(B, 75) if not flat else None)


# ---------------------------------------------------------------- 6. sharded: fused gather and merge on one GPU

@pytest.mark.parametrize("flat", [False, True])
def test_fused_gather_and_merge_with_request_limits(flat):
    import torch
    S, dim, n, B = 3, 32, 2500, 60
    Xall = synth.latent_gaussian(S * n, dim, seed=70, latent=8)
    Q = np.ascontiguousarray(synth.latent_gaussian(B, dim, seed=71, w_seed=70, latent=8), np.float32)
    rng = np.random.default_rng(9)
    lim, L = _mix(B, rng, tiny=False)
    KS = int(lim.max())
    shard = np.array([sharded.shard_limit(int(x), S, 75) for x in lim])
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    f = [torch.full((S, B, KS), -1, dtype=torch.int64, device=dev), torch.full((S, B, KS), -1.0, dtype=torch.float32, device=dev),
         torch.full((S, B), -1, dtype=torch.int32, device=dev)]
    o_ids, o_d, o_c = np.zeros((S, B, KS), np.uint64), np.full((S, B, KS), INF, np.float32), np.zeros((S, B), np.uint32)
    for s in range(S):
        X = np.ascontiguousarray(Xall[s * n:(s + 1) * n], np.float32)
        if flat:
            g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
            g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
        else:
            oix, pid, start = oracle_graph(X)
            g = mirror_to_gpu(oix, X, pid, start, relaxed=True)
        pg = _capi.SdbPeerGather()
        pg.n_peers, pg.shard, pg.per_shard_limit = 1, s, 1  # ignored by the request entries
        pg.ids[0], pg.dists[0], pg.counts[0] = f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr()
        rq = PackedRequests(B, lim, L, None, None, shard, default_L=75)
        li, ld, lc = _device(g, flat, Q, rq, KS, pg)
        want = _expect(g, flat, Q, lim, L, None, None, KS)
        assert _same(want, (li, ld, lc))
        o_ids[s] = np.where(ld < INF, li | (np.uint64(s) << np.uint64(40)), np.uint64(0))
        o_d[s], o_c[s] = ld, np.minimum(lc, shard)
    fi, fd, fc = (t.cpu().numpy() for t in f)
    assert (fi.view(np.uint64) == o_ids).all() and fd.tobytes() == o_d.tobytes() and (fc.view(np.uint32) == o_c).all()
    lib = _capi.lib()
    m = [torch.full((B, KS), -1, dtype=torch.int64, device=dev), torch.full((B, KS), -1.0, device=dev),
         torch.full((B,), -1, dtype=torch.int32, device=dev)]
    d_lim = torch.from_numpy(lim.astype(np.int32)).to(dev)
    _capi.check(lib.sdb_merge_topk_requests_device(0, S, B, KS, d_lim.data_ptr(), f[0].data_ptr(), f[1].data_ptr(),
                                                   f[2].data_ptr(), m[0].data_ptr(), m[1].data_ptr(), m[2].data_ptr(), st))
    torch.cuda.synchronize()
    mi, md, mc = (t.cpu().numpy() for t in m)
    oi, od, oc = O.merge_topk(o_ids, o_d, o_c, KS)
    cut = np.arange(KS)[None, :] < lim[:, None]
    assert (mi.view(np.uint64) == np.where(cut, oi, 0)).all()
    assert md.tobytes() == np.where(cut, od, INF).astype(np.float32).tobytes()
    assert (mc.view(np.uint32) == np.minimum(oc, lim)).all()
    # uniform limits: the bytes of sdb_merge_topk_device
    u = [torch.zeros_like(t) for t in m]
    _capi.check(lib.sdb_merge_topk_device(0, S, B, KS, f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr(), u[0].data_ptr(),
                                          u[1].data_ptr(), u[2].data_ptr(), st))
    d_all = torch.full((B,), KS, dtype=torch.int32, device=dev)
    _capi.check(lib.sdb_merge_topk_requests_device(0, S, B, KS, d_all.data_ptr(), f[0].data_ptr(), f[1].data_ptr(),
                                                   f[2].data_ptr(), m[0].data_ptr(), m[1].data_ptr(), m[2].data_ptr(), st))
    torch.cuda.synchronize()
    assert all(bool((x == y).all().item()) for x, y in zip(u, m))


# ---------------------------------------------------------------- 6b. ShardedSearcher on two GPUs

def _searcher_worker(rank, world, port, out_dir):
    import os

    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    dim, n, B = 32, 3000, 120
    X = np.ascontiguousarray(synth.latent_gaussian(world * n, dim, seed=80, latent=8)[rank * n:(rank + 1) * n], np.float32)
    Q = np.ascontiguousarray(synth.latent_gaussian(B, dim, seed=81, w_seed=80, latent=8), np.float32)
    d_q = torch.from_numpy(Q).to(dev)
    lim, L = _mix(B, np.random.default_rng(12), tiny=False)
    KS = int(lim.max())
    res = []
    for flat in (False, True):
        if flat:
            g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"), device=rank)
            g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
        else:
            from semadb_b200.vamana import IndexVamana, IndexVectorVamanaParameters
            oix, pid, start = oracle_graph(X)
            g = IndexVamana("p2p", IndexVectorVamanaParameters(dim, "euclidean"), device=rank, start_vector=start,
                            relaxed=True)
            g.set_vectors(pid.astype(np.uint64), X)
            adj, deg = oix.get_graph()
            g.set_graph_dense(adj[1:], deg[1:], first_id=1)
        a = sharded.ShardedSearcher(g, rank, world, exchange="nccl")
        want = [t.clone() for t in a.search_batch_device(d_q, KS, None, limits=lim, search_sizes=L)]
        b = sharded.ShardedSearcher(g, rank, world, exchange="p2p")
        got = b.search_batch_device(d_q, KS, None, limits=lim, search_sizes=L)
        torch.cuda.synchronize()
        same = all(bool((x == y).all().item()) for x, y in zip(got, want))
        c = sharded.ShardedSearcher(g, rank, world, exchange="p2p", pipeline=True)
        outs = []
        for _ in range(3):
            out = c.search_batch_device(d_q, KS, None, limits=lim, search_sizes=L)
            with torch.cuda.stream(c._side):
                outs.append([t.clone() for t in out])
        c.wait_pipeline()
        torch.cuda.synchronize()
        same_pipe = all(all(bool((x == y).all().item()) for x, y in zip(o, want)) for o in outs)
        cnt_ok = bool((want[2].cpu().numpy() <= lim).all())
        res += [same, same_pipe, cnt_ok]
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), res=np.array(res))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_searcher_requests_two_gpus_match_nccl_path(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from tests.test_sharded_gloo import _free_port
    mp.spawn(_searcher_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for i in range(2):
        assert np.load(tmp_path / f"r{i}.npz")["res"].all()


def test_sharded_searcher_requests_one_gpu_nccl_path():
    """world == 1 through the NCCL-path code: the request entry's rows, counts clamped per request."""
    g, _, _, Q = _vamana("l2_128")
    import torch
    lim, L = _mix(len(Q), np.random.default_rng(13), tiny=False)
    KS = int(lim.max())
    s = sharded.ShardedSearcher(g, 0, 1, exchange="nccl")
    got = [t.cpu().numpy() for t in s.search_batch_device(torch.from_numpy(Q).cuda(), KS, None, limits=lim, search_sizes=L)]
    want = _expect(g, False, Q, lim, L, None, None, KS)
    assert (got[0].view(np.uint64) == want[0]).all() and got[1].tobytes() == want[1].tobytes()
    assert (got[2].view(np.uint32) == want[2]).all()
