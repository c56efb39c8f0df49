"""Sharded search with per-request filters: the filtered device entries
(sdb_search_batch_filters_device, sdb_flat_search_batch_filters_device) against the host filter
entries on every store each serves, their enqueue without a host synchronisation, the reuse of the
handle's staging slots and filter buffers, the fused exchange with every shard on one GPU and
across two GPUs, and the argument errors."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oraclelib as O
from semadb_b200 import _capi, sharded, synth
from semadb_b200._capi import SdbError
from semadb_b200.vamana import (IndexFlat, IndexVectorFlatParameters, IndexVectorVamanaParameters,
                                ProductQuantizerParameters, Quantizer)
from tests.helpers import mirror_to_gpu, oracle_graph

pytestmark = pytest.mark.gpu

N_TC = 70_000  # above the flat tensor-core path's threshold (4 x 16 384 sample points)
K, L = 10, 75


def _outs(B, k, fill=-1):
    import torch
    dev = torch.device("cuda", 0)
    return (torch.full((B, k), fill, dtype=torch.int64, device=dev), torch.full((B, k), float(fill), dtype=torch.float32, device=dev),
            torch.full((B,), fill, dtype=torch.int32, device=dev))


def _np(outs):
    i, d, c = (t.cpu().numpy() for t in outs)
    return i.view(np.uint64), d, c.view(np.uint32)


def _same(a, b):
    return all(x.tobytes() == y.tobytes() for x, y in zip(a, b))


def _host(g, flat, Q, filters, qf, k=K):
    if flat:
        return g.flat_search_batch_filters(Q, filters, qf, k)
    return g.search_batch_filters(Q, filters, qf, k, L)


def _enqueue(g, flat, d_q, filters, qf, o, stream, k=K, peers=None):
    if flat:
        g.flat_search_batch_filters_device(d_q, filters, qf, k, *o, stream, peers)
    else:
        g.search_batch_filters_device(d_q, filters, qf, k, L, *o, stream, peers)


def _device(g, flat, Q, filters, qf, k=K):
    import torch
    d_q = torch.from_numpy(np.ascontiguousarray(Q)).cuda()
    o = _outs(len(Q), k)
    _enqueue(g, flat, d_q, filters, qf, o, torch.cuda.current_stream().cuda_stream, k)
    torch.cuda.synchronize()
    return _np(o)


def _batches(rng, ids, B, flat, rows=0, deleted=()):
    """(name, filters, query_filter) batch shapes: one shared filter, per-request filters with an
    empty one, a mixed batch with unfiltered requests; for flat search also lists naming deleted
    ids, ids beyond the store and ids 0 and 1, and filters of more than 1 024 ids."""
    pick = lambda m: np.sort(rng.choice(ids, size=min(m, len(ids)), replace=False)).astype(np.uint64)
    per = [pick(m) for m in (1, 40, 75, 76, 500, 2500)] + [np.zeros(0, np.uint64)]
    out = [("shared", [pick(600)], None),
           ("per_request", per, np.arange(B, dtype=np.int32) % len(per)),
           ("mixed", per, (np.arange(B, dtype=np.int32) % (len(per) + 2)) - 2)]
    if flat:
        odd = [np.union1d(pick(30), np.asarray(deleted, np.uint64)),
               np.union1d(pick(20), np.array([rows + 7, rows * 4 + 3, 1 << 40], np.uint64)),
               np.union1d(pick(K), np.array([0, 1], np.uint64)), pick(1500), pick(5000)]
        out.append(("odd_and_chunked", [f.astype(np.uint64) for f in odd], np.arange(B, dtype=np.int32) % len(odd) - (np.arange(B) % 7 == 0)))
    return out


def _check_all(g, flat, Q, batches):
    for name, filters, qf in batches:
        h = _host(g, flat, Q, filters, qf)
        d = _device(g, flat, Q, filters, qf)
        assert _same(h, d), name
    # n_filters == 0: the bytes of the unfiltered device entry
    import torch
    d_q = torch.from_numpy(np.ascontiguousarray(Q)).cuda()
    u = _outs(len(Q), K)
    st = torch.cuda.current_stream().cuda_stream
    if flat:
        g.flat_search_batch_device(d_q, K, *u, st)
    else:
        g.search_batch_device(d_q, K, L, *u, st)
    torch.cuda.synchronize()
    assert _same(_np(u), _device(g, flat, Q, [], None))


# ---------------------------------------------------------------- 1. device entry = host entry, Vamana

def _vamana(kind):
    if kind == "l2_128":
        X, Q = synth.sift_shaped(3000, 128, 3), synth.sift_shaped(96, 128, 4, w_seed=3)
        metric, quant = "euclidean", None
    elif kind == "l2_40":
        X, Q = synth.uniform(3000, 40, 7), synth.uniform(96, 40, 8)
        metric, quant = "euclidean", None
    elif kind in ("dot", "cosine"):
        X = synth.latent_gaussian(3000, 64, seed=11, latent=8, normalize=(kind == "cosine"))
        Q = synth.latent_gaussian(96, 64, seed=12, w_seed=11, latent=8, normalize=(kind == "cosine"))
        metric, quant = kind, None
    elif kind == "haversine":
        X, Q = synth.geo_points(3000, 5), synth.geo_points(96, 6, background=1.0)
        metric, quant = "haversine", None
    elif kind == "bq":
        X = synth.planted_bits(3000, 256, seed=7, n_proto=64)
        Q = synth.planted_bits(96, 256, seed=10, n_proto=64, proto_seed=7)
        metric, quant = "hamming", None
    else:  # pq
        X = synth.latent_gaussian(3000, 64, seed=41, latent=8)
        Q = synth.latent_gaussian(96, 64, seed=42, w_seed=41, latent=8)
        metric, quant = "euclidean", Quantizer("product", product=ProductQuantizerParameters(64, 8, 1000))
    X, Q = np.ascontiguousarray(X, np.float32), np.ascontiguousarray(Q, np.float32)
    oix, pid, start = oracle_graph(X, metric)
    g = mirror_to_gpu(oix, X, pid, start, metric, quantizer=quant)
    if quant is not None:
        assert g.fit(0) is True
    return g, pid, Q


@pytest.mark.parametrize("kind", ["l2_128", "l2_40", "dot", "cosine", "haversine", "bq", "pq"])
def test_vamana_device_entry_equals_host_entry(kind):
    g, pid, Q = _vamana(kind)
    _check_all(g, False, Q, _batches(np.random.default_rng(1), pid, len(Q), False))


def test_vamana_retry_launch_device_entry_equals_host_entry(monkeypatch):
    g, pid, Q = _vamana("l2_128")
    monkeypatch.setenv("SDB_VT_SLOTS", "64")  # every query overflows its visited table: RETRY launch
    _check_all(g, False, Q, _batches(np.random.default_rng(2), pid, len(Q), False))


# ---------------------------------------------------------------- 1. device entry = host entry, flat

def _flat(kind):
    if kind in ("f32_tc", "f32"):
        n = N_TC if kind == "f32_tc" else 3000
        X = synth.latent_gaussian(n, 96, seed=5, latent=8)
        Q = synth.latent_gaussian(96, 96, seed=6, w_seed=5, latent=8)
        g = IndexFlat(IndexVectorFlatParameters(96, "euclidean"))
    elif kind == "haversine":
        n = 5000
        X, Q = synth.geo_points(n, 5), synth.geo_points(96, 6, background=1.0)
        g = IndexFlat(IndexVectorFlatParameters(2, "haversine"))
    elif kind == "binary":
        n = 3000
        X = synth.planted_bits(n, 256, seed=7, n_proto=32)
        Q = synth.planted_bits(96, 256, seed=8, n_proto=32)
        g = IndexFlat(IndexVectorFlatParameters(256, "hamming"))
    else:  # pq
        n = 3000
        X = synth.latent_gaussian(n, 64, seed=21, latent=8)
        Q = synth.latent_gaussian(96, 64, seed=22, w_seed=21, latent=8)
        g = IndexFlat(IndexVectorFlatParameters(64, "euclidean", Quantizer("product", product=ProductQuantizerParameters(64, 16, 1000))))
    ids = np.arange(2, n + 2, dtype=np.uint64)
    g.set_vectors(ids, np.ascontiguousarray(X, np.float32))
    if kind == "pq":
        assert g.fit(3) is True
    deleted = ids[5:400:13]
    g.delete_rows(deleted)
    return g, ids, np.ascontiguousarray(Q, np.float32), deleted


@pytest.mark.parametrize("scan", [False, True])
@pytest.mark.parametrize("kind", ["f32_tc", "f32", "haversine", "binary", "pq"])
def test_flat_device_entry_equals_host_entry(kind, scan, monkeypatch):
    g, ids, Q, deleted = _flat(kind)
    if scan:
        monkeypatch.setenv("SDB_FLAT_EXACT", "1")  # every filter through the range scan
    batches = _batches(np.random.default_rng(3), ids, len(Q), True, rows=len(ids) + 2, deleted=deleted)
    _check_all(g, True, Q, batches)
    g.flat_search_batch_filters(Q, batches[-1][1], batches[-1][2])
    gathered, scanned, _ = g.flat_last_filter_stats()
    assert scanned > 0 if scan else gathered > 0


def test_scan_route_filter_stages_only_its_ids():
    """A filter shared by a large batch takes the range scan and needs no gather work items: the
    staging the handle keeps stays near the size of the id list, whatever the batch size."""
    import torch
    g, ids, _, _ = _flat("f32_tc")
    B = 4000
    Q = np.ascontiguousarray(synth.latent_gaussian(B, 96, seed=7, w_seed=5, latent=8), np.float32)
    filt = np.sort(np.random.default_rng(8).choice(ids, size=len(ids) // 2, replace=False))
    want = g.flat_search_batch(Q, K, filt)  # the single-filter host entry
    assert g.flat_last_filter_stats()[1] == 1  # range scan
    assert _same(want, _device(g, True, Q, [filt], None))
    pinned, device = g.filter_staging_bytes()
    slot = 4 * len(filt) + 12 * B + 256  # ids, offsets, request rows and gather requests of one slot
    assert pinned <= 2 * (1.25 * slot + 64), (pinned, slot)  # two slots, grow-only capacity
    assert device <= 1.25 * slot + 64, (device, slot)


# ---------------------------------------------------------------- 2. no host synchronisation

def _no_sync(g, flat, Q, filters, qf):
    import torch
    want = _host(g, flat, Q, filters, qf)
    side = torch.cuda.Stream()
    d_q = torch.from_numpy(Q).cuda()
    o = _outs(len(Q), K)
    for _ in range(2):  # same shapes through both staging slots: scratch is allocated
        _enqueue(g, flat, d_q, filters, qf, o, side.cuda_stream)
    side.synchronize()
    for t in o:
        t.fill_(-1)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # ~0.1 s of device time in front of the search
    _enqueue(g, flat, d_q, filters, qf, o, side.cuda_stream)
    assert side.query() is False  # the call returned while the stream was still busy
    side.synchronize()
    assert _same(want, _np(o))


@pytest.mark.parametrize("shape", ["per_request", "mixed"])
def test_vamana_device_entry_does_not_synchronise(shape):
    g, pid, Q = _vamana("l2_128")
    rng = np.random.default_rng(4)
    filters = [np.sort(rng.choice(pid, size=m, replace=False)) for m in (2000, 2500, 2999)]
    qf = np.arange(len(Q), dtype=np.int32) % 3 - (1 if shape == "mixed" else 0)
    _no_sync(g, False, Q, filters, qf)


@pytest.mark.parametrize("route", ["gather", "scan"])
def test_flat_device_entry_does_not_synchronise(route, monkeypatch):
    g, ids, Q, _ = _flat("f32_tc")
    rng = np.random.default_rng(5)
    if route == "scan":
        monkeypatch.setenv("SDB_FLAT_EXACT", "1")
    filters = [np.sort(rng.choice(ids, size=m, replace=False)) for m in (3000, 4500)]
    _no_sync(g, True, Q, filters, np.arange(len(Q), dtype=np.int32) % 3 - 1)  # a mixed batch


# ---------------------------------------------------------------- 3. staging reuse

@pytest.mark.parametrize("flat", [False, True])
def test_back_to_back_calls_and_a_host_call_between(flat):
    import torch
    if flat:
        g, ids, Q, _ = _flat("f32_tc")
    else:
        g, ids, Q = _vamana("l2_128")
    rng = np.random.default_rng(6)
    steps = []
    for i in range(8):
        filters = [np.sort(rng.choice(ids, size=int(m), replace=False)) for m in rng.integers(100, 2500, 1 + i % 3)]
        qf = rng.integers(-1, len(filters), len(Q)).astype(np.int32)
        steps.append((filters, qf, _host(g, flat, Q, filters, qf)))
    side = torch.cuda.Stream()
    d_q = torch.from_numpy(Q).cuda()
    outs = [_outs(len(Q), K) for _ in steps]
    _enqueue(g, flat, d_q, steps[0][0], steps[0][1], outs[0], side.cuda_stream)  # shapes warmed up
    side.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
    for (filters, qf, _), o in zip(steps, outs):
        _enqueue(g, flat, d_q, filters, qf, o, side.cuda_stream)
    side.synchronize()
    for (_, _, want), o in zip(steps, outs):
        assert _same(want, _np(o))
    # a host filtered call while a device filtered call is still queued on another stream
    o = _outs(len(Q), K)
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
    _enqueue(g, flat, d_q, steps[1][0], steps[1][1], o, side.cuda_stream)
    got = _host(g, flat, Q, steps[2][0], steps[2][1])
    side.synchronize()
    assert _same(steps[1][2], _np(o)) and _same(steps[2][2], got)


# ---------------------------------------------------------------- 4. fused gather, every shard on one GPU

def _pred_lists(global_ids, local_ids, n_pred=4):
    """Shard-local lists of n_pred global predicates (a hash of the global point index)."""
    h = (global_ids.astype(np.uint64) * np.uint64(2654435761)) >> np.uint64(7)
    return [np.sort(local_ids[(h % np.uint64(7)) == np.uint64(j)]).astype(np.uint64) for j in range(n_pred)]


def _publish(g, flat, d_q, filters, qf, l, f, shard, limit, st):
    pg = _capi.SdbPeerGather()
    pg.n_peers, pg.shard, pg.per_shard_limit = 1, shard, limit
    pg.ids[0], pg.dists[0], pg.counts[0] = f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr()
    _enqueue(g, flat, d_q, filters, qf, l, st, peers=pg)


@pytest.mark.parametrize("flat", [False, True])
def test_fused_gather_single_gpu(flat):
    import torch
    S, dim, n = 3, 32, 2500
    Xall = synth.latent_gaussian(S * n, dim, seed=70, latent=8)
    Q = np.ascontiguousarray(synth.latent_gaussian(60, dim, seed=71, w_seed=70, latent=8), np.float32)
    B = len(Q)
    qf = (np.arange(B, dtype=np.int32) % 5) - 1  # predicate qf[b], -1 = unfiltered on every shard
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_q = torch.from_numpy(Q).to(dev)
    f = [torch.full((S, B, K), -1, dtype=torch.int64, device=dev), torch.full((S, B, K), -1.0, dtype=torch.float32, device=dev),
         torch.full((S, B), -1, dtype=torch.int32, device=dev)]
    loc = []
    o_ids, o_d, o_c = np.zeros((S, B, K), np.uint64), np.zeros((S, B, K), np.float32), np.zeros((S, B), np.uint32)
    keep, lists_of = [], []
    for s in range(S):
        X = np.ascontiguousarray(Xall[s * n:(s + 1) * n], np.float32)
        local = np.arange(2, n + 2, dtype=np.uint64)
        lists = _pred_lists(np.arange(s * n, (s + 1) * n), local)
        lists_of.append(lists)
        if flat:
            g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
            g.set_vectors(local, X)
            oix = O.OracleIndex(dim, "euclidean")
            oix.set_vectors(local.astype(np.uint32), X)
        else:
            oix, pid, start = oracle_graph(X)
            g = mirror_to_gpu(oix, X, pid, start)
        keep.append(g)
        u = _outs(B, K)
        _enqueue(g, flat, d_q, lists, qf, u, st)
        l = _outs(B, K)
        _publish(g, flat, d_q, lists, qf, l, f, s, 0, st)
        torch.cuda.synchronize()
        assert _same(_np(u), _np(l))
        loc.append(_np(u))
        for b in range(B):
            fl = None if qf[b] < 0 else lists[qf[b]].astype(np.uint32)
            if flat:
                r = oix.flat_search(Q[b:b + 1], k=K, filter_ids=fl, threads=1)
            else:
                r = oix.search(Q[b:b + 1], k=K, search_size=L, filter_ids=fl, threads=1)
            c = int(r["counts"][0])
            o_ids[s, b, :c] = sharded.pack_global_ids(r["ids"][0, :c].astype(np.uint64), s)
            o_d[s, b], o_c[s, b] = r["dists"][0], c
    fi, fd, fc = _np(f)
    for s in range(S):  # the published slots: the local outputs tagged with the shard
        li, ld, lc = loc[s]
        tagged = np.where(np.arange(K)[None, :] < lc[:, None], li | (np.uint64(s) << np.uint64(40)), np.uint64(0))
        assert (fi[s] == tagged).all() and fd[s].tobytes() == ld.tobytes() and (fc[s] == lc).all()
    assert (fi == o_ids).all() and fd.tobytes() == o_d.tobytes() and (fc == o_c).all()
    # per-shard limit below k clamps the published counts only
    l = _outs(B, K)
    _publish(keep[1], flat, d_q, lists_of[1], qf, l, f, 1, 4, st)
    torch.cuda.synchronize()
    assert (_np(f)[2][1] == np.minimum(fc[1], 4)).all() and (_np(l)[2] == fc[1]).all()
    assert _np(f)[0][1].tobytes() == fi[1].tobytes() and _np(f)[1][1].tobytes() == fd[1].tobytes()
    _publish(keep[1], flat, d_q, lists_of[1], qf, l, f, 1, 0, st)
    # barrier + merge = the oracle chain
    lib = _capi.lib()
    flags = torch.zeros((64,), dtype=torch.int32, device=dev)
    _capi.check(lib.sdb_peer_barrier_device(0, 1, 0, (C.c_void_p * 1)(flags.data_ptr()), 1, st))
    m = list(_outs(B, K))
    _capi.check(lib.sdb_merge_topk_device(0, S, B, K, f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr(), m[0].data_ptr(),
                                          m[1].data_ptr(), m[2].data_ptr(), st))
    torch.cuda.synchronize()
    mi, md, mc = _np(m)
    oi, od, oc = O.merge_topk(o_ids, o_d, o_c, K)
    assert (mi == oi).all() and md.tobytes() == od.tobytes() and (mc == oc).all()
    if flat:  # one index over the union, filtered by the global predicates
        gu = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
        gu.set_vectors(np.arange(2, S * n + 2, dtype=np.uint64), np.ascontiguousarray(Xall, np.float32))
        ul = _pred_lists(np.arange(S * n), np.arange(2, S * n + 2, dtype=np.uint64))
        ui, ud, uc = gu.flat_search_batch_filters(Q, ul, qf, K)
        assert md.tobytes() == ud.tobytes() and (mc == uc).all()


# ---------------------------------------------------------------- 5. two GPUs, one process each

def _p2p_worker(rank, world, port, out_dir):
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
    local = np.arange(2, n + 2, dtype=np.uint64)
    lists = _pred_lists(np.arange(rank * n, (rank + 1) * n), local, 6)
    steps = [(np.roll(np.arange(-1, 6), i)[np.arange(B) % 7].astype(np.int32), torch.roll(d_q, 5 * i, 0).contiguous())
             for i in range(6)]
    res = {}
    for flat in (False, True):
        if flat:
            g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"), device=rank)
            g.set_vectors(local, X)
        else:
            oix, pid, start = oracle_graph(X)
            params = IndexVectorVamanaParameters(dim, "euclidean")
            from semadb_b200.vamana import IndexVamana
            g = IndexVamana("p2p", params, device=rank, start_vector=start)
            g.set_vectors(pid.astype(np.uint64), X)
            adj, deg = oix.get_graph()
            g.set_graph_dense(adj[1:], deg[1:], first_id=1)
        a = sharded.ShardedSearcher(g, rank, world, exchange="nccl")
        want = [[t.clone() for t in a.search_batch_device(q, K, None, filters=lists, query_filter=qf)] for qf, q in steps]
        b = sharded.ShardedSearcher(g, rank, world, exchange="p2p")
        same = True
        for (qf, q), w in zip(steps, want):
            got = b.search_batch_device(q, K, None, filters=lists, query_filter=qf)
            torch.cuda.synchronize()
            same = same and all(bool((x == y).all().item()) for x, y in zip(got, w))
        h_q = torch.from_numpy(Q).pin_memory()
        h = [torch.zeros((B, K), dtype=torch.int64).pin_memory(), torch.zeros((B, K), dtype=torch.float32).pin_memory(),
             torch.zeros((B,), dtype=torch.int32).pin_memory()]
        b.search_batch_pinned(h_q, K, None, *h, dev, filters=lists, query_filter=steps[0][0])
        same = same and all(bool((x == y.cpu()).all()) for x, y in zip(h, want[0]))
        c = sharded.ShardedSearcher(g, rank, world, exchange="p2p", pipeline=True)
        got_p = []
        for qf, q in steps:  # every step with other filters, no wait in between: steps overlap
            out = c.search_batch_device(q, K, None, filters=lists, query_filter=qf)
            with torch.cuda.stream(c._side):  # the merged lists of a step are final on the exchange stream
                got_p.append([t.clone() for t in out])
        c.wait_pipeline()
        torch.cuda.synchronize()
        same_pipe = all(all(bool((x == y).all().item()) for x, y in zip(gp, w)) for gp, w in zip(got_p, want))
        failed = b._peer.barrier_failed() or c._peer.barrier_failed()
        res[f"{'flat' if flat else 'vamana'}"] = (same, same_pipe, failed)
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), res=np.array([v for k_ in sorted(res) for v in res[k_]]))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_searcher_filters_two_gpus_match_nccl_path(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from tests.test_sharded_gloo import _free_port
    mp.spawn(_p2p_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for i in range(2):
        r = np.load(tmp_path / f"r{i}.npz")["res"].reshape(2, 3)
        assert r[:, 0].all() and r[:, 1].all() and not r[:, 2].any()


# ---------------------------------------------------------------- 6. errors leave the handle usable

@pytest.mark.parametrize("flat", [False, True])
def test_errors_leave_the_handle_usable(flat):
    import torch
    if flat:
        g, ids, Q, _ = _flat("f32")
    else:
        g, ids, Q = _vamana("l2_40")
    B = len(Q)
    rng = np.random.default_rng(9)
    good = [np.sort(rng.choice(ids, size=m, replace=False)) for m in (80, 1200)]
    good_qf = np.arange(B, dtype=np.int32) % 3 - 1
    want_f = _host(g, flat, Q, good, good_qf)
    want_u = _device(g, flat, Q, [], None)
    lib = _capi.lib()
    st = torch.cuda.current_stream().cuda_stream
    d_q = torch.from_numpy(Q).cuda()
    peer = _outs(B, 76)

    def pg_of(n_peers, null_peer=False):
        pg = _capi.SdbPeerGather()
        pg.n_peers, pg.shard, pg.per_shard_limit = n_peers, 0, 0
        for p in range(min(n_peers, _capi.MAX_PEERS)):
            pg.ids[p], pg.dists[p], pg.counts[p] = peer[0].data_ptr(), peer[1].data_ptr(), peer[2].data_ptr()
        if null_peer:
            pg.dists[0] = None
        return pg

    def call(filters, qf, k=K, search_size=L, pg=None):
        # packed as given (the Python layer sorts each list)
        ids_ = np.ascontiguousarray(np.concatenate(filters), np.uint64)
        off = np.zeros(len(filters) + 1, np.uint64)
        off[1:] = np.cumsum([len(f) for f in filters])
        qf_ = None if qf is None else np.ascontiguousarray(qf, np.int32)
        fa = (len(filters), ids_.ctypes.data_as(_capi.u64p), off.ctypes.data_as(_capi.u64p),
              None if qf_ is None else qf_.ctypes.data_as(_capi.i32p))
        o = _outs(B, 76)
        ptrs = [t.data_ptr() for t in o]
        if flat:
            return lib.sdb_flat_search_batch_filters_device(g._h, B, d_q.data_ptr(), k, *fa, *ptrs, pg, st)
        return lib.sdb_search_batch_filters_device(g._h, B, d_q.data_ptr(), k, search_size, *fa, *ptrs, pg, st)

    def expect(code, rc):
        assert rc == code
        assert _same(want_u, _device(g, flat, Q, [], None))
        assert _same(want_f, _device(g, flat, Q, good, good_qf))

    unsorted = good[1][::-1].copy()
    expect(_capi.ERR_INVALID, call([good[0], unsorted], good_qf))
    expect(_capi.ERR_INVALID, call(good, np.full(B, 2, np.int32)))
    if flat:
        for k in (0, 76):
            expect(_capi.ERR_INVALID, call(good, good_qf, k=k))
    else:
        missing = np.union1d(good[0][:10], [len(ids) + 50]).astype(np.uint64)  # a seed that is not stored
        expect(_capi.ERR_NOTFOUND, call([missing], None))
        expect(_capi.ERR_SEARCHSIZE, call(good, good_qf, k=30, search_size=25))
    for n_peers in (0, 17):
        expect(_capi.ERR_INVALID, call(good, good_qf, pg=C.byref(pg_of(n_peers))))
    expect(_capi.ERR_INVALID, call(good, good_qf, pg=C.byref(pg_of(1, True))))
    # an error half-way through the ids, after a failed call on each slot: both slots still work
    for _ in range(3):
        expect(_capi.ERR_INVALID, call([good[1], unsorted], np.zeros(B, np.int32)))
    with pytest.raises(SdbError):
        _enqueue(g, flat, d_q, good, np.full(B, 5, np.int32), _outs(B, K), st)
    assert _same(want_f, _device(g, flat, Q, good, good_qf))
