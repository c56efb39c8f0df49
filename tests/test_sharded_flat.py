"""Sharded flat search: the device entry (sdb_flat_search_batch_device) against the host entry on
every store the flat search serves, the device-side overflow fallback without a host
synchronisation, the gather entry (sdb_flat_search_batch_gather_device) with every shard on one
GPU and across two GPUs, and the argument errors."""
import ctypes as C

import numpy as np
import pytest

from oracle import oraclelib as O
from semadb_b200 import _capi, sharded, synth
from semadb_b200._capi import SdbError
from semadb_b200.vamana import (IndexFlat, IndexVamana, IndexVectorFlatParameters, IndexVectorVamanaParameters,
                                ProductQuantizerParameters, Quantizer)

pytestmark = pytest.mark.gpu

N_TC = 70_000  # above the tensor-core path's threshold (4 x 16 384 sample points)


def _outs(B, k, fill=-1):
    import torch
    dev = torch.device("cuda", 0)
    return (torch.full((B, k), fill, dtype=torch.int64, device=dev), torch.full((B, k), float(fill), dtype=torch.float32, device=dev),
            torch.full((B,), fill, dtype=torch.int32, device=dev))


def _np(outs):
    i, d, c = (t.cpu().numpy() for t in outs)
    return i.view(np.uint64), d, c.view(np.uint32)


def _device(g, Q, k, stream=None):
    import torch
    st = torch.cuda.current_stream() if stream is None else stream
    d_q = torch.from_numpy(np.ascontiguousarray(Q)).cuda()
    o = _outs(len(Q), k)
    g.flat_search_batch_device(d_q, k, *o, st.cuda_stream)
    torch.cuda.synchronize()
    return _np(o)


def _same(a, b):
    return all(x.tobytes() == y.tobytes() for x, y in zip(a, b))


def _near_copies(n, dim, n_base, seed, copies_of=None):
    """n points, the first `copies_of` (all by default) near-copies of n_base vectors: every query near
    one of them has thousands of points within the bf16 error bound of its k-th distance."""
    rng = np.random.default_rng(seed)
    X = synth.latent_gaussian(n, dim, seed=seed, latent=8) * np.float32(4.0)
    base = rng.normal(size=(n_base, dim)).astype(np.float32)
    m = n if copies_of is None else copies_of
    X[:m] = base[np.arange(m) % n_base] + rng.normal(size=(m, dim)).astype(np.float32) * np.float32(1e-4)
    return X.astype(np.float32), base


def _near_queries(base, B, seed):
    rng = np.random.default_rng(seed)
    return (base[rng.integers(0, len(base), B)] + rng.normal(size=(B, base.shape[1])).astype(np.float32) * np.float32(1e-3)).astype(np.float32)


# ---------------------------------------------------------------- 1. device entry = host entry

@pytest.mark.parametrize("metric,dim,n", [("euclidean", 128, N_TC), ("dot", 96, N_TC), ("cosine", 384, N_TC),
                                          ("euclidean", 128, 3000), ("dot", 96, 3000), ("cosine", 384, 3000)])
def test_device_entry_equals_host_entry_f32(metric, dim, n):
    X = synth.latent_gaussian(n, dim, seed=dim, latent=8, normalize=(metric == "cosine"))
    X[n // 2:n // 2 + 100] = X[:100]  # exact duplicates: ties by ascending id
    Q = np.concatenate([synth.latent_gaussian(300, dim, seed=dim + 1, w_seed=dim, latent=8, normalize=(metric == "cosine")), X[:20]])
    g = IndexFlat(IndexVectorFlatParameters(dim, metric))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    for k in (1, 10, 75):
        h = g.flat_search_batch(Q, k)
        ph = g.flat_last_stats()
        d = _device(g, Q, k)
        assert _same(h, d)
        assert g.flat_last_stats() == ph
        assert ph[0] == (2 if n == N_TC else 0)


def test_device_entry_equals_host_entry_haversine():
    n = 5000
    rng = np.random.Generator(np.random.PCG64(3))
    X = np.stack([rng.uniform(-80, 80, n), rng.uniform(-179, 179, n)], axis=1).astype(np.float32)
    Q = np.stack([rng.uniform(-80, 80, 200), rng.uniform(-179, 179, 200)], axis=1).astype(np.float32)
    g = IndexFlat(IndexVectorFlatParameters(2, "haversine"))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    for k in (1, 10, 75):
        assert _same(g.flat_search_batch(Q, k), _device(g, Q, k))


def test_device_entry_equals_host_entry_binary_and_pq():
    n, dim = 3000, 256
    X = synth.planted_bits(n, dim, seed=7, n_proto=32)
    Q = synth.planted_bits(100, dim, seed=8, n_proto=32)
    b = IndexVamana("bq", IndexVectorVamanaParameters(dim, "hamming"), start_vector=synth.start_vector(dim, 5))
    b.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    for k in (1, 10, 75):
        assert _same(b.flat_search_batch(Q, k), _device(b, Q, k))
    dim, M, K = 64, 16, 64
    X = synth.latent_gaussian(n, dim, seed=21, latent=8)
    Q = synth.latent_gaussian(100, dim, seed=22, w_seed=21, latent=8)
    p = IndexVamana("pq", IndexVectorVamanaParameters(dim, "euclidean", quantizer=Quantizer(
        "product", product=ProductQuantizerParameters(K, M, 1000))), start_vector=synth.start_vector(dim, 5))
    p.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    assert p.fit(3) is True
    for k in (1, 10, 75):
        assert _same(p.flat_search_batch(Q, k), _device(p, Q, k))


@pytest.mark.parametrize("share", ["all", "few", "many"])
def test_device_entry_overflow_equals_host_entry(share):
    """Queries whose candidate lists overflow go to the exact scan on the device: the same lists as the
    host entry and as the exact scan, and flat_last_stats reports them after the device call too.
    all: the near-duplicate shape of test_flat_tc_overflow_falls_back_to_exact_scan; few / many: a
    store with one cluster of near-copies, a few / most queries near it."""
    import os
    dim, B = 96, 300
    if share == "all":
        X, base = _near_copies(N_TC, dim, 7, seed=11)
        Q = _near_queries(base, 200, seed=12)
    else:
        X, base = _near_copies(N_TC, dim, 1, seed=13, copies_of=12_000)
        Q = synth.latent_gaussian(B, dim, seed=14, w_seed=13, latent=8) * np.float32(4.0)
        m = 6 if share == "few" else 250
        Q[:m] = _near_queries(base, m, seed=15)
        Q = np.ascontiguousarray(np.random.default_rng(16).permutation(Q)).astype(np.float32)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(np.arange(2, N_TC + 2, dtype=np.uint64), X)
    h = g.flat_search_batch(Q, 10)
    ph, ch, oh = g.flat_last_stats()
    d = _device(g, Q, 10)
    pd, cd, od = g.flat_last_stats()
    assert _same(h, d) and (ph, ch, oh) == (pd, cd, od) and ph == 2
    if share == "all":
        assert od > 0
    elif share == "few":
        assert 0 < od < len(Q) // 4
    else:
        assert od >= len(Q) // 2
    os.environ["SDB_FLAT_EXACT"] = "1"
    try:
        e = g.flat_search_batch(Q, 10)
    finally:
        os.environ.pop("SDB_FLAT_EXACT", None)
    assert _same(h, e)


def test_device_entry_reads_page_locked_queries():
    import torch
    n, dim = N_TC, 128
    X, Q = synth.sift_shaped(n, dim, 3), synth.sift_shaped(200, dim, 4, w_seed=3)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    h_q = torch.from_numpy(Q).pin_memory()
    o = _outs(len(Q), 10)
    g.flat_search_batch_device(h_q, 10, *o, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert _same(g.flat_search_batch(Q, 10), _np(o))


# ---------------------------------------------------------------- 2. no host synchronisation

@pytest.mark.parametrize("shape", ["overflow", "tensor_core"])
def test_device_entry_does_not_synchronise(shape):
    import torch
    dim = 96
    if shape == "overflow":
        X, base = _near_copies(N_TC, dim, 7, seed=11)
        Q = _near_queries(base, 200, seed=12)
    else:
        X = synth.latent_gaussian(N_TC, dim, seed=5, latent=8)
        Q = synth.latent_gaussian(200, dim, seed=6, w_seed=5, latent=8)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(np.arange(2, N_TC + 2, dtype=np.uint64), X)
    want = g.flat_search_batch(Q, 10)
    side = torch.cuda.Stream()
    d_q = torch.from_numpy(Q).cuda()
    o = _outs(len(Q), 10)
    g.flat_search_batch_device(d_q, 10, *o, side.cuda_stream)  # same shapes once: scratch is allocated
    side.synchronize()
    for t in o:
        t.fill_(-1)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # ~0.1 s of device time in front of the search
    g.flat_search_batch_device(d_q, 10, *o, side.cuda_stream)
    assert side.query() is False  # the call returned while the stream was still busy
    side.synchronize()
    assert _same(want, _np(o))
    if shape == "overflow":
        assert g.flat_last_stats()[2] > 0


# ---------------------------------------------------------------- 3. fused gather, every shard on one GPU

def _shards(dim=96):
    """Three flat shards of one collection (rows in shard order): one below the tensor-core
    threshold, one with a cluster of near-copies whose queries overflow, one ordinary."""
    X0 = synth.latent_gaussian(3000, dim, seed=40, latent=8) * np.float32(4.0)
    X1, base = _near_copies(N_TC, dim, 1, seed=41, copies_of=12_000)
    X2 = synth.latent_gaussian(N_TC, dim, seed=42, latent=8) * np.float32(4.0)
    Q = synth.latent_gaussian(240, dim, seed=43, w_seed=42, latent=8) * np.float32(4.0)
    Q[::8] = _near_queries(base, len(Q[::8]), seed=44)
    return [X0.astype(np.float32), X1, X2.astype(np.float32)], np.ascontiguousarray(Q, dtype=np.float32)


def _publish(g, d_q, k, l, f, shard, limit, st):
    pg = _capi.SdbPeerGather()
    pg.n_peers, pg.shard, pg.per_shard_limit = 1, shard, limit
    pg.ids[0], pg.dists[0], pg.counts[0] = f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr()
    _capi.check(_capi.lib().sdb_flat_search_batch_gather_device(g._h, d_q.shape[0], d_q.data_ptr(), k, l[0].data_ptr(),
                                                                l[1].data_ptr(), l[2].data_ptr(), C.byref(pg), st))
    return pg


def test_fused_gather_matches_device_entry_and_oracle_single_gpu():
    import torch
    Xs, Q = _shards()
    S, B, k, dim = len(Xs), len(Q), 10, Q.shape[1]
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_q = torch.from_numpy(Q).to(dev)
    lib = _capi.lib()
    u = [torch.zeros((S, B, k), dtype=torch.int64, device=dev), torch.zeros((S, B, k), dtype=torch.float32, device=dev),
         torch.zeros((S, B), dtype=torch.int32, device=dev)]
    f = [torch.full((S, B, k), -1, dtype=torch.int64, device=dev), torch.full((S, B, k), -1.0, dtype=torch.float32, device=dev),
         torch.full((S, B), -1, dtype=torch.int32, device=dev)]
    l = list(_outs(B, k))
    o_ids, o_d, o_c = np.zeros((S, B, k), np.uint64), np.zeros((S, B, k), np.float32), np.zeros((S, B), np.uint32)
    keep, overflowed = [], []
    for s, X in enumerate(Xs):
        g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
        g.set_vectors(np.arange(2, len(X) + 2, dtype=np.uint64), X)
        keep.append(g)
        g.flat_search_batch_device(d_q, k, u[0][s], u[1][s], u[2][s], st)
        u[0][s] = sharded.pack_global_ids(u[0][s], s)
        _publish(g, d_q, k, l, f, s, 0, st)
        overflowed.append(g.flat_last_stats()[2])
        oix = O.OracleIndex(dim, "euclidean")
        oix.set_vectors(np.arange(2, len(X) + 2, dtype=np.uint32), X)
        ref = oix.flat_search(Q, k=k, threads=8)
        o_ids[s] = sharded.pack_global_ids(ref["ids"].astype(np.uint64), s)
        o_d[s] = ref["dists"]
        o_c[s] = ref["counts"]
    torch.cuda.synchronize()
    assert overflowed[1] > 0 and keep[0].flat_last_stats()[0] == 0
    assert _same(_np(f), _np(u))
    assert (_np(u)[0] == o_ids).all() and _np(u)[1].tobytes() == o_d.tobytes() and (_np(u)[2] == o_c).all()
    # per-shard limit below k clamps the published counts only (cluster/actions.go:291-299)
    cnt = _np(u)[2]
    _publish(keep[1], d_q, k, l, f, 1, 4, st)
    torch.cuda.synchronize()
    assert (_np(f)[2][1] == np.minimum(cnt[1], 4)).all() and (_np(l)[2] == cnt[1]).all()
    assert _np(f)[0][1].tobytes() == _np(u)[0][1].tobytes() and _np(f)[1][1].tobytes() == _np(u)[1][1].tobytes()
    _publish(keep[1], d_q, k, l, f, 1, 0, st)
    # barrier + merge = the oracle chain
    flags = torch.zeros((64,), dtype=torch.int32, device=dev)
    _capi.check(lib.sdb_peer_barrier_device(0, 1, 0, (C.c_void_p * 1)(flags.data_ptr()), 1, st))
    m = list(_outs(B, k))
    _capi.check(lib.sdb_merge_topk_device(0, S, B, k, f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr(), m[0].data_ptr(),
                                          m[1].data_ptr(), m[2].data_ptr(), st))
    torch.cuda.synchronize()
    mi, md, mc = _np(m)
    oi, od, oc = O.merge_topk(o_ids, o_d, o_c, k)
    assert (mi == oi).all() and md.tobytes() == od.tobytes() and (mc == oc).all()
    # one index over the union: every pair is re-scored the same way in any shard
    U = np.concatenate(Xs)
    gu = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    gu.set_vectors(np.arange(2, len(U) + 2, dtype=np.uint64), U)
    ui, ud, uc = gu.flat_search_batch(Q, k + 1)
    assert md.tobytes() == np.ascontiguousarray(ud[:, :k]).tobytes() and (mc == k).all()
    first = np.cumsum([0] + [len(X) for X in Xs])
    shard, local = sharded.unpack_global_ids(mi.astype(np.int64))
    rows = first[shard] + local - 2 + 2  # union ids
    distinct = [len(np.unique(ud[b])) == k + 1 for b in range(B)]
    assert sum(distinct) >= B // 2
    for b in range(B):
        if distinct[b]:
            assert set(rows[b].tolist()) == set(ui[b, :k].astype(np.int64).tolist())


# ---------------------------------------------------------------- 4. two GPUs, one process each

def _flat_p2p_worker(rank, world, port, out_dir):
    import os

    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    dim, B, k = 96, 300, 10
    if rank == 0:
        X = synth.latent_gaussian(N_TC, dim, seed=50, latent=8) * np.float32(4.0)
    else:
        X, _ = _near_copies(N_TC, dim, 1, seed=51, copies_of=12_000)
    _, base = _near_copies(10, dim, 1, seed=51, copies_of=1)
    Q = synth.latent_gaussian(B, dim, seed=52, w_seed=50, latent=8) * np.float32(4.0)
    Q[::10] = _near_queries(base, len(Q[::10]), seed=53)
    Q = np.ascontiguousarray(Q, dtype=np.float32)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"), device=rank)
    g.set_vectors(np.arange(2, N_TC + 2, dtype=np.uint64), np.ascontiguousarray(X, dtype=np.float32))
    d_q = torch.from_numpy(Q).to(dev)
    a = sharded.ShardedSearcher(g, rank, world, exchange="nccl")
    ref = [t.clone() for t in a.search_batch_device(d_q, k, None)]
    b = sharded.ShardedSearcher(g, rank, world, exchange="p2p")
    same = True
    for _ in range(5):  # every buffer parity, growing epochs
        got = b.search_batch_device(d_q, k, None)
        torch.cuda.synchronize()
        same = same and all(bool((x == y).all().item()) for x, y in zip(got, ref))
    h_q = torch.from_numpy(Q).pin_memory()
    h_i = torch.zeros((B, k), dtype=torch.int64).pin_memory()
    h_d = torch.zeros((B, k), dtype=torch.float32).pin_memory()
    h_c = torch.zeros((B,), dtype=torch.int32).pin_memory()
    for _ in range(2):
        b.search_batch_pinned(h_q, k, None, h_i, h_d, h_c, dev)
        same = same and bool((h_i == ref[0].cpu()).all()) and bool((h_d == ref[1].cpu()).all()) and \
            bool((h_c == ref[2].cpu()).all())
    c = sharded.ShardedSearcher(g, rank, world, exchange="p2p", pipeline=True)
    batches = [torch.roll(d_q, shifts=7 * i, dims=0).contiguous() for i in range(7)]
    want = [[t.clone() for t in a.search_batch_device(qb, k, None)] for qb in batches]
    torch.cuda.synchronize()
    got_p = []
    for i, qb in enumerate(batches):
        out = c.search_batch_device(qb, k, None)
        if i >= 2:
            c.wait_pipeline()
        got_p.append([t.clone() for t in out])
    c.wait_pipeline()
    torch.cuda.synchronize()
    same_pipe = all(bool((x == y).all().item()) for x, y in zip([t.clone() for t in out], want[-1]))
    for i in range(2, len(batches)):
        same_pipe = same_pipe and all(bool((x == y).all().item()) for x, y in zip(got_p[i], want[i]))
    ovf = g.flat_last_stats()[2]
    failed = b._peer.barrier_failed() or c._peer.barrier_failed()
    np.savez(os.path.join(out_dir, f"flat{rank}.npz"), same=same, same_pipe=same_pipe, failed=failed, ovf=ovf,
             ids=ref[0].cpu().numpy(), d=ref[1].cpu().numpy())
    dist.barrier()
    dist.destroy_process_group()


def test_fused_gather_two_gpus_flat_shards_match_nccl_path(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from tests.test_sharded_gloo import _free_port
    mp.spawn(_flat_p2p_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r = [np.load(tmp_path / f"flat{i}.npz") for i in range(2)]
    assert all(bool(x["same"]) and bool(x["same_pipe"]) and not bool(x["failed"]) for x in r)
    assert int(r[1]["ovf"]) > 0  # rank 1's shard sent queries to the exact fallback
    assert (r[0]["ids"] == r[1]["ids"]).all() and r[0]["d"].tobytes() == r[1]["d"].tobytes()


# ---------------------------------------------------------------- 5. errors leave the handle usable

def test_errors_leave_the_handle_usable():
    import torch
    n, dim, B = N_TC, 96, 100
    X = synth.latent_gaussian(n, dim, seed=60, latent=8)
    Q = synth.latent_gaussian(B, dim, seed=61, w_seed=60, latent=8)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    want = g.flat_search_batch(Q, 10)
    lib = _capi.lib()
    st = torch.cuda.current_stream().cuda_stream
    d_q = torch.from_numpy(Q).cuda()
    o = _outs(B, 76)
    f = _outs(B, 76)
    ptrs = [t.data_ptr() for t in o]

    def pg_of(n_peers, null_peer=False):
        pg = _capi.SdbPeerGather()
        pg.n_peers, pg.shard, pg.per_shard_limit = n_peers, 0, 0
        for p in range(min(n_peers, _capi.MAX_PEERS)):
            pg.ids[p], pg.dists[p], pg.counts[p] = f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr()
        if null_peer:
            pg.dists[0] = None
        return pg

    def check_still_right():
        got = list(_outs(B, 10))
        g.flat_search_batch_device(d_q, 10, *got, st)
        torch.cuda.synchronize()
        assert _same(want, _np(got))

    def expect_invalid(rc):
        assert rc == _capi.ERR_INVALID
        check_still_right()

    for k in (0, 76):
        expect_invalid(lib.sdb_flat_search_batch_device(g._h, B, d_q.data_ptr(), k, *ptrs, st))
        expect_invalid(lib.sdb_flat_search_batch_gather_device(g._h, B, d_q.data_ptr(), k, *ptrs, C.byref(pg_of(1)), st))
    for i in range(4):
        args = [d_q.data_ptr()] + ptrs
        args[i] = None
        expect_invalid(lib.sdb_flat_search_batch_device(g._h, B, args[0], 10, *args[1:], st))
        expect_invalid(lib.sdb_flat_search_batch_gather_device(g._h, B, args[0], 10, *args[1:], C.byref(pg_of(1)), st))
    expect_invalid(lib.sdb_flat_search_batch_gather_device(g._h, B, d_q.data_ptr(), 10, *ptrs, None, st))
    for n_peers in (0, 17):
        expect_invalid(lib.sdb_flat_search_batch_gather_device(g._h, B, d_q.data_ptr(), 10, *ptrs, C.byref(pg_of(n_peers)), st))
    expect_invalid(lib.sdb_flat_search_batch_gather_device(g._h, B, d_q.data_ptr(), 10, *ptrs, C.byref(pg_of(1, True)), st))
    with pytest.raises(SdbError):
        g.flat_search_batch_device(d_q, 0, *o, st)
    check_still_right()
