"""Shard-per-GPU search: the collection is split into independent shards (one graph, one
start node, one id space per GPU), queries are broadcast, every GPU searches its own
shard (K1), the per-GPU top-k lists are exchanged with one NCCL all-gather over NVLink and
merged by the K6 kernel on every rank.

Mirrors ClusterNode.SearchPoints (cluster/actions.go:275-379): per-shard request limit
(actions.go:291-299), scatter to every shard (actions.go:316-351), concatenate + sort by
HybridScore descending + truncate (actions.go:357-376).

Point placement: the reference fills shards sequentially from the UUID-sorted batch
(cluster/placement.go:23-50; UUIDs are random, so the effect is a uniform random partition
into near-equal chunks). Here: a seeded shuffle, then `position mod n_shards` — also a
uniform random partition into near-equal shards (SURVEY.md §2a).

One process per GPU (torch.distributed, backend nccl); torch is plumbing only (device
tensors, the collective). The merge runs through the C ABI.

The shards carry either index kind: an IndexVamana shard runs the beam search, an IndexFlat shard
the flat search (every point of the shard scanned, so G GPUs each scan N/G points).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _capi

SHARD_SHIFT = 40  # global id = (shard << 40) | node id


def partition_points(n_points: int, n_shards: int, seed: int = 0) -> np.ndarray:
    """shard index of each of n_points (seeded shuffle then position mod n_shards)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    perm = rng.permutation(n_points)
    out = np.empty(n_points, dtype=np.int32)
    out[perm] = np.arange(n_points, dtype=np.int64) % n_shards
    return out


def shard_limit(limit: int, n_shards: int, max_search_limit: int = 75) -> int:
    """targetLimit of cluster/actions.go:291-299 (f32 arithmetic like the reference)."""
    return int(_capi.lib().sdb_shard_limit(int(limit), int(n_shards), int(max_search_limit)))


def pack_global_ids(local_ids, shard: int):
    """works on numpy arrays and torch tensors (int64/uint64)."""
    return local_ids + (int(shard) << SHARD_SHIFT)


def unpack_global_ids(global_ids):
    return global_ids >> SHARD_SHIFT, global_ids & ((1 << SHARD_SHIFT) - 1)


def exchange_topk(ids, dists, counts, group=None):
    """All-gather of per-rank [B,k] results into shard-major [S,B,k] / [S,B] tensors.
    12*k+4 bytes per query per rank — latency-bound, one collective per tensor."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)

    def gather(t):
        t = t.contiguous()
        # concatenated-along-dim-0 output is accepted by both nccl and gloo
        out = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t, group=group)
        return out.view((world,) + tuple(t.shape))

    g_ids, g_d, g_c = gather(ids), gather(dists), gather(counts)
    return g_ids, g_d, g_c


class PeerGatherBuffers:
    """Peer-mapped gather buffers for the exchange fused into the search kernel
    (sdb_search_batch_gather_device): one symmetric allocation per rank, laid out as
    [flag words | buffer 0 | buffer 1 | buffer 2], each buffer = ids [S][B][k] u64, dists [S][B][k] f32,
    counts [S][B] u32. torch symmetric memory only allocates and maps the pages across the
    processes (the job cudaDeviceEnablePeerAccess does inside one Go process); the stores, the
    barrier and the merge are this library's kernels."""

    FLAG_BYTES = 256  # 2 * SDB_MAX_PEERS u32 words, padded
    NBUF = 3          # gather buffers, used round-robin by epoch (see ShardedSearcher: pipeline)

    def __init__(self, rank: int, world: int, B: int, k: int, device, group=None):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        self.rank, self.world, self.B, self.k = rank, world, B, k
        ids_b, d_b, c_b = world * B * k * 8, world * B * k * 4, world * B * 4
        self.buf_bytes = (ids_b + d_b + c_b + 255) // 256 * 256
        self.off_d, self.off_c = ids_b, ids_b + d_b
        total = self.FLAG_BYTES + self.NBUF * self.buf_bytes
        grp = group if group is not None else dist.group.WORLD
        self.t = symm.empty(total, dtype=torch.uint8, device=device)
        self.t.zero_()
        torch.cuda.synchronize(device)
        self.hdl = symm.rendezvous(self.t, grp)
        self.peer_base = [int(p) for p in self.hdl.buffer_ptrs]
        if len(self.peer_base) != world:
            raise RuntimeError("symmetric memory rendezvous returned the wrong number of peers")
        dist.barrier(grp)  # every rank has zeroed its flags before anyone signals
        self.epoch = 0
        self.device = device
        self._flags = (C.c_void_p * world)(*self.peer_base)
        self._pg = []
        for par in range(self.NBUF):
            pg = _capi.SdbPeerGather()
            pg.n_peers, pg.shard, pg.per_shard_limit = world, rank, 0
            for p, base in enumerate(self.peer_base):
                b = base + self.FLAG_BYTES + par * self.buf_bytes
                pg.ids[p], pg.dists[p], pg.counts[p] = b, b + self.off_d, b + self.off_c
            self._pg.append(pg)

    def local(self, parity: int):
        b = self.peer_base[self.rank] + self.FLAG_BYTES + parity * self.buf_bytes
        return b, b + self.off_d, b + self.off_c

    def barrier_failed(self) -> bool:
        """True if a peer_barrier_kernel on this rank ever timed out (a peer never arrived)."""
        import torch
        w = self.t[:self.FLAG_BYTES].view(torch.int32)[_capi.MAX_PEERS:2 * _capi.MAX_PEERS]
        return bool((w != 0).any().item())


class ShardedSearcher:
    """One rank's view of a sharded collection.

    exchange = "p2p": the search kernel's epilogue stores each query's top-k into every peer
    GPU's gather buffer over NVLink, one cross-GPU flag barrier, merge (K6) — no collective
    call on the data path. exchange = "nccl": one all-gather per result tensor, then K6 (also
    the path the gloo CPU tests drive). "auto" = p2p on CUDA, falling back to nccl with a
    warning on stderr if symmetric memory cannot be set up on this box."""

    def __init__(self, index, rank: Optional[int] = None, world: Optional[int] = None, group=None,
                 exchange: str = "auto", pipeline: bool = False):
        import torch.distributed as dist
        from .vamana import IndexFlat
        self.index = index
        self._flat = isinstance(index, IndexFlat)  # search_size is unused for a flat index
        self.group = group
        self.exchange = exchange
        self.pipeline = pipeline  # fused exchange only: barrier + merge of step e overlap the search of step e+1
        self._side = None
        self._pending = False
        self._peer = None
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self._bufs = None

    def _ensure_pipeline(self, B, k, device):
        import torch
        if self._side is not None and self._pipe_out[0][0].shape == (B, k):
            return
        self._side = torch.cuda.Stream(device, priority=-1)
        n = self._peer.NBUF
        self._bar_done = [torch.cuda.Event() for _ in range(n)]
        self._k1_done = torch.cuda.Event()
        self._pipe_out = [(torch.zeros((B, k), dtype=torch.int64, device=device), torch.zeros((B, k), dtype=torch.float32, device=device),
                           torch.zeros((B,), dtype=torch.int32, device=device)) for _ in range(n)]

    def wait_pipeline(self):
        """Block the caller's stream until the exchange of every submitted step has completed."""
        import torch
        if self._side is not None and self._pending:
            torch.cuda.current_stream(self._side.device).wait_stream(self._side)
            self._pending = False

    def _drain_pipeline(self):
        if self._pending:
            self._side.synchronize()
            self._pending = False

    def _ensure(self, B, k, device):
        import torch
        if self._bufs is not None and self._bufs[0].shape == (B, k):
            return
        self._bufs = (torch.zeros((B, k), dtype=torch.int64, device=device),
                      torch.zeros((B, k), dtype=torch.float32, device=device),
                      torch.zeros((B,), dtype=torch.int32, device=device),
                      torch.zeros((B, k), dtype=torch.int64, device=device),
                      torch.zeros((B, k), dtype=torch.float32, device=device),
                      torch.zeros((B,), dtype=torch.int32, device=device))

    def _requests(self, B: int, k: int, limits, search_sizes, filters, query_filter, max_search_limit: int, dev):
        """Per-request parameters of a step with `limits`: (PackedRequests, device limits for the
        merge, device shard limits), or None without them. Each request publishes
        sdb_shard_limit(limit_b, S, max_search_limit) ranks; k is the row stride."""
        if limits is None:
            return None
        import torch
        from .vamana import PackedRequests
        lim = np.broadcast_to(np.asarray(limits, dtype=np.int64), (B,))
        if B and int(lim.max()) > k:
            raise _capi.SdbError(_capi.ERR_INVALID, "limits must not exceed k, the row stride")
        shard = np.array([shard_limit(int(x), self.world, max_search_limit) for x in lim], dtype=np.int64)
        rq = PackedRequests(B, lim, search_sizes, filters, query_filter, shard, default_L=self.index.L)
        # page-locked, copied without blocking the host: a pipelined step does not wait for the last one
        d_lim = torch.from_numpy(lim.astype(np.int32)).pin_memory().to(dev, non_blocking=True)
        d_shard = torch.from_numpy(np.minimum(shard, lim).astype(np.int32)).pin_memory().to(dev, non_blocking=True)
        return rq, d_lim, d_shard

    def _merge(self, di: int, B: int, k: int, g_i, g_d, g_c, o_ids, o_d, o_c, stream, rq=None):
        """K6 over the gathered shard lists: per-request output limits when the step has them."""
        lib = _capi.lib()
        outs = (o_ids.data_ptr(), o_d.data_ptr(), o_c.data_ptr())
        if rq is None:
            _capi.check(lib.sdb_merge_topk_device(di, self.world, B, k, g_i, g_d, g_c, *outs, stream))
        else:
            _capi.check(lib.sdb_merge_topk_requests_device(di, self.world, B, k, rq[1].data_ptr(), g_i, g_d, g_c, *outs,
                                                           stream))

    def _search_shard(self, q, k: int, search_size, l_ids, l_d, l_c, stream, pg=None, filters=None, query_filter=None,
                      rq=None):
        """This rank's shard search of the [B, dim] query tensor q (device or page-locked) into l_*
        and, with pg, into slot [rank] of every peer's gather buffer: the flat entries for an
        IndexFlat, the beam-search entries otherwise, their filtered forms when `filters` is given,
        their request forms when the step has per-request parameters (rq, from _requests).
        Enqueued on `stream`, no synchronisation."""
        B = int(q.shape[0])
        if rq is not None:
            entry = self.index.flat_search_batch_requests_device if self._flat else self.index.search_batch_requests_device
            entry(q, rq[0], k, l_ids, l_d, l_c, stream, pg)
            return
        L = None if self._flat else (self.index.L if search_size is None else int(search_size))
        if filters is not None:
            if self._flat:
                self.index.flat_search_batch_filters_device(q, filters, query_filter, k, l_ids, l_d, l_c, stream, pg)
            else:
                self.index.search_batch_filters_device(q, filters, query_filter, k, L, l_ids, l_d, l_c, stream, pg)
            return
        if pg is None:
            if self._flat:
                self.index.flat_search_batch_device(q, k, l_ids, l_d, l_c, stream)
            else:
                self.index.search_batch_device(q, k, L, l_ids, l_d, l_c, stream)
            return
        lib = _capi.lib()
        outs = (l_ids.data_ptr(), l_d.data_ptr(), l_c.data_ptr())
        if self._flat:
            rc = lib.sdb_flat_search_batch_gather_device(self.index._h, B, q.data_ptr(), k, *outs, C.byref(pg), stream)
        else:
            rc = lib.sdb_search_batch_gather_device(self.index._h, B, q.data_ptr(), k, L, *outs, C.byref(pg), stream)
        _capi.check(rc)

    def search_batch_pinned(self, h_queries, k: int, search_size: Optional[int], h_ids, h_dists, h_counts, device,
                            max_search_limit: int = 75, filters=None, query_filter=None, limits=None, search_sizes=None):
        """Host-facing twin of search_batch_device for page-locked (pinned) torch CPU tensors:
        pinned memory is mapped into the device address space, so K1 reads the broadcast query
        batch straight from host memory (no staging copy in front of the kernel); the merged
        lists come back with one small copy. Falls back to explicit copies when the fused
        exchange is not active. Synchronises before returning. filters / query_filter, limits /
        search_sizes: as in search_batch_device."""
        import torch
        B = int(h_queries.shape[0])
        stream = torch.cuda.current_stream(device).cuda_stream
        fused = self.world > 1 and self.exchange != "nccl" and self._peer is not None and \
            (self._peer.B, self._peer.k) == (B, k) and h_queries.is_pinned() and h_ids.is_pinned() and \
            h_dists.is_pinned() and h_counts.is_pinned()
        if not fused:
            r_ids, r_d, r_c = self.search_batch_device(h_queries.to(device, non_blocking=True), k, search_size,
                                                       max_search_limit, filters, query_filter, limits, search_sizes)
            h_ids.copy_(r_ids, non_blocking=True)
            h_dists.copy_(r_d, non_blocking=True)
            h_counts.copy_(r_c, non_blocking=True)
            torch.cuda.synchronize(device)
            return
        l_ids, l_d, l_c = self._bufs[0], self._bufs[1], self._bufs[2]
        pb = self._peer
        self._drain_pipeline()
        pb.epoch += 1
        par = pb.epoch % pb.NBUF
        pg = pb._pg[par]
        pg.per_shard_limit = shard_limit(k, self.world, max_search_limit)
        lib = _capi.lib()
        di = device.index or 0
        rq = self._requests(B, k, limits, search_sizes, filters, query_filter, max_search_limit, device)
        self._search_shard(h_queries, k, search_size, l_ids, l_d, l_c, stream, pg, filters, query_filter, rq)
        _capi.check(lib.sdb_peer_barrier_device(di, self.world, self.rank, pb._flags, pb.epoch, stream))
        g_i, g_dd, g_cc = pb.local(par)
        # The merge is a short kernel: its 300 k small stores would sit exposed on PCIe if they went
        # to mapped host memory (measured: +0.3 ms per step at B = 10 k), so it writes device buffers
        # and one 1.24 MB copy brings the lists back. K1's query reads stay zero-copy.
        m_ids, m_d, m_c = self._bufs[3], self._bufs[4], self._bufs[5]
        self._merge(di, B, k, g_i, g_dd, g_cc, m_ids, m_d, m_c, stream, rq)
        h_ids.copy_(m_ids, non_blocking=True)
        h_dists.copy_(m_d, non_blocking=True)
        h_counts.copy_(m_c, non_blocking=True)
        torch.cuda.synchronize(device)
        # the step is complete on this GPU: a barrier that gave up on a peer makes it an error
        _capi.check(lib.sdb_peer_barrier_check(di, 0))

    def search_batch_device(self, d_queries, k: int, search_size: Optional[int], max_search_limit: int = 75,
                            filters=None, query_filter=None, limits=None, search_sizes=None):
        """d_queries: [B, dim] f32 CUDA tensor, identical on every rank (broadcast by the
        caller). Returns merged (global ids [B,k] int64, dists [B,k], counts [B]) on every rank.
        search_size: the beam width of a Vamana shard (None = the index's); unused for a flat one.

        filters: this rank's shard-local id lists (as in IndexVamana.search_batch_filters: the
        reference evaluates a request's filter on every shard against that shard's own points,
        shard/index/search.go:59-85); query_filter[b]: the list request b uses on this rank, -1 for
        none (None: every request uses filters[0]). A request filtered on one rank must be filtered
        on every rank — its list there may be empty — or the merged list mixes filtered and
        unfiltered shard results; the library cannot check this across ranks. The filters are
        copied before the call returns. A vamana.PackedFilters (which carries its query_filter) may
        stand for the lists.

        A filter error is local to the rank whose lists it finds (unsorted ids, a query_filter index
        out of range, a missing seed): that rank raises before it reaches the step's barrier, and with
        the fused exchange its peers' barrier of that step times out (~20 s), after which their
        exchange calls fail with SDB_ERR_STATE until sdb_peer_barrier_check(clear) (semadb_b200.h).
        The epoch has advanced on every rank, so the ranks stay in step once cleared. Callers that
        cannot rule such errors out check each rank's lists first (the host filter entries apply the
        same checks).

        limits / search_sizes: every request's own limit and searchSize (models/search.go:268-314),
        one value per request or one for all (search_sizes None: search_size, else the index's). k is
        then the row stride of the results and must be at least every limit; row b holds at most
        limits[b] results, each shard contributing sdb_shard_limit(limits[b], S, max_search_limit)
        of them, and is padded with id 0 / +inf. The limits are the same on every rank."""
        import torch
        B = int(d_queries.shape[0])
        dev = d_queries.device
        if limits is not None and search_sizes is None and search_size is not None:
            search_sizes = search_size
        self._ensure(B, k, dev)
        rq = self._requests(B, k, limits, search_sizes, filters, query_filter, max_search_limit, dev)
        l_ids, l_d, l_c, m_ids, m_d, m_c = self._bufs
        stream = torch.cuda.current_stream(dev).cuda_stream
        # the reference asks each shard for min(k, floor(k/S*1.42+10)) results; the local
        # search still fills k slots and the merge reads only the first `per_shard`
        per_shard = shard_limit(k, self.world, max_search_limit)
        if self.world > 1 and self.exchange in ("auto", "p2p") and d_queries.is_cuda:
            if self._peer is None or (self._peer.B, self._peer.k) != (B, k):
                try:
                    self._peer = PeerGatherBuffers(self.rank, self.world, B, k, dev, self.group)
                except Exception as e:  # noqa: BLE001
                    if self.exchange == "p2p":
                        raise
                    import sys
                    print(f"[semadb_b200] peer-mapped gather buffers unavailable ({e!r}); using the NCCL all-gather",
                          file=sys.stderr, flush=True)
                    self.exchange = "nccl"
        if self.world > 1 and self._peer is not None and self.exchange != "nccl":
            pb = self._peer
            lib = _capi.lib()
            di = dev.index or 0
            if not self.pipeline:
                pb.epoch += 1
                par = pb.epoch % pb.NBUF
                pg = pb._pg[par]
                pg.per_shard_limit = per_shard
                self._search_shard(d_queries, k, search_size, l_ids, l_d, l_c, stream, pg, filters, query_filter, rq)
                _capi.check(lib.sdb_peer_barrier_device(di, self.world, self.rank, pb._flags, pb.epoch, stream))
                g_i, g_dd, g_cc = pb.local(par)
                self._merge(di, B, k, g_i, g_dd, g_cc, m_ids, m_d, m_c, stream, rq)
                return m_ids, m_d, m_c
            # Pipelined steps: the search of step e runs on the caller's stream; its barrier and merge
            # run on a side stream, so the search of step e+1 starts without waiting for the slowest
            # peer of step e. Three gather buffers: step e+3 reuses the buffer of step e, and every
            # rank's merge(e) has completed once the barrier of step e+1 has (a rank reaches that
            # barrier after its own merge(e), side-stream order) — so search(e) waits for the local
            # barrier(e-2). Results of a step are valid once the side stream has drained
            # (torch.cuda.synchronize / wait_pipeline).
            self._ensure_pipeline(B, k, dev)
            main = torch.cuda.current_stream(dev)
            side = self._side
            pb.epoch += 1
            e = pb.epoch
            par = e % pb.NBUF
            if e >= 3:
                main.wait_event(self._bar_done[(e - 2) % pb.NBUF])
            pg = pb._pg[par]
            pg.per_shard_limit = per_shard
            self._search_shard(d_queries, k, search_size, l_ids, l_d, l_c, main.cuda_stream, pg, filters, query_filter, rq)
            self._k1_done.record(main)
            side.wait_event(self._k1_done)
            o_ids, o_d, o_c = self._pipe_out[par]
            _capi.check(lib.sdb_peer_barrier_device(di, self.world, self.rank, pb._flags, e, side.cuda_stream))
            self._bar_done[par].record(side)
            g_i, g_dd, g_cc = pb.local(par)
            if rq is not None:  # the side stream reads the step's limits: keep them alive until it has
                self._pipe_rq = getattr(self, "_pipe_rq", [None] * pb.NBUF)
                self._pipe_rq[par] = rq
            self._merge(di, B, k, g_i, g_dd, g_cc, o_ids, o_d, o_c, side.cuda_stream, rq)
            self._pending = True
            return o_ids, o_d, o_c
        self._search_shard(d_queries, k, search_size, l_ids, l_d, l_c, stream, None, filters, query_filter, rq)
        if rq is not None:
            torch.minimum(l_c, rq[2], out=l_c)
        elif per_shard < k:
            l_c.clamp_(max=per_shard)
        if self.world == 1:
            return l_ids, l_d, l_c
        g_ids, g_d, g_c = exchange_topk(pack_global_ids(l_ids, self.rank), l_d, l_c, self.group)
        self._merge(dev.index or 0, B, k, g_ids.data_ptr(), g_d.data_ptr(), g_c.data_ptr(), m_ids, m_d, m_c, stream, rq)
        return m_ids, m_d, m_c


def replica_slice(B: int, rank: int, world: int):
    """Batch positions [lo, hi) served by replica `rank`: contiguous, sizes differing by at most one."""
    base, rem = divmod(B, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class ReplicatedSearcher:
    """Replicated mode (SURVEY.md §8e-iii): every GPU holds the WHOLE index and serves a contiguous
    slice of the query batch; the slices are concatenated with one all-gather per result tensor.
    Results are those of a single-GPU search — same graph, same queries — so user-visible QPS grows
    with the number of GPUs (strong scaling) for collections that fit one GPU. The reference's
    counterpart is several replicas of a shard behind its RPC layer, each serving whole requests
    (shard/cache/manager.go:151-182 serves concurrent readers of one shard)."""

    def __init__(self, index, rank: Optional[int] = None, world: Optional[int] = None, group=None):
        import torch.distributed as dist
        self.index, self.group = index, group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self._bufs = None

    def search_batch_device(self, d_queries, k: int, search_size: int):
        """d_queries [B, dim] identical on every rank; returns (ids [B,k], dists [B,k], counts [B]) on every rank."""
        import torch
        import torch.distributed as dist
        B = int(d_queries.shape[0])
        dev = d_queries.device
        per = (B + self.world - 1) // self.world  # padded slice so that the gather is regular
        if self._bufs is None or self._bufs[0].shape != (per, k):
            self._bufs = (torch.zeros((per, k), dtype=torch.int64, device=dev), torch.zeros((per, k), dtype=torch.float32, device=dev),
                          torch.zeros((per,), dtype=torch.int32, device=dev))
        l_ids, l_d, l_c = self._bufs
        lo, hi = replica_slice(B, self.rank, self.world)
        if hi > lo:
            self.index.search_batch_device(d_queries[lo:hi], k, search_size, l_ids, l_d, l_c,
                                           torch.cuda.current_stream(dev).cuda_stream if d_queries.is_cuda else 0)
        if self.world == 1:
            return l_ids[:B], l_d[:B], l_c[:B]
        outs = []
        for t in (l_ids, l_d, l_c):
            g = torch.empty((self.world * per,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
            dist.all_gather_into_tensor(g, t, group=self.group)
            outs.append(g.view((self.world, per) + tuple(t.shape[1:])))
        sizes = [replica_slice(B, r, self.world) for r in range(self.world)]
        return tuple(torch.cat([o[r, :hi_ - lo_] for r, (lo_, hi_) in enumerate(sizes)]) for o in outs)
