"""Sharded search with per-request filters (sdb_search_batch_filters_device,
sdb_flat_search_batch_filters_device through ShardedSearcher) over G GPUs, and the host filter
entries of this build against another build.

Scaling (one process per GPU):
  torchrun --nproc_per_node G scripts/bench_sharded_filters.py scale --kind vamana|flat --out DIR
    vamana  1M x 128 f32 squared-L2 points per GPU (the synth.sift_shaped law, one seed per rank), the
            graph built on the GPU; 10 000 queries, k 10, L 75. Filter mixes: unfiltered; one shared
            10 % filter; an own random filter per request at 1 % and at 10 %; half the batch with
            an own 1 % filter, half unfiltered. The 10 % own-filter mix runs 1 000 queries: at
            10 000 its lists alone would be 10^9 ids (8 GB) per step.
    flat    8M x 128 (bench_sharded_flat.py's strong workload) split G ways; an own filter per
            request at 0.01 % and at 0.1 % of the shard.
  Filters are shard-local random ids drawn per rank (the same request is filtered on every rank).
  Per mix: ms per step (device-resident queries and results) unpipelined and, at G > 1, pipelined;
  host_ms_until_return = host clock around the enqueuing call alone, mean over the timed steps: the
  filter staging (validation, narrowing, work lists) plus any wait for a staging slot; at G > 1 the
  p2p lists equal the NCCL lists. The filters are packed once (vamana.PackedFilters), as a caller
  that keeps its lists would. Rank 0 writes DIR/<kind>_g<G>.json.

Host entries, this build against another (one process, one GPU):
  python scripts/bench_sharded_filters.py ab --parent-lib PATH --out DIR
    sdb_flat_search_batch_filters and sdb_search_batch_filters of both builds, alternately, at the
    shapes of profiles/r03_flat_filters.json: 1M x 128 sift_shaped, 10 000 requests, an own random
    filter per request at 0.01 %, 0.1 % and 1 %, and for flat search one filter shared by the batch
    at 50 % (the range-scan route) (beam search: the graph is built once per build). This build's
    staging memory after each shape is reported (sdb_filter_staging_bytes).
    Page-locked queries and outputs. Lists of both builds are compared byte for byte. Writes DIR/ab.json.

  python scripts/bench_sharded_filters.py report --out DIR --profile FILE   assembles FILE from DIR.
Every timed call is warmed up with the same shapes first; the card name and power limit are read
(nvidia-smi, read-only) in the same process as the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))

K, L = 10, 75


def own_filters(B, n_ids, frac, seed, first_id=2):
    """B strictly ascending random id lists, each keeping about frac of the ids first_id ..
    first_id + n_ids - 1 (geometric gaps), packed: (ids, offsets)."""
    rng = np.random.default_rng(seed)
    m = max(1, int(round(n_ids * frac)))
    ids = np.cumsum(rng.geometric(frac, size=(B, m)), axis=1, dtype=np.uint64) + np.uint64(first_id - 1)
    keep = ids < np.uint64(first_id + n_ids)
    lens = keep.sum(1)
    off = np.zeros(B + 1, np.uint64)
    off[1:] = np.cumsum(lens)
    return np.ascontiguousarray(ids[keep]), off


def mixes(kind, n_local, B, rank):
    """(name, batch, PackedFilters or None) of every filter mix; seeds differ per rank."""
    from semadb_b200.vamana import PackedFilters
    s = 1000 * rank
    if kind == "flat":
        return [(f"own filter per request {p} %", B, PackedFilters.from_csr(*own_filters(B, n_local, p / 100, s + i)))
                for i, p in enumerate((0.01, 0.1))]
    half_ids, half_off = own_filters(B // 2, n_local, 0.01, s + 4)
    half_qf = np.full(B, -1, np.int32)
    half_qf[::2] = np.arange(B // 2, dtype=np.int32)
    shared = own_filters(1, n_local, 0.10, s + 1)
    return [("unfiltered", B, None),
            ("one shared 10 % filter", B, PackedFilters.from_csr(*shared)),
            ("own filter per request 1 %", B, PackedFilters.from_csr(*own_filters(B, n_local, 0.01, s + 2))),
            ("own filter per request 10 %", 1000, PackedFilters.from_csr(*own_filters(1000, n_local, 0.10, s + 3))),
            ("half the batch: own 1 % filter", B, PackedFilters.from_csr(half_ids, half_off, half_qf))]


def build(kind, rank, world, dev):
    import torch
    from semadb_b200 import synth
    from semadb_b200.vamana import IndexVamana, IndexVectorVamanaParameters
    if kind == "flat":
        from bench_sharded_flat import build_shard
        return build_shard("strong", rank, world, dev)
    n = 1_000_000
    X = synth.sift_shaped(n, 128, seed=3 + 101 * rank, w_seed=3)
    g = IndexVamana("shard", IndexVectorVamanaParameters(128, "euclidean"), device=dev.index, start_seed=99)
    g.insert_batch_device(np.arange(2, n + 2, dtype=np.uint64), torch.from_numpy(X).to(dev))
    torch.cuda.synchronize(dev)
    return g, n


def scale(args):
    import torch
    import torch.distributed as dist
    from bench_sharded_flat import card
    from semadb_b200 import sharded, synth
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    t0 = time.time()
    g, n_local = build(args.kind, rank, world, dev)
    load_s = time.time() - t0
    Qall = torch.from_numpy(synth.sift_shaped(10_000, 128, seed=4, w_seed=3)).to(dev)
    ex = "p2p" if world > 1 else "nccl"
    rows = []
    for name, B, pf in mixes(args.kind, n_local, 10_000, rank):
        d_q = Qall[:B].contiguous()

        def timed(searcher):
            for _ in range(args.warmup):
                searcher.search_batch_device(d_q, K, None, filters=pf)
            searcher.wait_pipeline()
            torch.cuda.synchronize(dev)
            dist.barrier()
            host = []
            t = time.perf_counter()
            for _ in range(args.steps):
                h = time.perf_counter()
                r = searcher.search_batch_device(d_q, K, None, filters=pf)
                host.append(time.perf_counter() - h)
            searcher.wait_pipeline()
            torch.cuda.synchronize(dev)
            return (time.perf_counter() - t) / args.steps, float(np.mean(host)), [x.clone() for x in r]

        s_un = sharded.ShardedSearcher(g, rank, world, exchange=ex)
        dt_un, host_un, lists = timed(s_un)
        dt_pi = host_pi = None
        parity = {}
        if world > 1:
            s_pi = sharded.ShardedSearcher(g, rank, world, exchange=ex, pipeline=True)
            dt_pi, host_pi, _ = timed(s_pi)
            ref = sharded.ShardedSearcher(g, rank, world, exchange="nccl").search_batch_device(d_q, K, None, filters=pf)
            torch.cuda.synchronize(dev)
            parity["p2p_equals_nccl"] = all(bool((a == b).all().item()) for a, b in zip(lists, ref))
            parity["barrier_failed"] = bool(s_un._peer.barrier_failed() or s_pi._peer.barrier_failed())
        good = parity.get("p2p_equals_nccl", True) and not parity.get("barrier_failed", False)
        ok = torch.tensor([int(good)], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        n_ids = 0 if pf is None else int(pf.off[-1])
        rows.append({"mix": name, "batch": B, "filter_ids_rank0": n_ids,
                     "ms_per_step_unpipelined": dt_un * 1e3, "ms_per_step_pipelined": None if dt_pi is None else dt_pi * 1e3,
                     "host_ms_until_return_unpipelined": host_un * 1e3,
                     "host_ms_until_return_pipelined": None if host_pi is None else host_pi * 1e3,
                     "user_qps_unpipelined": B / dt_un, "parity_rank0": parity, "parity_all_ranks": bool(ok.item())})
        if rank == 0:
            print(json.dumps(rows[-1]), flush=True)
    if rank == 0:
        desc = {"vamana": "1M x 128 f32 squared-L2 per GPU (sift_shaped law), graph built on the GPU; k 10, L 75",
                "flat": "8M x 128 f32 squared-L2 (sift_shaped law) split over the GPUs; k 10"}[args.kind]
        res = {"kind": args.kind, "workload": desc, "gpus": world, "points_per_gpu_rank0": n_local, "k": K,
               "card": card(), "load_s_rank0": round(load_s, 1), "steps": args.steps, "warmup": args.warmup,
               "exchange": "fused peer stores over NVLink + flag barrier" if world > 1 else "none (one shard)", "mixes": rows}
        (out / f"{args.kind}_g{world}.json").write_text(json.dumps(res, indent=1))
    dist.barrier()
    dist.destroy_process_group()


class _Lib:
    """The entries the comparison needs, from one build of the library."""

    NAMES = ("sdb_index_create", "sdb_index_destroy", "sdb_index_set_start", "sdb_index_set_vectors", "sdb_insert_batch",
             "sdb_search_batch_filters", "sdb_flat_search_batch_filters", "sdb_last_error")

    def __init__(self, path, extra=()):
        from semadb_b200 import _capi
        self.L = C.CDLL(str(path))
        for name in self.NAMES + tuple(extra):
            fn = getattr(self.L, name)
            fn.restype, fn.argtypes = _capi._SIGS[name]
        self.c = _capi

    def index(self, X, vamana):
        from semadb_b200 import synth
        from semadb_b200.vamana import IndexVectorVamanaParameters, _params_struct
        c = self.c
        h = c.H()
        ps = _params_struct(IndexVectorVamanaParameters(X.shape[1], "euclidean"), 0, not vamana)
        c.check(self.L.sdb_index_create(C.byref(ps), C.byref(h)))
        ids = np.arange(2, len(X) + 2, dtype=np.uint64)
        x = np.ascontiguousarray(X)
        if vamana:
            c.check(self.L.sdb_index_set_start(h, synth.start_vector(X.shape[1], 99).ctypes.data_as(c.f32p)))
            c.check(self.L.sdb_insert_batch(h, len(ids), ids.ctypes.data_as(c.u64p), x.ctypes.data_as(c.f32p)))
        else:
            c.check(self.L.sdb_index_set_vectors(h, len(ids), ids.ctypes.data_as(c.u64p), x.ctypes.data_as(c.f32p)))
        return h


def ab(args):
    import torch
    from bench_sharded_flat import card
    from semadb_b200 import _capi, synth
    from semadb_b200.vamana import PackedFilters
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    libs = {"this": _Lib(_capi.LIB_PATH, ("sdb_filter_staging_bytes",)), "parent": _Lib(args.parent_lib)}
    n, B = 1_000_000, 10_000
    X = synth.sift_shaped(n, 128, seed=3)
    h_q = torch.from_numpy(synth.sift_shaped(B, 128, seed=4, w_seed=3)).pin_memory()
    res = {"card": card(), "reps": args.reps, "shapes": {}}
    for entry in ("flat", "vamana"):
        hs = {tag: lb.index(X, entry == "vamana") for tag, lb in libs.items()}
        shapes = [(p, False) for p in (0.01, 0.1, 1.0)] + ([(50.0, True)] if entry == "flat" else [])
        for p, shared in shapes:
            pf = PackedFilters.from_csr(*own_filters(1 if shared else B, n, p / 100, 7))
            bufs = {tag: (torch.zeros((B, K), dtype=torch.int64).pin_memory(), torch.zeros((B, K), dtype=torch.float32).pin_memory(),
                          torch.zeros((B,), dtype=torch.int32).pin_memory()) for tag in libs}

            def call(tag):
                lb, (i, d, c) = libs[tag], bufs[tag]
                outs = (C.cast(i.data_ptr(), _capi.u64p), C.cast(d.data_ptr(), _capi.f32p), C.cast(c.data_ptr(), _capi.u32p))
                q = C.cast(h_q.data_ptr(), _capi.f32p)
                if entry == "flat":
                    rc = lb.L.sdb_flat_search_batch_filters(hs[tag], B, q, K, *pf.args(), *outs)
                else:
                    rc = lb.L.sdb_search_batch_filters(hs[tag], B, q, K, L, *pf.args(), *outs)
                _capi.check(rc)

            for tag in libs:
                for _ in range(2):
                    call(tag)
            times = {t: [] for t in libs}
            for _ in range(args.reps):
                for tag in libs:  # alternate the builds
                    t = time.perf_counter()
                    call(tag)
                    times[tag].append((time.perf_counter() - t) * 1e3)
            same = all(bufs["this"][j].numpy().tobytes() == bufs["parent"][j].numpy().tobytes() for j in range(3))
            name = f"{entry} 1M x 128, 10 000 requests, " + (f"one shared filter {p} %" if shared else f"own filter per request {p} %")
            pinned, device = C.c_uint64(0), C.c_uint64(0)
            _capi.check(libs["this"].L.sdb_filter_staging_bytes(hs["this"], C.byref(pinned), C.byref(device)))
            res["shapes"][name] = {
                "filter_ids": int(pf.off[-1]), "lists_identical": same,
                "this_staging_pinned_bytes": pinned.value, "this_staging_device_bytes": device.value,
                **{f"{t}_ms_median": float(np.median(v)) for t, v in times.items()},
                **{f"{t}_ms_min": float(np.min(v)) for t, v in times.items()},
                **{f"{t}_ms_each": [round(x, 3) for x in v] for t, v in times.items()}}
            print(name, json.dumps(res["shapes"][name]), flush=True)
        for tag, lb in libs.items():
            lb.L.sdb_index_destroy(hs[tag])
    (out / "ab.json").write_text(json.dumps(res, indent=1))


def report(args):
    out = Path(args.out)
    res = {"script": "scripts/bench_sharded_filters.py", "scaling": {}}
    for kind in ("vamana", "flat"):
        rows = [json.loads(p.read_text()) for p in sorted(out.glob(f"{kind}_g*.json"))]
        res["scaling"][kind] = sorted(rows, key=lambda r: r["gpus"])
    if (out / "ab.json").exists():
        res["host_entries_this_vs_parent"] = json.loads((out / "ab.json").read_text())
    Path(args.profile).write_text(json.dumps(res, indent=1) + "\n")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("mode", choices=["scale", "ab", "report"])
    ap.add_argument("--kind", choices=["vamana", "flat"], default="vamana")
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-lib")
    ap.add_argument("--profile")
    args = ap.parse_args()
    {"scale": scale, "ab": ab, "report": report}[args.mode](args)


if __name__ == "__main__":
    main()
