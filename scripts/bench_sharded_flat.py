"""Sharded flat search: strong scaling of one fixed collection over G GPUs, and the cost of the
device-side overflow fallback of the flat search.

Scaling (one process per GPU):
  torchrun --nproc_per_node G scripts/bench_sharded_flat.py scale --workload strong|c3 --out DIR
    strong  8M x 128 f32 squared-L2 points (the synth.sift_shaped law, generated on the device), 10 000
            queries, k 10
    c3      the C3 collection of bench.py (10M x 384, latent-16, L2-normalised, cosine): exact search
  The collection is split by sharded.partition_points; every rank holds one IndexFlat shard and runs
  ShardedSearcher over it. Per G: ms per step (device-resident queries and results) unpipelined and
  pipelined, user QPS, and the whole step's useful bf16 rate per GPU, 2 * B * (N / G) * D / step time
  (a whole-step rate, not a kernel's share of peak). Parity: at G > 1 the p2p lists equal the
  NCCL-path lists; on a 1 000-query probe the merged distances are bit-identical to the G = 1 run's,
  which G = 1 saves to DIR. Rank 0 writes DIR/<workload>_g<G>.json.

Fallback overhead (one process, one GPU):
  python scripts/bench_sharded_flat.py ab --parent-lib PATH --out DIR
    times sdb_flat_search_batch of this build and of another build of the library (PATH, e.g. the
    parent commit's) alternately: bench.py's extra_configs.flat workload (10 000 x 1M x 128, page-
    locked buffers) and the near-duplicate overflow shape of tests/test_flat_tc.py at 200 and 10 000
    queries. Lists of both builds are compared byte for byte. Writes DIR/ab.json.

  python scripts/bench_sharded_flat.py report --out DIR --profile FILE   assembles FILE from DIR.
Every timed call is warmed up with the same shapes first; the card name and power limit are read
(nvidia-smi, read-only) in the same process as the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

K = 10
PROBE = 1000
WORKLOADS = {
    "strong": dict(n=8_000_000, dim=128, metric="euclidean", nq=10_000,
                   desc="8M x 128 f32 squared-L2 (sift_shaped law, device-generated), 10 000 queries, k 10"),
    "c3": dict(n=10_000_000, dim=384, metric="cosine", nq=10_000,
               desc="C3: 10M x 384 (latent-16, L2-normalised) cosine, exact flat search, 10 000 queries, k 10"),
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        return [x.strip() for x in out]
    except Exception as e:  # noqa: BLE001
        return [f"unavailable: {e!r}"]


def chunks(name, dev, queries=False):
    """(start, chunk) pairs of the whole collection (or of its queries) on `dev`."""
    from semadb_b200 import synth
    w = WORKLOADS[name]
    n = w["nq"] if queries else w["n"]
    if name == "strong":  # sift_shaped: clip(rint(32 * (zW + 0.1e) + 64), 0, 255)
        for s, x in synth.latent_gaussian_torch(n, 128, 4 if queries else 3, dev, w_seed=3, latent=16):
            yield s, x.mul_(32).add_(64).round_().clamp_(0, 255)
    else:  # bench.py's C3 generator: data seed 5, query seed 6
        yield from synth.latent_gaussian_torch(n, 384, 6 if queries else 5, dev, w_seed=5, latent=16, normalize=True)


def build_shard(name, rank, world, dev):
    import torch
    from semadb_b200 import sharded
    from semadb_b200.vamana import IndexFlat, IndexVectorFlatParameters
    w = WORKLOADS[name]
    part = sharded.partition_points(w["n"], world, seed=0)
    g = IndexFlat(IndexVectorFlatParameters(w["dim"], w["metric"]), device=dev.index)
    nxt = 2
    g.reserve(int((part == rank).sum()) + 2)
    for s, x in chunks(name, dev):
        mine = torch.from_numpy(np.nonzero(part[s:s + len(x)] == rank)[0]).to(dev)
        xs = x.index_select(0, mine).cpu().numpy()
        g.set_vectors(np.arange(nxt, nxt + len(xs), dtype=np.uint64), xs)
        nxt += len(xs)
    torch.cuda.synchronize(dev)
    return g, nxt - 2


def scale(args):
    import torch
    import torch.distributed as dist
    from semadb_b200 import sharded
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    w = WORKLOADS[args.workload]
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    t0 = time.time()
    g, n_local = build_shard(args.workload, rank, world, dev)
    load_s = time.time() - t0
    d_q = torch.cat([x for _, x in chunks(args.workload, dev, queries=True)]).contiguous()
    B = d_q.shape[0]

    def timed(searcher, steps, pipelined):
        for _ in range(args.warmup):
            searcher.search_batch_device(d_q, K, None)
        searcher.wait_pipeline()
        torch.cuda.synchronize(dev)
        dist.barrier()
        t = time.perf_counter()
        for _ in range(steps):
            r = searcher.search_batch_device(d_q, K, None)
        searcher.wait_pipeline()
        torch.cuda.synchronize(dev)
        dt = (time.perf_counter() - t) / steps
        return dt, [x.clone() for x in r]

    ex = "p2p" if world > 1 else "nccl"
    s_un = sharded.ShardedSearcher(g, rank, world, exchange=ex)
    dt_un, lists = timed(s_un, args.steps, False)
    dt_pipe = None
    if world > 1:
        s_pi = sharded.ShardedSearcher(g, rank, world, exchange=ex, pipeline=True)
        dt_pipe, _ = timed(s_pi, args.steps, True)
    parity = {}
    if world > 1:
        ref = sharded.ShardedSearcher(g, rank, world, exchange="nccl").search_batch_device(d_q, K, None)
        torch.cuda.synchronize(dev)
        parity["p2p_equals_nccl"] = all(bool((a == b).all().item()) for a, b in zip(lists, ref))
        parity["barrier_failed"] = bool(s_un._peer.barrier_failed() or s_pi._peer.barrier_failed())
    probe_d = lists[1][:PROBE].cpu().numpy()
    probe_file = out / f"{args.workload}_probe_g1.npy"
    if world == 1 and rank == 0:
        np.save(probe_file, probe_d)
    elif probe_file.exists():
        parity["probe_dists_equal_g1"] = probe_d.tobytes() == np.load(probe_file).tobytes()
    else:
        parity["probe_dists_equal_g1"] = None
    good = parity.get("p2p_equals_nccl", True) and parity.get("probe_dists_equal_g1", True) is not False and \
        not parity.get("barrier_failed", False)
    ok = torch.tensor([int(good)], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    path, cand, ovf = g.flat_last_stats()
    if rank == 0:
        D, N = w["dim"], w["n"]
        flop = 2.0 * B * (N / world) * D
        res = {"workload": w["desc"], "gpus": world, "points_per_gpu_rank0": n_local, "batch": B, "k": K,
               "card": card(), "load_s_rank0": round(load_s, 1),
               "ms_per_step_unpipelined": dt_un * 1e3, "ms_per_step_pipelined": None if dt_pipe is None else dt_pipe * 1e3,
               "user_qps_unpipelined": B / dt_un, "user_qps_pipelined": None if dt_pipe is None else B / dt_pipe,
               "whole_step_bf16_tflops_per_gpu_unpipelined": flop / dt_un / 1e12,
               "whole_step_bf16_tflops_per_gpu_pipelined": None if dt_pipe is None else flop / dt_pipe / 1e12,
               "flat_path_rank0": path, "candidates_per_query_rank0": cand / B, "overflowed_rank0": ovf,
               "exchange": "fused peer stores over NVLink + flag barrier" if world > 1 else "none (one shard)",
               "parity_rank0": parity, "parity_all_ranks": bool(ok.item()), "steps": args.steps, "warmup": args.warmup}
        (out / f"{args.workload}_g{world}.json").write_text(json.dumps(res, indent=1))
        print(json.dumps(res), flush=True)
    dist.barrier()
    dist.destroy_process_group()


class _Lib:
    """The three entries the comparison needs, from one build of the library."""

    def __init__(self, path):
        from semadb_b200 import _capi
        self.L = C.CDLL(str(path))
        for name in ("sdb_index_create", "sdb_index_destroy", "sdb_index_set_vectors", "sdb_flat_search_batch",
                     "sdb_flat_last_stats", "sdb_last_error"):
            fn = getattr(self.L, name)
            fn.restype, fn.argtypes = _capi._SIGS[name]
        self.c = _capi

    def index(self, dim, X):
        from semadb_b200.vamana import IndexVectorFlatParameters, _params_struct
        h = self.c.H()
        ps = _params_struct(IndexVectorFlatParameters(dim, "euclidean"), 0, True)
        self.c.check(self.L.sdb_index_create(C.byref(ps), C.byref(h)))
        ids = np.arange(2, len(X) + 2, dtype=np.uint64)
        self.c.check(self.L.sdb_index_set_vectors(h, len(ids), ids.ctypes.data_as(self.c.u64p),
                                                  np.ascontiguousarray(X).ctypes.data_as(self.c.f32p)))
        return h


def ab(args):
    import torch
    from semadb_b200 import _capi, synth
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    libs = {"this": _Lib(_capi.LIB_PATH), "parent": _Lib(args.parent_lib)}
    rng = np.random.default_rng(11)
    base = rng.normal(size=(7, 96)).astype(np.float32)
    Xo = (base[np.arange(70_000) % 7] + rng.normal(size=(70_000, 96)).astype(np.float32) * np.float32(1e-4)).astype(np.float32)
    Qo = (base[rng.integers(0, 7, 10_000)] + rng.normal(size=(10_000, 96)).astype(np.float32) * np.float32(1e-3)).astype(np.float32)
    shapes = {"flat_10k_x_1M_x_128": (synth.sift_shaped(1_000_000, 128, seed=3), synth.sift_shaped(10_000, 128, seed=4, w_seed=3)),
              "overflow_200": (Xo, Qo[:200]), "overflow_10k": (Xo, Qo)}
    res = {"card": card(), "reps": args.reps, "shapes": {}}
    for name, (X, Q) in shapes.items():
        B, dim = Q.shape
        h_q = torch.from_numpy(np.ascontiguousarray(Q)).pin_memory()
        bufs = {}
        hs = {}
        for tag, lb in libs.items():
            hs[tag] = lb.index(dim, X)
            bufs[tag] = (torch.zeros((B, K), dtype=torch.int64).pin_memory(), torch.zeros((B, K), dtype=torch.float32).pin_memory(),
                         torch.zeros((B,), dtype=torch.int32).pin_memory())

        def call(tag):
            lb, (i, d, c) = libs[tag], bufs[tag]
            _capi.check(lb.L.sdb_flat_search_batch(hs[tag], B, C.cast(h_q.data_ptr(), _capi.f32p), K, None, 0,
                                                   C.cast(i.data_ptr(), _capi.u64p), C.cast(d.data_ptr(), _capi.f32p),
                                                   C.cast(c.data_ptr(), _capi.u32p)))

        for tag in libs:
            for _ in range(3):
                call(tag)
        times = {t: [] for t in libs}
        for _ in range(args.reps):
            for tag in libs:  # alternate the builds
                t = time.perf_counter()
                call(tag)
                times[tag].append((time.perf_counter() - t) * 1e3)
        same = all(bufs["this"][j].numpy().tobytes() == bufs["parent"][j].numpy().tobytes() for j in range(3))
        st = {}
        for tag, lb in libs.items():
            p, cnd, o = C.c_int32(0), C.c_uint64(0), C.c_uint32(0)
            lb.L.sdb_flat_last_stats(hs[tag], C.byref(p), C.byref(cnd), C.byref(o))
            st[tag] = {"path": p.value, "overflowed": o.value}
            lb.L.sdb_index_destroy(hs[tag])
        res["shapes"][name] = {
            "queries": B, "points": len(X), "dim": dim, "k": K, "lists_identical": same, "stats": st,
            **{f"{t}_ms_median": float(np.median(v)) for t, v in times.items()},
            **{f"{t}_ms_min": float(np.min(v)) for t, v in times.items()},
            **{f"{t}_ms_each": [round(x, 3) for x in v] for t, v in times.items()}}
        print(name, json.dumps(res["shapes"][name]), flush=True)
    (out / "ab.json").write_text(json.dumps(res, indent=1))


def report(args):
    out = Path(args.out)
    res = {"script": "scripts/bench_sharded_flat.py", "scaling": {}}
    for name in WORKLOADS:
        rows = [json.loads(p.read_text()) for p in sorted(out.glob(f"{name}_g*.json"))]
        rows.sort(key=lambda r: r["gpus"])
        base = next((r for r in rows if r["gpus"] == 1), None)
        for r in rows:
            if base:
                r["speedup_unpipelined_vs_g1"] = base["ms_per_step_unpipelined"] / r["ms_per_step_unpipelined"]
                if r["ms_per_step_pipelined"]:
                    r["speedup_pipelined_vs_g1"] = base["ms_per_step_unpipelined"] / r["ms_per_step_pipelined"]
        res["scaling"][name] = rows
    if (out / "ab.json").exists():
        res["fallback_overhead_host_entry"] = json.loads((out / "ab.json").read_text())
    Path(args.profile).write_text(json.dumps(res, indent=1) + "\n")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("mode", choices=["scale", "ab", "report"])
    ap.add_argument("--workload", choices=list(WORKLOADS), default="strong")
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--parent-lib")
    ap.add_argument("--profile")
    args = ap.parse_args()
    {"scale": scale, "ab": ab, "report": report}[args.mode](args)


if __name__ == "__main__":
    main()
