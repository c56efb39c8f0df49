"""Mixed per-request limits and searchSizes in one call against one call per (limit, searchSize) group.

Workload: 1M x 128 f32 squared-L2 points (the synth.sift_shaped law, C2-shaped), graph built on the
GPU, device-resident queries. Three beam-search arms at 1 024 requests (one coalescer batch) and at
10 000 requests:
    mixed   one sdb_search_batch_requests_device call over the whole mix;
    groups  one sdb_search_batch_device call per (limit, searchSize) group, in sequence on one stream
            (what a coalescer that only batches equal pairs issues);
    uniform the same requests all at k 10 / L 75 through sdb_search_batch_device.
The mix draws limits from {1, 5, 10, 37, 75} and searchSizes from {max(limit, 25), 25, 50, 75}
(>= limit; the reference's searchSize range is 25..75). Flat search over the same points: mixed
limits in one sdb_flat_search_batch_requests_device call against one sdb_flat_search_batch_device
call per limit group.

Each arm: median of --steps CUDA-event-timed calls after --warmup calls of the same shapes. The
points (512 MB) do not fit the 126 MB L2. The card name and power limit are read with nvidia-smi
(read-only query) in the same run.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

LIMITS = (1, 5, 10, 37, 75)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clk}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def mix(B, seed):
    rng = np.random.default_rng(seed)
    lim = np.array(LIMITS)[rng.integers(0, len(LIMITS), B)]
    L = np.array([rng.choice([x for x in (max(int(l), 25), 25, 50, 75) if x >= l]) for l in lim])
    return lim.astype(np.int64), L.astype(np.int64)


def timed(fn, steps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)), "steps": steps}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    from semadb_b200 import synth
    from semadb_b200.vamana import IndexFlat, IndexVamana, IndexVectorFlatParameters, IndexVectorVamanaParameters, PackedRequests
    dev = torch.device("cuda", 0)
    res = {"card": card(), "workload": f"{args.n} x 128 f32 squared-L2 (sift_shaped law), device-resident queries",
           "limits": LIMITS, "searchSizes": "max(limit, 25), 25, 50, 75 (>= limit)", "vamana": {}, "flat": {}}
    X = synth.sift_shaped(args.n, 128, seed=3, w_seed=3)
    ids = np.arange(2, args.n + 2, dtype=np.uint64)
    g = IndexVamana("bench", IndexVectorVamanaParameters(128, "euclidean"), device=0, start_seed=99)
    g.insert_batch_device(ids, torch.from_numpy(X).to(dev))
    torch.cuda.synchronize()
    f = IndexFlat(IndexVectorFlatParameters(128, "euclidean"), device=0)
    f.set_vectors(ids, X)
    del X
    st = lambda: torch.cuda.current_stream().cuda_stream
    for B in (1024, 10_000):
        Q = torch.from_numpy(synth.sift_shaped(B, 128, seed=4, w_seed=3)).to(dev)
        lim, L = mix(B, 5)
        KS = int(lim.max())
        out = (torch.zeros((B, KS), dtype=torch.int64, device=dev), torch.zeros((B, KS), dtype=torch.float32, device=dev),
               torch.zeros((B,), dtype=torch.int32, device=dev))
        rq = PackedRequests(B, lim, L)
        groups = sorted(set(zip(lim.tolist(), L.tolist())))
        sub = []
        for k, l in groups:
            idx = torch.from_numpy(np.nonzero((lim == k) & (L == l))[0]).to(dev)
            n = len(idx)
            sub.append((k, l, Q[idx].contiguous(), torch.zeros((n, k), dtype=torch.int64, device=dev),
                        torch.zeros((n, k), dtype=torch.float32, device=dev), torch.zeros((n,), dtype=torch.int32, device=dev)))

        def mixed():
            g.search_batch_requests_device(Q, rq, KS, *out, st())

        def per_group():
            for k, l, q, i, d, c in sub:
                g.search_batch_device(q, k, l, i, d, c, st())

        u = (torch.zeros((B, 10), dtype=torch.int64, device=dev), torch.zeros((B, 10), dtype=torch.float32, device=dev),
             torch.zeros((B,), dtype=torch.int32, device=dev))

        def uniform():
            g.search_batch_device(Q, 10, 75, *u, st())

        # the mixed call's rows equal the group calls' rows
        mixed()
        per_group()
        torch.cuda.synchronize()
        same = True
        for k, l, q, i, d, c in sub:
            idx = torch.from_numpy(np.nonzero((lim == k) & (L == l))[0]).to(dev)
            same = same and bool((out[0][idx, :k] == i).all().item()) and bool((out[1][idx, :k] == d).all().item()) and \
                bool((out[2][idx] == c).all().item())
        res["vamana"][str(B)] = {"groups": len(groups), "rows_equal_group_calls": same,
                                 "mixed": timed(mixed, args.steps, args.warmup),
                                 "groups_in_sequence": timed(per_group, args.steps, args.warmup),
                                 "uniform_k10_L75": timed(uniform, args.steps, args.warmup)}
        # flat: per limit group
        frq = PackedRequests(B, lim)
        fgroups = sorted(set(lim.tolist()))
        fsub = []
        for k in fgroups:
            idx = torch.from_numpy(np.nonzero(lim == k)[0]).to(dev)
            n = len(idx)
            fsub.append((k, Q[idx].contiguous(), torch.zeros((n, k), dtype=torch.int64, device=dev),
                         torch.zeros((n, k), dtype=torch.float32, device=dev), torch.zeros((n,), dtype=torch.int32, device=dev)))

        def fmixed():
            f.flat_search_batch_requests_device(Q, frq, KS, *out, st())

        def fgroup():
            for k, q, i, d, c in fsub:
                f.flat_search_batch_device(q, k, i, d, c, st())

        def funiform():
            f.flat_search_batch_device(Q, 10, *u, st())

        fmixed()
        fgroup()
        torch.cuda.synchronize()
        same = True
        for k, q, i, d, c in fsub:
            idx = torch.from_numpy(np.nonzero(lim == k)[0]).to(dev)
            same = same and bool((out[0][idx, :k] == i).all().item()) and bool((out[2][idx] == c).all().item())
        res["flat"][str(B)] = {"groups": len(fgroups), "rows_equal_group_calls": same,
                               "mixed": timed(fmixed, args.steps, args.warmup),
                               "groups_in_sequence": timed(fgroup, args.steps, args.warmup),
                               "uniform_k10": timed(funiform, args.steps, args.warmup)}
        print(json.dumps({"B": B, "vamana": res["vamana"][str(B)], "flat": res["flat"][str(B)]}), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
