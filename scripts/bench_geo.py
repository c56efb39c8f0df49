#!/usr/bin/env python
"""bench_geo.py — haversine (geo) Vamana indexes on one GPU: build, search, recall, and the
visited-table sizes of the geo beam-search kernel (GeoEval, csrc/search_geo.cu).

    python scripts/bench_geo.py [--sizes 1000000,10000000] [--out profiles/r03_geo.json]

Data: synth.geo_points (clustered cities + 10 % uniform background, lat/lon degrees), queries
synth.geo_queries, 10 k per batch, k 10, L 75, R 64, alpha 1.2. Per size:
  build    batched insert from an empty index with the default schedule (three builds at the
           first size, one at the others): seconds, points/s, sdb_insert_stats, sdb_insert_truncated,
           and the build's GPU time per kernel (torch.profiler with CUDA activities, in one extra,
           untimed build at the first size: the library has no events between its build phases, and
           the profiler's kernel records are the only per-phase split available without adding any);
  search   device-resident batches (sdb_search_batch_device, warmed up), CUDA events around each
           batch, plus the beam-search kernel alone (sdb_search_profile); the same batch through
           sdb_search_batch with host buffers; hops and evaluations per query (sdb_last_search_stats)
           and the algorithmic bytes n_dist*16 + n_hops*R*4 per query;
  recall   recall@10 of 1 000 queries against the exact GPU flat scan (sdb_flat_search_batch), and the
           oracle's search on the GPU-built graph (OracleIndex.set_graph) against the same lists;
  slots    the insert-built handle searched with SDB_VT_SLOTS = 1024 .. 8192 (where the span is valid).
The CTAs/SM x slots sweep in profiles/r03_geo.json ("sweep") chose the geo kernel's launch bound;
the residency cap it varied has been removed since, so this script no longer repeats it.
Timing uses CUDA events and host clocks around synchronised work only. The card's name, power limit
and maximum SM clock are read with nvidia-smi (read-only query) in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

K, L, R, ALPHA, B = 10, 75, 64, 1.2, 10_000
SEED = 2026


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clk}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def slots_valid(rows, slots):
    """VisitedCompactN::init: span = ceil(2^b / buckets) must fit a 16-bit entry."""
    b = 1 if rows <= 2 else int(rows - 1).bit_length()
    b = max(b, 16)
    buckets = slots // 4
    return ((1 << b) + buckets - 1) // buckets <= 65534


def build(X, start, ids, profile=False):
    import torch
    from semadb_b200 import _capi
    from semadb_b200.vamana import IndexVamana, IndexVectorVamanaParameters
    g = IndexVamana("geo", IndexVectorVamanaParameters(2, "haversine", L, R, ALPHA), start_vector=start)
    g.reserve(int(ids[-1]))
    g.insert_stats(reset=True)
    torch.cuda.synchronize()
    prof = None
    if profile:
        from torch.profiler import ProfilerActivity, profile as tprof
        prof = tprof(activities=[ProfilerActivity.CUDA])
        prof.__enter__()
    t0 = time.perf_counter()
    g.insert_batch(ids, X)
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    kernels = None
    if prof is not None:
        prof.__exit__(None, None, None)
        rows = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = getattr(ev, "cuda_time_total", 0)
            if t:
                rows[ev.key[:120]] = {"ms": round(t / 1000.0, 3), "calls": ev.count}
        kernels = dict(sorted(rows.items(), key=lambda kv: -kv[1]["ms"])[:15])
    return g, {"seconds": round(secs, 3), "points_per_s": round(len(X) / secs), "insert_stats": g.insert_stats(),
               "insert_truncated": int(_capi.lib().sdb_insert_truncated(g._h)), "gpu_ms_by_kernel": kernels}


def search_device(g, Q, reps=5):
    import torch
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_q = torch.from_numpy(Q).to(dev)
    ids = torch.zeros((len(Q), K), dtype=torch.int64, device=dev)
    d = torch.zeros((len(Q), K), dtype=torch.float32, device=dev)
    c = torch.zeros((len(Q),), dtype=torch.int32, device=dev)
    for _ in range(2):
        g.search_batch_device(d_q, K, L, ids, d, c, st)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    g.search_profile(True)
    for a, b in ev:
        a.record()
        g.search_batch_device(d_q, K, L, ids, d, c, st)
        b.record()
    torch.cuda.synchronize()
    kern = g.search_profile_read()
    g.search_profile(False)
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    med = ms[len(ms) // 2]
    hops, nd = g.last_search_stats(len(Q))
    assert int(c.min().item()) >= 0
    return {"batch_ms": [round(x, 4) for x in ms], "qps": round(len(Q) / (med / 1e3)),
            "kernel_ms": [round(float(x), 4) for x in kern], "hops_mean": float(hops.mean()),
            "ndist_mean": float(nd.mean()), "ndist_p99": float(np.percentile(nd, 99)), "ndist_max": int(nd.max())}


def search_host(g, Q, reps=3):
    g.search_batch(Q, K, L)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        g.search_batch(Q, K, L)
        ts.append(time.perf_counter() - t0)
    med = sorted(ts)[len(ts) // 2]
    return {"batch_ms": [round(t * 1e3, 3) for t in ts], "qps": round(len(Q) / med)}


def graph_of(g, n_rows, chunk=1 << 20):
    """The GPU graph as the oracle's dense u32 [rows][R] + degrees (rows 0..n_rows-1)."""
    adj = np.full((n_rows, R), 0xFFFFFFFF, dtype=np.uint32)
    deg = np.zeros(n_rows, dtype=np.uint16)
    for s in range(1, n_rows, chunk):
        idx = np.arange(s, min(n_rows, s + chunk), dtype=np.uint64)
        dg, e = g.get_edges(idx)
        adj[s:s + len(idx)] = e.astype(np.uint32)
        deg[s:s + len(idx)] = dg
    return adj, deg


def recall(a, b):
    return float(np.mean([len(set(a[i].tolist()) & set(b[i].tolist())) / b.shape[1] for i in range(len(b))]))


def run_size(n, first, out_sizes):
    from oracle import oraclelib as O
    from semadb_b200 import synth
    from semadb_b200.vamana import IndexVamana, IndexVectorVamanaParameters
    X = synth.geo_points(n, SEED)
    Q = synth.geo_queries(B, SEED)
    ids = np.arange(2, n + 2, dtype=np.uint64)
    start = synth.start_vector(2, 99)
    res = {"n": n, "queries": B}
    builds = []
    g = None
    for i in range(3 if first else 1):
        if g is not None:
            g.close()
        g, info = build(X, start, ids)
        builds.append(info)
        print(f"[geo {n}] build {i}: {info['seconds']} s", flush=True)
    res["build"] = builds
    res["build_seconds_median"] = sorted(b["seconds"] for b in builds)[len(builds) // 2]
    if first:
        gp, info = build(X, start, ids, profile=True)
        res["build_profiled"] = {"seconds_under_profiler": info["seconds"], "gpu_ms_by_kernel": info["gpu_ms_by_kernel"]}
        gp.close()
    res["search_device"] = sd = search_device(g, Q)
    res["search_host_buffers"] = search_host(g, Q)
    res["algorithmic_bytes_per_query"] = round(sd["ndist_mean"] * 16 + sd["hops_mean"] * R * 4, 1)
    built = []
    for slots in (1024, 2048, 4096, 8192):
        row = {"slots": slots}
        if not slots_valid(n + 2, slots):
            row["result"] = "invalid: quotient span beyond 16 bits for this store"
        else:
            os.environ["SDB_VT_SLOTS"] = str(slots)
            r = search_device(g, Q)
            os.environ.pop("SDB_VT_SLOTS")
            row.update(qps=r["qps"], batch_ms=r["batch_ms"], kernel_ms=r["kernel_ms"])
        built.append(row)
        print(f"[geo {n}] built handle {row}", flush=True)
    res["slots_built_handle"] = built
    print(f"[geo {n}] search {sd['qps']} q/s, ndist {sd['ndist_mean']:.1f}, hops {sd['hops_mean']:.1f}", flush=True)
    # recall: exact GPU flat scan as ground truth; the oracle on the same (GPU-built) graph
    Qr = Q[:1000]
    fi, fd, fc = g.flat_search_batch(Qr, K)
    gi, gd, gc = g.search_batch(Qr, K, L)
    adj, deg = graph_of(g, n + 2)
    oix = O.OracleIndex(2, "haversine", L, R, ALPHA)
    oix.set_start(start)
    oix.set_vectors(ids.astype(np.uint32), X)
    oix.set_graph(adj, deg)
    ref = oix.search(Qr, k=K, threads=os.cpu_count() or 8)
    del oix
    res["recall_at_10"] = {"gpu_search_gpu_graph": recall(gi, fi), "oracle_search_gpu_graph": recall(ref["ids"].astype(np.uint64), fi),
                           "rows_identical_to_oracle": int(((gi == ref["ids"].astype(np.uint64)).all(1)).sum()),
                           "ground_truth": "sdb_flat_search_batch (exact haversine scan)", "flat_path": g.flat_last_stats()[0]}
    print(f"[geo {n}] recall {res['recall_at_10']}", flush=True)
    g.close()
    out_sizes.append(res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,10000000")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r03_geo.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_geo.py needs a CUDA device")
    out = {"card": card(), "config": {"k": K, "L": L, "R": R, "alpha": ALPHA, "batch": B, "seed": SEED,
                                      "data": "synth.geo_points (200 cities, spread 0.5 deg, 10 % uniform background)"},
           "note": ("The geo search reads 16-byte rows (8 used) and 256-byte adjacency rows; at ~450 evaluations and ~80 "
                    "hops per query that is ~28 KB per query. HBM bandwidth is not expected to bound this kernel (a "
                    "chain of ~80 dependent hops with float64 transcendental math per evaluation); no roofline "
                    "fraction is stated."),
           "sizes": []}
    for i, n in enumerate(int(s) for s in args.sizes.split(",")):
        run_size(n, i == 0, out["sizes"])
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(out, indent=1))
    print(json.dumps({"card": out["card"], "sizes": [{"n": s["n"], "qps": s["search_device"]["qps"]} for s in out["sizes"]]}))


if __name__ == "__main__":
    main()
