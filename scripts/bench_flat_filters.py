#!/usr/bin/env python3
"""IndexFlat.Search with one filter per request (sdb_flat_search_batch_filters) on one GPU.

Store: 1M x 128 synth.sift_shaped, squared L2; batches of 10k requests; queries, outputs, filter ids,
offsets and per-request filter indices in page-locked host memory; warm-up, then timed calls.
Workloads:
  per-request random filters at 0.01 %, 0.1 % and 1 % of the store (each request its own filter);
  one filter shared by the batch at 0.1 % (gather route) and at 50 % (range-scan route);
  0.1 % per request on wider and quantised stores: 1.25M x 384 cosine, 1M x 1024-bit hamming,
  1M x 768 dot PQ M=96 K=256 (C4-shaped).
Per workload:
  wall_ms            end-to-end time of one call (host clock around a synchronous call), mean of the
                     timed calls, profiler off;
  kernel_ms, h2d_ms, d2h_ms   device time of the kernels and of the copies of one call, from a
                     torch.profiler pass of its own; host_ms = wall_ms - (kernel + copies): host
                     staging (validation, id lists, routing, work items) and launch gaps;
  gathered_pairs     (request, id) pairs the gather route scored (sdb_flat_last_filter_stats);
  gather_GBps, gather_frac_of_6553   gathered_pairs x row bytes over kernel time, and its share of
                     the 6 553 GB/s copy peak DESIGN.md uses;
  today_ms           the same requests served the way the library allowed before this entry: one
                     sdb_flat_search_batch call per distinct filter, through --baseline-lib (a build of
                     the library from before the per-request entry, whose filtered flat calls run the
                     range scan over the store) or, without it, through this build's single-filter
                     entry. Per-request filters: 1 000 calls timed (requests 0..999), the mean times
                     the batch's distinct filters; a shared filter: the one call, timed like the new entry;
  same_bytes         the new entry's rows equal those per-filter calls byte for byte.
Route constant: one filter of 16 384 random ids shared by 1, 128 and 1 024 requests on the 1M x 128
store, served by both routes (the second with SDB_FLAT_EXACT=1); per route, kernel time per gathered
pair and per scanned point-pass, and their ratio (FLAT_GATHER_PAIRS_PER_POINT in csrc/flat.cu).

usage: python scripts/bench_flat_filters.py [--out profiles/r03_flat_filters.json] [--only name,...]
                                           [--baseline-lib path/to/libsemadb_b200.so]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

from semadb_b200 import _capi, synth  # noqa: E402
from semadb_b200.vamana import (IndexFlat, IndexVamana, IndexVectorFlatParameters, IndexVectorVamanaParameters,  # noqa: E402
                                ProductQuantizerParameters, Quantizer)

K = 10
B = 10_000
COPY_PEAK_GBPS = 6553.0


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def pinned(a):
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t, t.numpy()


class Batch:
    """A batch in page-locked memory and the raw call of the new entry."""

    def __init__(self, g, Q, filters, qf):
        self.g, self.B = g, len(Q)
        lens = np.array([len(f) for f in filters], dtype=np.uint64)
        off = np.zeros(len(filters) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens)
        self._t = [pinned(Q), pinned(np.concatenate(filters) if off[-1] else np.zeros(1, np.uint64)), pinned(off),
                   pinned(qf if qf is not None else np.zeros(1, np.int32))]
        self.q, self.ids, self.off, self.qf = (t[1] for t in self._t)
        self.has_qf = qf is not None
        self.n_filters = len(filters)
        self.filters = filters
        self.qf_np = qf
        self.out = [pinned(np.zeros((self.B, K), np.uint64)), pinned(np.zeros((self.B, K), np.float32)),
                    pinned(np.zeros(self.B, np.uint32))]

    def call(self):
        o = [t[1] for t in self.out]
        _capi.check(self.g._lib.sdb_flat_search_batch_filters(
            self.g._h, self.B, self.q.ctypes.data_as(_capi.f32p), K, self.n_filters, self.ids.ctypes.data_as(_capi.u64p),
            self.off.ctypes.data_as(_capi.u64p), self.qf.ctypes.data_as(_capi.i32p) if self.has_qf else None,
            o[0].ctypes.data_as(_capi.u64p), o[1].ctypes.data_as(_capi.f32p), o[2].ctypes.data_as(_capi.u32p)))
        return o


def old_call(g, q, filt, out):
    _capi.check(g._lib.sdb_flat_search_batch(g._h, len(q), q.ctypes.data_as(_capi.f32p), K, filt.ctypes.data_as(_capi.u64p),
                                             len(filt), out[0].ctypes.data_as(_capi.u64p), out[1].ctypes.data_as(_capi.f32p),
                                             out[2].ctypes.data_as(_capi.u32p)))


def wall(fn, reps):
    fn()  # warm-up: scratch, modules
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t) * 1e3)
    return float(np.mean(ts)), float(np.min(ts)), float(np.max(ts))


def profiled(fn):
    """Device time of one call: kernels, host-to-device and device-to-host copies (ms)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        fn()
        torch.cuda.synchronize()
    kern = h2d = d2h = 0.0
    names = {}
    for e in p.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        n = e.name
        if "Memcpy HtoD" in n:
            h2d += us
        elif "Memcpy DtoH" in n:
            d2h += us
        elif "Memcpy" in n or "Memset" in n:
            pass
        else:
            kern += us
            m = re.search(r"(\w+)\s*[<(]", n)
            short = m.group(1) if m else n[:40]
            names[short] = names.get(short, 0.0) + us / 1e3
    return kern / 1e3, h2d / 1e3, d2h / 1e3, {k: round(v, 4) for k, v in sorted(names.items(), key=lambda x: -x[1])[:6]}


def load_baseline(path):
    """Another build of the library (its own handles), with the signatures it exports."""
    L = C.CDLL(str(path))
    for name, (res, args) in _capi._SIGS.items():
        if hasattr(L, name):
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
    return L


def build_with(lib, build):
    """build() with every handle it creates on `lib`."""
    if lib is None:
        return build()
    saved = _capi._lib
    _capi._lib = lib
    try:
        return build()
    finally:
        _capi._lib = saved


def sample_filter(rng, ids, m):
    return np.sort(rng.choice(ids, size=m, replace=False)).astype(np.uint64)


def per_request_filters(rng, n, m, count):
    """count sorted random id sets of about m ids of [2, n+2) (duplicate draws merged)."""
    return [np.unique(rng.integers(2, n + 2, size=m, dtype=np.uint64)) for _ in range(count)]


def run_workload(name, g, gb, Q, filters, qf, row_bytes, reps, today_calls=1000):
    log(f"[{name}] {len(filters)} filters, {sum(len(f) for f in filters)} ids")
    bt = Batch(g, Q, filters, qf)
    w_mean, w_min, w_max = wall(bt.call, reps)
    res = [x.copy() for x in bt.call()]
    gathered, scanned, pairs = g.flat_last_filter_stats()
    kern, h2d, d2h, top = profiled(bt.call)
    r = {"workload": name, "requests": len(Q), "filters": len(filters),
         "filter_ids_total": int(sum(len(f) for f in filters)), "filter_id_bytes_u64": int(8 * sum(len(f) for f in filters)),
         "wall_ms": round(w_mean, 3), "wall_ms_min": round(w_min, 3), "wall_ms_max": round(w_max, 3), "timed_calls": reps,
         "kernel_ms": round(kern, 3), "h2d_ms": round(h2d, 3), "d2h_ms": round(d2h, 3),
         "host_ms": round(w_mean - kern - h2d - d2h, 3), "top_kernels_ms": top,
         "gathered_filters": gathered, "scanned_filters": scanned, "gathered_pairs": pairs, "row_bytes": row_bytes}
    if pairs:
        gbps = pairs * row_bytes / (kern * 1e-3) / 1e9
        r["gather_GBps"] = round(gbps, 1)
        r["gather_frac_of_6553"] = round(gbps / COPY_PEAK_GBPS, 4)
    r["bound"] = max(("kernel", kern), ("h2d copies", h2d), ("host staging", w_mean - kern - h2d - d2h), key=lambda x: x[1])[0]
    # today's cost: one sdb_flat_search_batch per distinct filter
    g = gb if gb is not None else g
    r["today_library"] = "baseline build (--baseline-lib)" if gb is not None else "this build"
    out1 = [np.zeros((1, K), np.uint64), np.zeros((1, K), np.float32), np.zeros(1, np.uint32)]
    same = True
    if qf is None:  # one shared filter: one call with the whole batch
        outb = [t[1] for t in bt.out]
        qp = bt.q
        t_mean, _, _ = wall(lambda: old_call(g, qp, filters[0], outb), max(2, reps))
        old_call(g, qp, filters[0], outb)
        same = all(a.tobytes() == b.tobytes() for a, b in zip(res, outb))
        r["today_ms"] = round(t_mean, 3)
        r["today_calls"] = 1
    else:
        n = min(today_calls, len(Q))
        for b in range(2):
            old_call(g, bt.q[b:b + 1], filters[qf[b]], out1)  # warm-up
        t = time.perf_counter()
        for b in range(n):
            old_call(g, bt.q[b:b + 1], filters[qf[b]], out1)
        per_call = (time.perf_counter() - t) * 1e3 / n
        for b in range(n):
            old_call(g, bt.q[b:b + 1], filters[qf[b]], out1)
            same &= res[0][b].tobytes() == out1[0][0].tobytes() and res[1][b].tobytes() == out1[1][0].tobytes() and \
                res[2][b] == out1[2][0]
        distinct = len(set(int(x) for x in qf if x >= 0))
        r["today_calls_timed"] = n
        r["today_ms_per_call"] = round(per_call, 4)
        r["today_ms"] = round(per_call * distinct, 1)
        r["today_basis"] = f"{n} calls timed, mean x {distinct} distinct filters"
    r["same_bytes"] = bool(same)
    r["speedup_vs_today"] = round(r["today_ms"] / w_mean, 2)
    log(json.dumps(r))
    return r


def route_constant(g, n, rng):
    """Kernel time of both routes for one shared 16 384-id filter over 1, 128 and 1 024 requests."""
    filt = sample_filter(rng, np.arange(2, n + 2, dtype=np.uint64), 16384)
    rows = []
    for nf in (1, 128, 1024):
        Q = synth.sift_shaped(nf, 128, seed=40 + nf, w_seed=3)
        bt = Batch(g, Q, [filt], None)
        os.environ.pop("SDB_FLAT_EXACT", None)
        kg = profiled(bt.call)[0]
        st_g = g.flat_last_filter_stats()
        a = [x.copy() for x in bt.call()]
        os.environ["SDB_FLAT_EXACT"] = "1"
        ks = profiled(bt.call)[0]
        st_s = g.flat_last_filter_stats()
        b = bt.call()
        os.environ.pop("SDB_FLAT_EXACT", None)
        passes = (nf + 127) // 128
        ns_pair = kg * 1e6 / (nf * len(filt))
        ns_point = ks * 1e6 / (passes * n)
        rows.append({"requests": nf, "filter_ids": len(filt), "gather_kernel_ms": round(kg, 4), "scan_kernel_ms": round(ks, 4),
                     "gather_ns_per_pair": round(ns_pair, 5), "scan_ns_per_point_pass": round(ns_point, 5),
                     "pairs_per_point": round(ns_point / ns_pair, 2), "stats_default": st_g, "stats_forced_scan": st_s,
                     "same_bytes": all(x.tobytes() == y.tobytes() for x, y in zip(a, b))})
        log(json.dumps(rows[-1]))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r03_flat_filters.json"))
    ap.add_argument("--only", default="", help="comma list of: route,l2,shared,c3,bq,pq")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--baseline-lib", default="", help="a build of the library before the per-request entry, for today_ms")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_flat_filters.py needs a GPU")
    only = set(a.only.split(",")) if a.only else {"route", "l2", "shared", "c3", "bq", "pq"}
    result = {"card": card(), "k": K, "batch": B, "copy_peak_GBps": COPY_PEAK_GBPS, "workloads": []}
    log("card:", result["card"])
    rng = np.random.Generator(np.random.PCG64(2024))
    base = load_baseline(a.baseline_lib) if a.baseline_lib else None
    result["today_library"] = ("a build of the library before the per-request entry (--baseline-lib)" if a.baseline_lib
                               else "this build's single-filter entry")

    def stores(build):
        g = build()
        return g, build_with(base, build) if base is not None else None

    n = 1_000_000
    if only & {"route", "l2", "shared"}:
        def build_l2():
            g = IndexFlat(IndexVectorFlatParameters(128, "euclidean"))
            g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), synth.sift_shaped(n, 128, seed=3))
            return g
        g, gb = stores(build_l2)
        Q = synth.sift_shaped(B, 128, seed=4, w_seed=3)
        if "route" in only:
            result["route_constant"] = route_constant(g, n, rng)
        if "l2" in only:
            for frac, m in (("0.01%", 100), ("0.1%", 1000), ("1%", 10000)):
                fs = per_request_filters(rng, n, m, B)
                result["workloads"].append(run_workload(f"1M x 128 L2, per-request filters {frac}", g, gb, Q, fs,
                                                        np.arange(B, dtype=np.int32), 512, a.reps if m < 10000 else 3))
                del fs
        if "shared" in only:
            ids = np.arange(2, n + 2, dtype=np.uint64)
            for frac, m in (("0.1%", 1000), ("50%", n // 2)):
                result["workloads"].append(run_workload(f"1M x 128 L2, one shared filter {frac}", g, gb, Q,
                                                        [sample_filter(rng, ids, m)], None, 512, a.reps))
        del g, gb
        torch.cuda.empty_cache()
    if "c3" in only:
        n3 = 1_250_000

        def build_c3():
            g = IndexFlat(IndexVectorFlatParameters(384, "cosine"))
            for s in range(0, n3, 250_000):
                Xc = synth.latent_gaussian(min(250_000, n3 - s), 384, seed=5 + s, w_seed=5, latent=32, normalize=True)
                g.set_vectors(np.arange(2 + s, 2 + s + len(Xc), dtype=np.uint64), Xc)
            return g
        g, gb = stores(build_c3)
        Q = synth.latent_gaussian(B, 384, seed=6, w_seed=5, latent=32, normalize=True)
        fs = per_request_filters(rng, n3, n3 // 1000, B)
        result["workloads"].append(run_workload("1.25M x 384 cosine, per-request filters 0.1%", g, gb, Q, fs,
                                                np.arange(B, dtype=np.int32), 1536, a.reps))
        del g, gb, fs
    if "bq" in only:
        nb, dim = 1_000_000, 1024

        def build_bq():
            g = IndexVamana("bq", IndexVectorVamanaParameters(dim, "hamming"), start_vector=synth.start_vector(dim, 5))
            for s in range(0, nb, 100_000):
                Xc = synth.planted_bits(100_000, dim, seed=7 + s, n_proto=4096, proto_seed=7)
                g.set_vectors(np.arange(2 + s, 2 + s + len(Xc), dtype=np.uint64), Xc)
            return g
        g, gb = stores(build_bq)
        Q = synth.planted_bits(B, dim, seed=10, n_proto=4096, proto_seed=7)
        fs = per_request_filters(rng, nb, nb // 1000, B)
        result["workloads"].append(run_workload("1M x 1024-bit hamming, per-request filters 0.1%", g, gb, Q, fs,
                                                np.arange(B, dtype=np.int32), 128, a.reps))
        del g, gb, fs
    if "pq" in only:
        n4, dim, M, KC = 1_000_000, 768, 96, 256

        def build_pq():
            q = Quantizer("product", product=ProductQuantizerParameters(KC, M, 10000))
            g = IndexVamana("c4", IndexVectorVamanaParameters(dim, "dot", quantizer=q), start_vector=synth.start_vector(dim, 99))
            g.set_vectors(np.arange(2, 10_002, dtype=np.uint64), synth.latent_gaussian(10_000, dim, seed=8, latent=64))
            assert g.fit(0)
            for s in range(10_000, n4, 200_000):
                Xc = synth.latent_gaussian(min(200_000, n4 - s), dim, seed=8 + s, w_seed=8, latent=64)
                g.set_vectors(np.arange(2 + s, 2 + s + len(Xc), dtype=np.uint64), Xc)
            return g
        g, gb = stores(build_pq)
        Q = synth.latent_gaussian(B, dim, seed=9, w_seed=8, latent=64)
        fs = per_request_filters(rng, n4, n4 // 1000, B)
        result["workloads"].append(run_workload("1M x 768 dot PQ M=96 K=256 (C4-shaped), per-request filters 0.1%", g, gb, Q,
                                                fs, np.arange(B, dtype=np.int32), 96, a.reps))
        del g, gb, fs
    result["card_after"] = card()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps({"out": a.out, "workloads": len(result["workloads"])}))


if __name__ == "__main__":
    main()
