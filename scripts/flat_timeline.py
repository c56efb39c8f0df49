#!/usr/bin/env python
"""K5 (IndexFlat.Search, 10k queries x 1M x 128 f32 L2, k = 10) through sdb_flat_search_batch:
  * wall time per call with pageable numpy buffers and with page-locked buffers (host buffers in
    and out either way, copies inside the timed region);
  * one call's kernel timeline (torch.profiler / CUPTI: name, start offset, duration) so that the
    share of every launch of the call is on record (profiles/r02_flat_timeline.json).
usage: python scripts/flat_timeline.py [--n 1000000] [--B 10000] [--reps 5] [--timeline]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from semadb_b200 import _capi, synth  # noqa: E402
from semadb_b200.vamana import IndexFlat, IndexVectorFlatParameters  # noqa: E402

K = 10


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--B", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--timeline", action="store_true")
    ap.add_argument("--tag", default="")
    a = ap.parse_args()
    n, B = a.n, a.B
    X = synth.sift_shaped(n, 128, 3)
    Q = synth.sift_shaped(B, 128, 4, w_seed=3)
    g = IndexFlat(IndexVectorFlatParameters(128, "euclidean"))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    lib = _capi.lib()

    ref_ids, ref_d, _ = g.flat_search_batch(Q, K)  # warm-up: scratch, bf16 shadow
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(a.reps):
        g.flat_search_batch(Q, K)
    pageable = (time.perf_counter() - t) / a.reps

    h_q = torch.from_numpy(Q).pin_memory()
    h_ids = torch.zeros((B, K), dtype=torch.int64).pin_memory()
    h_d = torch.zeros((B, K), dtype=torch.float32).pin_memory()
    h_c = torch.zeros((B,), dtype=torch.int32).pin_memory()

    def call():
        _capi.check(lib.sdb_flat_search_batch(g._h, B, C.cast(h_q.data_ptr(), _capi.f32p), K, None, 0,
                                              C.cast(h_ids.data_ptr(), _capi.u64p), C.cast(h_d.data_ptr(), _capi.f32p),
                                              C.cast(h_c.data_ptr(), _capi.u32p)))

    call()
    times = []
    for _ in range(a.reps):
        t = time.perf_counter()
        call()
        times.append(time.perf_counter() - t)
    pinned = float(np.median(times))
    same = bool((h_ids.numpy().view(np.uint64) == ref_ids).all() and h_d.numpy().tobytes() == ref_d.tobytes())
    path, cand, ovf = g.flat_last_stats()
    out = {"config": "flat", "tag": a.tag, "env": {k: v for k, v in os.environ.items() if k.startswith("SDB_FLAT")},
           "workload": f"IndexFlat.Search {B} queries x {n} x 128 f32 L2, k={K}, host buffers in and out",
           "pageable_ms": pageable * 1e3, "pinned_ms": pinned * 1e3, "pinned_ms_all": [x * 1e3 for x in times],
           "pinned_qps": B / pinned, "tflops_useful_pinned": 2.0 * B * n * 128 / pinned / 1e12,
           "pinned_equals_pageable_results": same, "path": path, "candidates_last_level": cand, "overflowed": ovf}
    if a.timeline:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        evs.sort(key=lambda e: e.time_range.start)
        if evs:
            t0 = evs[0].time_range.start
            out["timeline_us"] = [[e.name[:60], round(e.time_range.start - t0, 1), round(e.time_range.end - e.time_range.start, 1)]
                                  for e in evs]
            out["timeline_span_us"] = round(max(e.time_range.end for e in evs) - t0, 1)
            out["timeline_busy_us"] = round(sum(e.time_range.end - e.time_range.start for e in evs), 1)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
