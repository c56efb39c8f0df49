#!/usr/bin/env python
"""bench.py — Vamana search throughput on the BASELINE.json configs on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c2|c3|c4|c5b|c5a] [--extra auto|none|c3,c5b,...] [--dump-outputs DIR]

The default line (what the driver runs) is C2, the config the metric is quoted on: a "step" is
one pass of the hot path over one 10k-query batch — batched greedy beam search (K1) over a
1M x 128 f32 L2 shard per GPU (R=64, L=75, alpha=1.2, k=10), searching the reference-built
graph, plus, at N>1, the cross-shard exchange fused into the search epilogue (peer stores over
NVLink + flag barrier) and the merge kernel (K6).

  value   = shard-searches per second over the whole job = n_gpus * batch / step time,
            queries resident in HBM, timed with CUDA events (max over ranks). Every query
            visits every shard (cluster/actions.go:316-376), so the end-user QPS over the
            N x 1M collection is value / n_gpus (config.user_qps).
  e2e     = the same metric through the C-ABI call with HOST (page-locked) query / result
            buffers: H2D + kernels + D2H inside the timed region.
  roofline= algorithmic bytes per launch (n_dist*row_bytes + n_hops*R*4 per query, counted by
            the kernel itself) / the beam-search kernel's duration, measured with CUDA events
            around that kernel inside the same timed loop (sdb_search_profile), vs the
            measured HBM copy bandwidth.
  cpu_baseline / --impl reference = the reference-equivalent C++ restatement (oracle/) timed
            on this box's host cores on the same graph. The Go reference itself cannot be
            built in this image (no Go toolchain).
  extra_configs = further BASELINE.json configs measured in the same run, untimed setup +
            timed search each: c5a (batched graph build, K8, at every N: each GPU builds its
            own 1M x 128 shard) and, at --gpus 8, c3 (10M x 384 cosine, 1.25M per GPU) and c5b
            (50M x 1024-bit hamming, 6.25M per GPU) with merged recall, per-GPU HBM fraction and
            a 1k-query oracle parity probe at shard size. `--workload X` makes X the headline.
            At N = 1 also `flat` (K5): IndexFlat.Search of the whole batch over the headline
            shard through sdb_flat_search_batch with page-locked buffers, lists compared with
            the exact scan's, useful TFLOP/s against the measured bf16 peak.

Nothing on a timed GPU path touches oracle/: it builds the C2 graph during untimed input
preparation ("searching the reference-built graph"), serves as the parity checker in the
untimed tail and as the CPU baseline.

--dump-outputs DIR writes what the headline's last timed step returned to its caller as DIR/<name>.npy
(float32 / float64, under 64 MB in all: past that a seeded sample of rows, listed in rows.npy), for comparing
two builds output for output. Every input of the timed path is the same in every run with the same
arguments: points and queries are seeded, and the reference-built C2 graph is inserted on all host cores
in rounds of at most ORACLE_ROUND points (OracleIndex.insert max_round), which make it independent of
the core count and of thread timing. The bench writes nothing into the repository tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

L, R, ALPHA, K = 75, 64, 1.2, 10
# points per round of the reference-built graph: a few times the reference's concurrent workers in
# flight, same recall and hop count as their graph at 100k points
ORACLE_ROUND = 64
DUMP_BYTES = 60_000_000  # array bytes of --dump-outputs: with the .npy headers, under 64 MB
_OUT = sys.stdout
_T0 = time.time()

# BASELINE.json configs (BASELINE.md §4). n = points per GPU shard; row_bytes = bytes gathered per
# distance evaluation (SURVEY.md §8d); seeds as BASELINE.md.
WORKLOADS = {
    "c2": dict(dim=128, metric="euclidean", n=1_000_000, row_bytes=512, data_seed=3, query_seed=4, integer=False,
               desc="C2: SIFT-shaped synthetic {n}x128 f32 L2 Vamana shard per GPU"),
    "c3": dict(dim=384, metric="cosine", n=1_250_000, row_bytes=1536, data_seed=5, query_seed=6, integer=False,
               desc="C3: sentence-embedding-shaped {n}x384 (latent-16, L2-normalised) cosine Vamana shard per GPU"),
    "c4": dict(dim=768, metric="dot", n=1_250_000, row_bytes=96, data_seed=8, query_seed=9, integer=False,
               desc="C4: {n}x768 (latent-16, L2-normalised) dot-product shard per GPU, product quantizer M=96 K=256 "
                    "trained on the first 10k points, ADC table search"),
    # the same points under the cosine metric (PQ then works on squared L2, product.go:52-61): for
    # L2-normalised vectors the ranking is the dot product's, but distances are positive, so alpha scales
    # them the way robustPrune expects (search.go:132) — with "dot" the distances are negative and the
    # reference's prune keeps ~9 edges per node (both implementations alike; BASELINE.md §4)
    "c4cos": dict(dim=768, metric="cosine", n=1_250_000, row_bytes=96, data_seed=8, query_seed=9, integer=False,
                  desc="C4 (cosine variant): {n}x768 (latent-16, L2-normalised) cosine shard per GPU, product quantizer M=96 "
                       "K=256 trained on the first 10k points, ADC table search"),
    "c5b": dict(dim=1024, metric="hamming", n=6_250_000, row_bytes=128, data_seed=7, query_seed=10, integer=True,
                desc="C5b: {n}x1024-bit binary-quantized (sign bits of a latent-16 embedding) hamming Vamana shard per GPU"),
}


PQ_WORKLOADS = ("c4", "c4cos")


def log(*a):
    print(f"[{time.time() - _T0:7.1f}s]", *a, file=sys.stderr, flush=True)


def dump_rows(n, row_bytes):
    """Rows of an n-row output that --dump-outputs keeps: None (all of them) up to DUMP_BYTES,
    else a fixed seeded sample, sized to leave room for its own float64 index."""
    if n * row_bytes <= DUMP_BYTES:
        return None
    return np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // (row_bytes + 8), replace=False))


def dump_outputs(out_dir, arrays):
    """Writes each array (same number of rows, float32 / float64) as out_dir/<name>.npy; a sample
    of rows (dump_rows) is listed in rows.npy."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    n = len(next(iter(arrays.values())))
    keep = dump_rows(n, sum(a.nbytes for a in arrays.values()) // max(1, n))
    if keep is not None:
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays["rows"] = keep.astype(np.float64)
    for k, a in arrays.items():
        np.save(out_dir / f"{k}.npy", np.ascontiguousarray(a))
    log(f"outputs written to {out_dir}: " + ", ".join(f"{k} {a.shape} {a.dtype}" for k, a in arrays.items()))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def kernel_source_hash():
    """sha of the beam-search kernel sources: a committed ncu traffic figure is only quoted for
    the kernel it was captured from."""
    import hashlib
    h = hashlib.sha256()
    for f in ("search.cuh", "search_launch.cuh", "search.cu", "common.cuh"):
        h.update((ROOT / "semadb_b200" / "csrc" / f).read_bytes())
    return h.hexdigest()[:16]


def measured_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture of
    this same command (profiles/k1_traffic.json) — refused (None) when the capture was taken from
    other kernel sources than the ones in this tree."""
    p = ROOT / "profiles" / "k1_traffic.json"
    try:
        t = json.loads(p.read_text())
        if t.get("kernel_source_sha16") != kernel_source_hash():
            return None
        return float(t["dram_bytes_read"]) + float(t["dram_bytes_write"])
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                pw.append(float(r[3]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------

def c2_data(n, rank, nq):
    from semadb_b200 import synth
    X = synth.sift_shaped(n, 128, seed=3 + 1000 * rank, w_seed=3)
    Q = synth.sift_shaped(nq, 128, seed=4, w_seed=3)
    return X, Q


def device_chunks(name, n, rank, dev, queries=False, nq=0):
    """Device-generated points (or queries) of a workload, as (start, chunk) pairs."""
    from semadb_b200 import synth
    w = WORKLOADS[name]
    seed = w["query_seed"] if queries else w["data_seed"] + 1000 * rank
    m = nq if queries else n
    if name == "c5b":
        return synth.sign_bits_torch(m, w["dim"], seed, dev, w_seed=w["data_seed"], latent=16)
    return synth.latent_gaussian_torch(m, w["dim"], seed, dev, w_seed=w["data_seed"], latent=16, normalize=True)


def build_oracle_index(X, start, threads, dim=128, metric="euclidean"):
    from oracle import oraclelib as O
    oix = O.OracleIndex(dim, metric, L, R, ALPHA)
    oix.set_start(start)
    ids = np.arange(2, len(X) + 2, dtype=np.uint32)
    t = time.time()
    oix.insert(ids, X, threads=threads, max_round=ORACLE_ROUND)
    return oix, ids, time.time() - t


def workload_config(name, n, B, world, graph):
    w = WORKLOADS[name]
    adj_mb = n * R * 4 / 1e6
    data_mb = n * w["row_bytes"] / 1e6
    return {"workload": w["desc"].format(n=n) + f" (R={R}, L={L}, alpha={ALPHA}), {B}-query batch, k={K}",
            "points_per_gpu": n, "dim": w["dim"], "batch": B, "k": K, "search_size": L, "degree_bound": R, "graph": graph,
            "l2_policy": f"dataset (rows+adjacency {data_mb + adj_mb:.0f} MB/GPU) >> 126 MB L2, no explicit flush",
            "parallelism": f"shard-per-gpu x{world}, queries broadcast, per-GPU top-k exchanged and merged on every GPU"
            if world > 1 else "single shard"}


# ------------------------------------------------------------------------------------------
# --impl reference
# ------------------------------------------------------------------------------------------

def run_reference(args):
    """--impl reference: the reference-equivalent C++ restatement of the CPU path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import oraclelib as O
    from semadb_b200 import synth
    threads = O.hw_threads()
    n = args.n or WORKLOADS["c2"]["n"]
    X, Q = c2_data(n, 0, args.queries)
    oix, ids, tb = build_oracle_index(X, synth.start_vector(128, 99), threads)
    log(f"[reference] graph built in {tb:.1f}s with {threads} threads")
    nq = min(args.queries, args.ref_queries)
    for _ in range(args.warmup):
        oix.search(Q[:nq], k=K, search_size=L, threads=threads)
    t0 = time.time()
    for _ in range(args.steps):
        oix.search(Q[:nq], k=K, search_size=L, threads=threads)
    dt = (time.time() - t0) / args.steps
    qps = nq / dt
    cfg = workload_config("c2", n, args.queries, world, "oracle")
    if world > 1:
        cfg["note"] = (f"shard-searches/s of the host CPU measured on one {n}-point shard: a query over the {world}-shard "
                       f"collection costs the host {world} of them, so its user-visible QPS is value / {world}")
    cfg["user_qps"] = qps / world
    out = {
        "impl": "reference", "metric": "vamana_search_qps", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
                         "sample": f"{nq} of {args.queries} queries per step, {threads} threads, one query per thread"},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), file=_OUT, flush=True)


def _quarantine_stdout():
    """Libraries (NCCL's version banner, torchrun notices) write to fd 1; the driver expects
    exactly one JSON line there. Route fd 1 to stderr and keep a private handle for the line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------

class Ctx:
    """Process-wide state of one bench run (rank, device, torch.distributed handles)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.args = args
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.ncpu = os.cpu_count() or 1

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, vals):
        if self.world == 1:
            return [float(v) for v in vals]
        t = self.torch.tensor(vals, dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def min_over_ranks(self, val):
        if self.world == 1:
            return float(val)
        t = self.torch.tensor([val], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return float(t.item())


def new_index(name, rank, local_rank):
    from semadb_b200 import synth
    from semadb_b200.vamana import (IndexVamana, IndexVectorVamanaParameters, ProductQuantizerParameters, Quantizer)
    w = WORKLOADS[name]
    q = Quantizer("product", product=ProductQuantizerParameters(256, 96, 10000)) if name in PQ_WORKLOADS else None
    start = synth.start_vector(w["dim"], 99 + rank)
    g = IndexVamana(name, IndexVectorVamanaParameters(w["dim"], w["metric"], L, R, ALPHA, q), device=local_rank,
                    start_vector=start)
    return g, start


def build_device_generated(cx, name, n, Qr):
    """Untimed setup of a device-generated workload: K8 batched insert of n points per GPU, the
    points produced chunk by chunk on the device. Returns (index, start vector, build seconds,
    float ground truth of the recall queries or None)."""
    torch = cx.torch
    g, start = new_index(name, cx.rank, cx.local_rank)
    g.reserve(n + 2)
    if os.environ.get("SDB_INSERT_CONFIG"):  # "min,max,growth_div": A/B of the mini-batch schedule
        g.insert_config(*[int(x) for x in os.environ["SDB_INSERT_CONFIG"].split(",")])
    t_ins = 0.0
    fit_s = None
    truth = None
    if name in PQ_WORKLOADS:  # exact -dot top-k of the recall queries over this shard, accumulated chunk by chunk (fp32)
        torch.backends.cuda.matmul.allow_tf32 = False
        d_qr = torch.from_numpy(Qr).to(cx.dev)
        best_d = torch.full((len(Qr), K), float("inf"), device=cx.dev)
        best_i = torch.zeros((len(Qr), K), dtype=torch.int64, device=cx.dev)
    for s, x in device_chunks(name, n, cx.rank, cx.dev):
        ids = np.arange(2 + s, 2 + s + len(x), dtype=np.uint64)
        if name in PQ_WORKLOADS:
            sc = -(d_qr @ x.T)
            cd, ci = torch.topk(sc, K, dim=1, largest=False)
            alld = torch.cat([best_d, cd], 1)
            alli = torch.cat([best_i, ci + (2 + s)], 1)
            o = torch.argsort(alld, dim=1, stable=True)[:, :K]
            best_d, best_i = torch.gather(alld, 1, o), torch.gather(alli, 1, o)
        torch.cuda.synchronize()
        t = time.time()
        if name in PQ_WORKLOADS and fit_s is None:
            g.insert_batch_device(ids[:10000], x[:10000].contiguous())
            t1 = time.time()
            g.fit(0)
            fit_s = time.time() - t1
            g.insert_batch_device(ids[10000:], x[10000:].contiguous())
        else:
            g.insert_batch_device(ids, x)
        t_ins += time.time() - t
        del x
    if name in PQ_WORKLOADS:
        truth = (best_i.cpu().numpy().astype(np.uint64), best_d.cpu().numpy())
    return g, start, t_ins, fit_s, truth


def merged_truth(cx, t_ids, t_d):
    """Per-rank exact top-k lists -> exact top-k of the union (ids tagged shard << 40)."""
    torch, dist = cx.torch, cx.dist
    from semadb_b200.sharded import SHARD_SHIFT
    ids = torch.from_numpy(t_ids.astype(np.int64)).to(cx.dev) + (cx.rank << SHARD_SHIFT)
    d = torch.from_numpy(t_d).to(cx.dev)
    if cx.world == 1:
        return ids.cpu().numpy(), d.cpu().numpy()
    gi = [torch.empty_like(ids) for _ in range(cx.world)]
    gd = [torch.empty_like(d) for _ in range(cx.world)]
    dist.all_gather(gi, ids)
    dist.all_gather(gd, d)
    ai, ad = torch.cat(gi, 1), torch.cat(gd, 1)
    o = torch.argsort(ad, dim=1, stable=True)[:, :K]
    return torch.gather(ai, 1, o).cpu().numpy(), torch.gather(ad, 1, o).cpu().numpy()


def recall_of(got_ids, got_d, got_c, true_ids, true_d):
    nq = len(true_ids)
    strict, tie = [], []
    for b in range(nq):
        c = int(got_c[b])
        strict.append(len(set(got_ids[b, :c].tolist()) & set(true_ids[b].tolist())) / K)
        tie.append(float((got_d[b, :c] <= true_d[b, K - 1]).sum()) / K)
    return float(np.mean(strict)), float(np.mean(tie))


def oracle_probe(cx, name, g, start, n, Q, local_ids, local_d, oix=None):
    """1k-query parity probe at shard size on rank 0: the oracle searches the SAME graph (downloaded
    from the device unless it built it) and must return the same ids and bit-identical distances
    as this rank's shard-local GPU result."""
    from oracle import oraclelib as O
    w = WORKLOADS[name]
    nq = len(Q)
    t = time.time()
    if oix is None:
        if name in PQ_WORKLOADS:
            oix = O.OracleIndex(w["dim"], w["metric"], L, R, ALPHA, quantizer="product", pq_m=96, pq_k=256, pq_trigger=10000)
            fc, cd = g.get_pq()
            oix.set_pq(fc, cd, reencode=False)
        else:
            oix = O.OracleIndex(w["dim"], w["metric"], L, R, ALPHA)
        ids = np.arange(1, n + 2, dtype=np.uint64)
        adj = np.full((n + 2, R), 0xFFFFFFFF, dtype=np.uint32)
        deg = np.zeros(n + 2, dtype=np.uint16)
        step = 1 << 20
        for s in range(0, len(ids), step):
            dg, e = g.get_edges(ids[s:s + step])
            m = np.arange(R)[None, :] < dg[:, None]
            blk = adj[1 + s:1 + s + len(dg)]
            blk[m] = e[m].astype(np.uint32)
            deg[1 + s:1 + s + len(dg)] = dg
        if name == "c5b" or name in PQ_WORKLOADS:
            for s in range(0, len(ids), step):  # codes only, like hydrating n<id>q keys
                oix.set_codes(ids[s:s + step].astype(np.uint32), g.get_codes(ids[s:s + step]))
        else:
            oix.set_start(start)
            for s in range(1, len(ids), step):
                oix.set_vectors(ids[s:s + step].astype(np.uint32), g.get_vectors(ids[s:s + step]))
        oix.set_graph(adj, deg)
        del adj
    ref = oix.search(Q, k=K, search_size=L, threads=O.hw_threads())
    same = float((local_ids[:nq] == ref["ids"].astype(np.int64)).all(axis=1).mean())
    bits = bool(local_d[:nq].tobytes() == ref["dists"].tobytes())
    return {"queries": nq, "id_rows_identical_to_oracle": same, "dists_bit_identical": bits,
            "seconds": round(time.time() - t, 1)}, oix, ref


def run_search(cx, name, n, B, steps, warmup, graph, headline):
    """Untimed setup + timed search of one workload. Returns the measured pieces as a dict."""
    torch = cx.torch
    from semadb_b200 import _capi
    from semadb_b200.sharded import ShardedSearcher
    args = cx.args
    w = WORKLOADS[name]
    lib = _capi.lib()
    rank, world, dev = cx.rank, cx.world, cx.dev
    replicated = args.mode == "replicated"
    data_rank = 0 if replicated else rank  # replicas hold the same points
    nq_recall = min(args.recall_queries, B)
    oix = None
    X = None
    fit_s = None
    truth_float = None
    t0 = time.time()
    if name == "c2":
        from semadb_b200 import synth
        X, Q = c2_data(n, data_rank, B)
        start = synth.start_vector(128, 99 + data_rank)
        g, _ = new_index("c2", data_rank, cx.local_rank)
        ids = np.arange(2, n + 2, dtype=np.uint64)
        if graph == "oracle":
            # BASELINE.json config[1]: "searching the reference-built graph" — at every N, so that the
            # scaling curve compares like with like (N ranks share the host cores during this setup)
            threads = max(1, cx.ncpu // world)
            oix, _, tb = build_oracle_index(X, start, threads)
            log(f"[rank {rank}] {name}: reference-built graph: {tb:.1f}s on {threads} threads")
            g.set_vectors(ids, X)
            adj, deg = oix.get_graph()
            g.set_graph_dense(adj[1:], deg[1:], first_id=1)
            del adj
            build_s = tb
        else:
            t = time.time()
            g.insert_batch(ids, X)
            build_s = time.time() - t
    else:
        Q = torch.cat([x for _, x in device_chunks(name, 0, rank, dev, queries=True, nq=B)]).cpu().numpy()
        g, start, build_s, fit_s, truth_float = build_device_generated(cx, name, n, Q[:nq_recall])
        graph = "gpu"
    log(f"[rank {rank}] {name}: setup {time.time() - t0:.1f}s (build {build_s:.1f}s)")

    d_q = torch.from_numpy(Q).to(dev)  # the broadcast query batch, resident on every rank
    if replicated:
        from semadb_b200.sharded import ReplicatedSearcher
        searcher = ReplicatedSearcher(g, rank, world)
        searcher.exchange = "nccl"
    else:
        searcher = ShardedSearcher(g, rank, world, exchange=args.exchange)
    stream = torch.cuda.current_stream()
    # device-resident loop at N > 1: the exchange (barrier + K6) of step e runs on a side stream under the
    # search of step e+1 (ShardedSearcher pipeline, three gather buffers); SDB_NO_PIPELINE=1 = A/B
    pipelined = world > 1 and not replicated and not os.environ.get("SDB_NO_PIPELINE")
    launches = [0]
    result = [None]

    def step():
        before = g.launch_count
        result[0] = searcher.search_batch_device(d_q, K, L)  # K1 (+ fused exchange + K6 at N>1)
        # + K6 merge, + the peer barrier kernel when the exchange is fused (NCCL's kernels are not ours)
        launches[0] += g.launch_count - before + (0 if world == 1 else 2 if searcher.exchange != "nccl" else 1)

    # ---- device-resident timing; the kernel's own duration comes from events inside the same loop
    for _ in range(max(3, warmup)):
        step()
        torch.cuda.synchronize()  # the visited-table size adapts between searches that find the stream idle
    cx.barrier()
    if pipelined and searcher.exchange != "nccl" and searcher._peer is not None:
        searcher.pipeline = True
        for _ in range(3):
            step()
        searcher.wait_pipeline()
        cx.barrier()
    sampler = ClockSampler(cx.local_rank) if headline else None
    if sampler:
        sampler.start()
    launches[0] = 0
    g.search_profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    if os.environ.get("SDB_PROFILE"):  # ncu --profile-from-start off: capture the timed searches only
        torch.cuda.profiler.start()
    e0.record(stream)
    for _ in range(steps):
        step()
    if searcher.__dict__.get("pipeline"):
        searcher.wait_pipeline()  # the last steps' exchanges are part of the timed region
    e1.record(stream)
    cx.barrier()
    if os.environ.get("SDB_PROFILE"):
        torch.cuda.profiler.stop()
    if searcher.__dict__.get("pipeline"):
        searcher.pipeline = False  # the untimed tail and the e2e loop use the one-stream path
    ms_total = e0.elapsed_time(e1)
    kern = g.search_profile_read()
    g.search_profile(False)
    kern_ms = float(kern.mean()) if len(kern) else float("nan")
    n_launch = launches[0]
    m_ids, m_d, m_c = [t.clone() for t in result[0]]
    # this rank's shard-local lists (what the oracle probe and the N=1 recall compare)
    k_ids = torch.zeros((B, K), dtype=torch.int64, device=dev)
    k_d = torch.zeros((B, K), dtype=torch.float32, device=dev)
    k_c = torch.zeros((B,), dtype=torch.int32, device=dev)
    g.search_batch_device(d_q, K, L, k_ids, k_d, k_c, stream.cuda_stream)
    torch.cuda.synchronize()
    hops, ndist = g.last_search_stats(B)

    # ---- end-to-end through the C-ABI with host buffers
    h_q = torch.from_numpy(Q).pin_memory()
    h_ids = torch.zeros((B, K), dtype=torch.int64).pin_memory()
    h_d = torch.zeros((B, K), dtype=torch.float32).pin_memory()
    h_c = torch.zeros((B,), dtype=torch.int32).pin_memory()
    import ctypes as C

    def e2e_step():
        if world == 1:
            _capi.check(lib.sdb_search_batch(g._h, B, C.cast(h_q.data_ptr(), _capi.f32p), K, L, None, 0,
                                             C.cast(h_ids.data_ptr(), _capi.u64p), C.cast(h_d.data_ptr(), _capi.f32p),
                                             C.cast(h_c.data_ptr(), _capi.u32p)))
            return
        # N > 1: every rank receives the broadcast query batch in host memory (the Go cluster layer
        # fans requests out to shards, cluster/actions.go:316-351), runs the sharded search (K1 with
        # the fused peer gather, barrier, K6) and receives the merged lists. The buffers are
        # page-locked: the kernels read the queries in place (mapped host memory).
        if replicated:
            r_ids, r_d, r_c = searcher.search_batch_device(h_q.to(dev, non_blocking=True), K, L)
            h_ids.copy_(r_ids, non_blocking=True)
            h_d.copy_(r_d, non_blocking=True)
            h_c.copy_(r_c, non_blocking=True)
            torch.cuda.synchronize()
            return
        searcher.search_batch_pinned(h_q, K, L, h_ids, h_d, h_c, dev)

    for _ in range(2):
        e2e_step()
    cx.barrier()
    t1 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    cx.barrier()
    e2e_s = (time.perf_counter() - t1) / steps
    e2e_same = bool((h_ids.numpy() == m_ids.cpu().numpy()).all() and h_d.numpy().tobytes() == m_d.cpu().numpy().tobytes())

    ms_total, e2e_s, kern_ms = cx.max_over_ranks([ms_total, e2e_s, kern_ms])
    if sampler:
        # the two timed loops last ~0.1 s — two or three nvidia-smi samples. Keep the same search running
        # (untimed) for about half a second more so that the clocks / throttle reasons reported are those of a
        # GPU under this load, not of its first milliseconds (same step count on every rank).
        for _ in range(max(1, min(400, int(0.5 / max(e2e_s, 1e-4))))):
            step()
        cx.barrier()
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["window"] = "device-resident loop + e2e loop + ~0.5 s of the same search steps (untimed)"

    # ---- untimed tail: merged recall, fused-vs-NCCL parity, oracle probe
    if truth_float is not None:
        t_ids, t_d = truth_float  # exact fp32 -dot over the raw vectors (what a PQ search approximates)
    else:
        t_ids, t_d, _ = g.flat_search_batch(Q[:nq_recall], K)  # exact ground truth on the GPU (K5)
    if replicated:
        mt_ids, mt_d = t_ids.astype(np.int64), t_d
    else:
        mt_ids, mt_d = merged_truth(cx, t_ids, t_d)
    got_ids, got_d, got_c = m_ids.cpu().numpy()[:nq_recall], m_d.cpu().numpy()[:nq_recall], m_c.cpu().numpy()[:nq_recall]
    if world == 1 and not replicated:
        from semadb_b200.sharded import SHARD_SHIFT
        got_ids = got_ids + (rank << SHARD_SHIFT)
    strict, tie = recall_of(got_ids, got_d, got_c, mt_ids, mt_d)
    out = {"recall_at_10": strict, "recall_at_10_tie_aware": tie}
    if name in PQ_WORKLOADS:  # how much of the loss is the quantizer's: recall against the exhaustive ADC ranking
        a_ids, a_d, _ = g.flat_search_batch(Q[:nq_recall], K)
        ma_ids, ma_d = merged_truth(cx, a_ids, a_d)
        out["recall_at_10_vs_exhaustive_adc"], out["recall_at_10_vs_exhaustive_adc_tie_aware"] = recall_of(
            got_ids, got_d, got_c, ma_ids, ma_d)
    parity_merged = None
    if replicated:
        # every rank's concatenated lists must be what one GPU returns for the whole batch
        same = bool((k_ids == m_ids).all().item() and (k_c == m_c).all().item() and
                    k_d.cpu().numpy().tobytes() == m_d.cpu().numpy().tobytes())
        parity_merged = {"replicated_lists_equal_single_gpu_search_on_every_rank": bool(cx.min_over_ranks(1.0 if same else 0.0) == 1.0)}
    if world > 1 and not replicated and searcher.exchange != "nccl":
        # the fused exchange must give exactly what the NCCL all-gather + K6 path gives (actions.go:357-376)
        ref_s = ShardedSearcher(g, rank, world, exchange="nccl")
        n_ids, n_d, n_c = ref_s.search_batch_device(d_q, K, L)
        torch.cuda.synchronize()
        same = bool((n_ids == m_ids).all().item() and (n_c == m_c).all().item() and
                    n_d.cpu().numpy().tobytes() == m_d.cpu().numpy().tobytes())
        parity_merged = {"fused_equals_nccl_allgather_on_every_rank": bool(cx.min_over_ranks(1.0 if same else 0.0) == 1.0),
                         "e2e_lists_equal_device_lists": bool(cx.min_over_ranks(1.0 if e2e_same else 0.0) == 1.0),
                         "peer_barrier_timed_out": searcher._peer.barrier_failed() if searcher._peer is not None else None}
    parity = None
    oracle_recall = None
    if rank == 0 and not args.no_probe:
        npq = B if (name == "c2" and world == 1 and graph == "oracle") else min(args.probe_queries, B)
        try:
            parity, oix, ref = oracle_probe(cx, name, g, start, n, Q[:npq], k_ids.cpu().numpy(), k_d.cpu().numpy(), oix)
            if name in PQ_WORKLOADS and world == 1:
                nn = min(npq, nq_recall)
                oracle_recall = recall_of(ref["ids"][:nn].astype(np.int64), ref["dists"][:nn], ref["counts"][:nn],
                                          mt_ids[:nn], mt_d[:nn])[0]
        except MemoryError as e:  # noqa: PERF203
            parity = {"skipped": f"host memory: {e}"}
    # K7 beside the oracle: productQuantizer.Fit on the same first 10 000 points (product.go:175-236,
    # kmeans.go:34-150) on the host cores, and the centroids / centroidDists it yields
    fit_cpu = None
    if name in PQ_WORKLOADS and rank == 0 and not args.no_probe:
        from oracle import oraclelib as O
        _, x0 = next(iter(device_chunks(name, n, rank, dev)))
        x0 = x0[:10000].cpu().numpy()
        of = O.OracleIndex(w["dim"], w["metric"], L, R, ALPHA, quantizer="product", pq_m=96, pq_k=256, pq_trigger=10000)
        of.set_start(start)
        of.set_vectors(np.arange(2, 2 + len(x0), dtype=np.uint32), x0)
        t = time.time()
        of.fit(0, True, O.hw_threads())
        fit_cpu_s = time.time() - t
        ofc, ocd = of.get_pq()
        gfc, gcd = g.get_pq()
        fit_cpu = {"oracle_fit_s": fit_cpu_s, "oracle_threads": O.hw_threads(), "gpu_fit_s": fit_s,
                   "centroids_bit_identical": bool(ofc.tobytes() == gfc.tobytes()),
                   "centroid_dists_bit_identical": bool(ocd.tobytes() == gcd.tobytes())}
        del of
    cx.barrier()

    ms_step = ms_total / steps
    bytes_q = float(ndist.mean()) * w["row_bytes"] + float(hops.mean()) * R * 4
    launch_queries = -(-B // world) if replicated else B  # queries one launch of the kernel processes
    achieved = bytes_q * launch_queries / (kern_ms * 1e-3) / 1e9
    peak, peak_kind = measured_peaks()
    out.update({
        "name": name, "g": g, "oix": oix, "X": X, "Q": Q, "start": start, "graph": graph,
        "ms_step": ms_step, "value": (1 if replicated else world) * B / (ms_step * 1e-3), "user_qps": B / (ms_step * 1e-3),
        "kern_ms": kern_ms, "e2e_s": e2e_s, "e2e_value": (1 if replicated else world) * B / e2e_s, "n_launch": n_launch,
        "mean_hops": float(hops.mean()), "mean_ndist": float(ndist.mean()), "bytes_q": bytes_q,
        "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "clocks": clocks, "build_s": build_s, "fit_s": fit_s,
        "parity": parity, "parity_merged": parity_merged, "oracle_recall": oracle_recall, "k_ids": k_ids, "k_d": k_d,
        "pq_fit": fit_cpu,
        "exchange": searcher.exchange, "searcher": searcher, "launch_queries": launch_queries, "pipelined": pipelined,
        "outputs": {"ids": m_ids.cpu().numpy().astype(np.float64), "dists": m_d.cpu().numpy().astype(np.float32),
                    "counts": m_c.cpu().numpy().astype(np.float32)} if headline else None,
    })
    return out


def extra_block(r, world, B):
    """The JSON form of a non-headline workload."""
    w = WORKLOADS[r["name"]]
    d = {"workload": w["desc"].format(n=r["n"]) + f", {B}-query batch, k={K}, GPU-built graph (K8)",
         "shard_searches_per_s": r["value"], "user_qps": r["user_qps"], "ms_per_step": r["ms_step"],
         "e2e_shard_searches_per_s": r["e2e_value"], "recall_at_10_merged": r["recall_at_10"],
         "recall_at_10_merged_tie_aware": r["recall_at_10_tie_aware"] if w["integer"] or r["name"] == "c3" else None,
         "mean_hops": r["mean_hops"],
         "mean_ndist": r["mean_ndist"], "bytes_per_query": r["bytes_q"],
         "roofline": {"bound": "hbm", "achieved": r["achieved"], "peak": r["peak"], "unit": "GB/s",
                      "frac": r["achieved"] / r["peak"], "kernel_ms": r["kern_ms"], "per": "GPU"},
         "build_s_per_gpu": r["build_s"], "parity": r["parity"], "parity_merged": r["parity_merged"], "n_gpus": world}
    if d["roofline"]["frac"] > 1.0:
        d["roofline"]["note"] = ("algorithmic bytes count every gathered row; the first hops and hub rows are L2 hits, so DRAM "
                                 "traffic is lower than that and the fraction of the measured copy peak can exceed 1")
    if w["integer"]:
        d["recall_note"] = "integer distances: tie-aware recall counts a result as a hit when its distance <= the k-th true distance"
    for k_ in ("recall_at_10_vs_exhaustive_adc", "recall_at_10_vs_exhaustive_adc_tie_aware", "oracle_recall", "fit_s", "pq_fit"):
        if r.get(k_) is not None:
            d[k_] = r[k_]
    return d


def run_flat(cx, g, Q, n, reps=7):
    """K5: IndexFlat.Search of the whole query batch over the headline shard through
    sdb_flat_search_batch with page-locked host buffers (copies inside the timed calls); the
    first 2000 lists are compared with the exact CUDA-core scan's."""
    import ctypes as C
    torch = cx.torch
    from semadb_b200 import _capi
    lib = _capi.lib()
    B, dim = Q.shape
    h_q = torch.from_numpy(Q).pin_memory()
    h_ids = torch.zeros((B, K), dtype=torch.int64).pin_memory()
    h_d = torch.zeros((B, K), dtype=torch.float32).pin_memory()
    h_c = torch.zeros((B,), dtype=torch.int32).pin_memory()

    def call(nq=B):
        _capi.check(lib.sdb_flat_search_batch(g._h, nq, C.cast(h_q.data_ptr(), _capi.f32p), K, None, 0,
                                              C.cast(h_ids.data_ptr(), _capi.u64p), C.cast(h_d.data_ptr(), _capi.f32p),
                                              C.cast(h_c.data_ptr(), _capi.u32p)))

    for _ in range(2):
        call()
    times = []
    for _ in range(reps):
        t = time.perf_counter()
        call()
        times.append(time.perf_counter() - t)
    path, cand, ovf = g.flat_last_stats()
    tc_ids, tc_d = h_ids.numpy().copy(), h_d.numpy().copy()
    nx = min(B, 2000)
    os.environ["SDB_FLAT_EXACT"] = "1"
    try:
        call(nx)
    finally:
        os.environ.pop("SDB_FLAT_EXACT", None)
    same = bool((tc_ids[:nx] == h_ids.numpy()[:nx]).all() and tc_d[:nx].tobytes() == h_d.numpy()[:nx].tobytes())
    dt = float(np.median(times))
    peak_tf = None
    try:
        peak_tf = float(json.loads((ROOT / "MEASURED_PEAKS.json").read_text())["bf16_tflops"])
    except Exception:
        pass
    tf = 2.0 * B * n * dim / dt / 1e12
    return {"workload": f"IndexFlat.Search (K5): {B} queries x {n} x {dim} f32, k={K}, through sdb_flat_search_batch with "
                        f"page-locked host buffers (tcgen05 sample pass + candidate pass + exact re-score)",
            "ms_per_batch": dt * 1e3, "ms_each": [round(x * 1e3, 3) for x in times], "queries_per_s": B / dt,
            "path": {0: "exact CUDA-core scan", 1: "mma.sync candidate pass", 2: "tcgen05 candidate pass"}.get(path, path),
            "candidates_per_query": cand / B, "fell_back_to_exact_scan": ovf,
            "lists_identical_to_exact_scan": {"queries": nx, "identical": same},
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (tf / peak_tf) if peak_tf else None,
                         "note": "useful FLOP (2 x queries x points x dim) / whole call incl. copies, sample pass and re-score"}}


def run_build(cx, n, steps, warmup, stat="mean", outputs=False):
    """C5a: batched graph build (K8) of one n x 128 shard per GPU from empty; points/s over all GPUs.
    stat: how the timed builds are summarised — "mean" (the headline contract) or "median" (the
    extra block: one build in a few runs long on some hosts, DESIGN.md K8; every time is listed).
    outputs: also return the graph of the last timed build (degree and edge list of nodes 1..n+1,
    unused slots -1)."""
    torch = cx.torch
    from semadb_b200 import synth
    X = synth.sift_shaped(n, 128, seed=3 + 1000 * cx.rank, w_seed=3)
    d_x = torch.from_numpy(X).to(cx.dev)
    ids = np.arange(2, n + 2, dtype=np.uint64)
    times, stats, g = [], None, None
    for it in range(warmup + steps):
        if g is not None:
            g.close()
        g, _ = new_index("c2", cx.rank, cx.local_rank)
        g.reserve(n + 2)
        if os.environ.get("SDB_INSERT_CONFIG"):  # "min,max,growth_div": A/B of the mini-batch schedule
            g.insert_config(*[int(x) for x in os.environ["SDB_INSERT_CONFIG"].split(",")])
        cx.barrier()
        t = time.perf_counter()
        g.insert_batch_device(ids, d_x)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t
        dt = cx.max_over_ranks([dt])[0]
        if it >= warmup:
            times.append(dt)
            stats = g.insert_stats()
    dt = float(np.median(times)) if stat == "median" else float(np.mean(times))
    graph = None
    if outputs:
        keep = dump_rows(n + 1, 4 + R * 8)
        rows = np.arange(n + 1) if keep is None else keep
        deg, edges = g.get_edges((rows + 1).astype(np.uint64))
        edges = np.where(np.arange(R)[None, :] < deg[:, None], edges.astype(np.float64), -1.0)
        graph = {"degree": deg.astype(np.float32), "edges": edges}
        if keep is not None:
            graph["rows"] = keep.astype(np.float64)
    # algorithmic bytes of the build (DESIGN.md K8): the searches' gathers, the candidate rows of
    # robustPrune(new), the adjacency rows of the back-edge targets (read + write) and the
    # candidate rows of robustPrune(B) on saturated targets
    row = 512
    by = (stats["ndist"] * row + stats["hops"] * R * 4 + stats["hops"] * row + stats["points"] * R * 4 +
          stats["targets"] * 2 * R * 4 + stats["prune_candidates"] * row)
    peak, peak_kind = measured_peaks()
    Q = synth.sift_shaped(2000, 128, seed=4, w_seed=3)
    ids_, d_, c_ = g.search_batch(Q, K, L)
    fi, fd, _ = g.flat_search_batch(Q, K)
    rec = float(np.mean([len(set(ids_[b].tolist()) & set(fi[b].tolist())) / K for b in range(len(Q))]))
    g.close()
    res = {"workload": f"C5a: batched graph build from empty, {n}x128 f32 L2 per GPU (greedySearch + robustPrune + "
                       f"back-edges, K8), vectors resident in HBM",
           "points_per_s": cx.world * n / dt, "build_s": dt, "build_s_is": stat + f" of {len(times)} builds",
           "builds_timed": len(times), "build_s_each": [round(t, 4) for t in times],
           "n_gpus": cx.world,
           "recall_at_10_of_built_graph": rec, "insert_stats": stats,
           "roofline": {"bound": "hbm", "achieved": by / dt / 1e9, "peak": peak, "unit": "GB/s", "frac": by / dt / 1e9 / peak,
                        "algorithmic_bytes_per_point": by / max(1, stats["points"]), "per": "GPU"}}
    if graph is not None:
        res["outputs"] = graph
    return res


def main():
    global _OUT
    _OUT = _quarantine_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4", "c4cos", "c5b", "c5a"])
    ap.add_argument("--extra", default="auto", help="auto | none | comma list of c3,c4,c5b,c5a")
    ap.add_argument("--mode", default="sharded", choices=["sharded", "replicated"],
                    help="sharded: one shard per GPU, every query visits every shard (weak scaling, the reference's "
                         "cluster semantics); replicated: the whole index on every GPU, the batch split N ways (strong scaling)")
    ap.add_argument("--points", "--n", dest="n", type=int, default=0,
                    help="points per GPU shard of the headline workload (0 = the config's)")
    ap.add_argument("--extra-n", default="", help="name=points,... overrides for the extra workloads (tests)")
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--ref-queries", type=int, default=10_000)
    ap.add_argument("--graph", default="oracle", choices=["auto", "oracle", "gpu"])
    ap.add_argument("--exchange", default=os.environ.get("SDB_EXCHANGE", "auto"), choices=["auto", "p2p", "nccl"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-probe", action="store_true")
    ap.add_argument("--recall-queries", type=int, default=2000)
    ap.add_argument("--probe-queries", type=int, default=1000)
    ap.add_argument("--extra-budget-s", type=float, default=560.0,
                    help="no further extra workload is started once this much wall time has passed")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline's last timed step returned as DIR/<name>.npy (float32/float64, < 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if args.graph == "auto":
        args.graph = "oracle"

    cx = Ctx(args)
    torch = cx.torch
    rank, world = cx.rank, cx.world
    B = args.queries

    if args.workload == "c5a":
        n = args.n or 1_000_000
        r = run_build(cx, n, args.steps, min(args.warmup, 1), outputs=args.dump_outputs is not None)
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, r["outputs"])
        if rank == 0:
            out = {"metric": "vamana_build_points_per_s", "value": r["points_per_s"], "unit": "points/s", "n_gpus": world,
                   "steps": r["builds_timed"], "warmup": min(args.warmup, 1), "ms_per_step": r["build_s"] * 1e3,
                   "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                   "data": "synthetic", "config": {"workload": r["workload"], "points_per_gpu": n,
                                                   "recall_at_10_of_built_graph": r["recall_at_10_of_built_graph"],
                                                   "build_s_each": r["build_s_each"], "insert_stats": r["insert_stats"]},
                   "roofline": r["roofline"], "cpu_baseline": None, "e2e": None, "gpu_launches": None}
            print(json.dumps(out), file=_OUT, flush=True)
        if world > 1:
            cx.dist.destroy_process_group()
        return

    name = args.workload
    if args.mode == "replicated":
        if name != "c2":
            raise SystemExit("--mode replicated is measured on c2")
        # every replica must hold the same graph: the batched GPU build is deterministic, the oracle's
        # concurrent workers are not
        args.graph = "gpu"
        if args.extra == "auto":
            args.extra = "none"
    n = args.n or WORKLOADS[name]["n"]
    h = run_search(cx, name, n, B, args.steps, max(3, args.warmup), args.graph, headline=True)
    h["n"] = n
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, h["outputs"])

    # ---- cpu baseline (untimed, rank 0, N = 1, C2)
    cpu = None
    if rank == 0 and name == "c2" and world == 1 and not args.no_cpu_baseline:
        from oracle import oraclelib as O
        threads = O.hw_threads()
        oix = h["oix"]
        if oix is None:
            oix, _, _ = build_oracle_index(h["X"], h["start"], threads)
        Q = h["Q"]
        oix.search(Q[:1000], k=K, search_size=L, threads=threads)
        t0 = time.time()
        reps = 0
        while reps < 3 or (time.time() - t0 < 5.0 and reps < 50):
            oix.search(Q, k=K, search_size=L, threads=threads)
            reps += 1
        cdt = (time.time() - t0) / reps
        t1 = time.time()
        oix.search(Q[:2000], k=K, search_size=L, threads=1)
        qps1 = 2000 / (time.time() - t1)
        cpu = {"value": B / cdt, "unit": "queries/s", "cores": threads, "kind": "port",
               "sample": f"all {B} queries x {reps} passes, {threads} threads, one query per thread",
               "single_thread_qps": qps1}
    # ---- K5 on the same shard (rank-local, N = 1): IndexFlat.Search of the whole batch
    flat = None
    if name == "c2" and world == 1 and args.extra != "none" and h.get("g") is not None:
        try:
            flat = run_flat(cx, h["g"], h["Q"], n)
        except Exception as e:  # noqa: BLE001 — an extra block must never cost the headline line
            import traceback
            traceback.print_exc(file=sys.stderr)
            flat = {"error": repr(e)[:300]}
    # release the headline index before the extra workloads need the memory
    for k_ in ("g", "oix", "X", "searcher", "k_ids", "k_d"):
        h[k_] = None
    import gc
    gc.collect()
    torch.cuda.empty_cache()

    # ---- extra workloads
    extra_names = []
    if args.extra == "auto":
        extra_names = ["c5a"] + (["c3", "c5b"] if world == 8 else [])
    elif args.extra != "none":
        extra_names = [x for x in args.extra.split(",") if x]
    extra_n = dict((kv.split("=")[0], int(kv.split("=")[1])) for kv in args.extra_n.split(",") if kv)
    extras = {}
    if flat is not None:
        extras["flat"] = flat
    for en in extra_names:
        if en == name:
            continue
        # every rank takes the same decision (rank 0's clock)
        elapsed = time.time() - _T0
        if world > 1:
            t = torch.tensor([elapsed], dtype=torch.float64, device=cx.dev)
            cx.dist.broadcast(t, 0)
            elapsed = float(t.item())
        if elapsed > args.extra_budget_s:
            extras[en] = {"skipped": f"{elapsed:.0f}s of wall time already used (budget {args.extra_budget_s:.0f}s)"}
            continue
        try:
            if en == "c5a":
                extras[en] = run_build(cx, extra_n.get(en, 1_000_000), 3, 1, stat="median")
            else:
                en_n = extra_n.get(en, WORKLOADS[en]["n"])
                r = run_search(cx, en, en_n, B, max(5, args.steps // 2), 3, "gpu", headline=False)
                r["n"] = en_n
                extras[en] = extra_block(r, world, B)
                for k_ in ("g", "oix", "X", "searcher", "k_ids", "k_d"):
                    r[k_] = None
                del r
        except Exception as e:  # noqa: BLE001 — an extra block must never cost the headline line
            import traceback
            traceback.print_exc(file=sys.stderr)
            extras[en] = {"error": repr(e)[:300]}
            if world > 1:
                break  # ranks may be out of step after a failure: stop here
        gc.collect()
        torch.cuda.empty_cache()
        log(f"[rank {rank}] extra {en} done")

    if rank == 0:
        w = WORKLOADS[name]
        cfg = workload_config(name, n, B, world, h["graph"])
        if args.mode == "replicated":
            cfg.update(parallelism=f"replicated x{world}: the whole {n}-point index on every GPU, the batch split {world} ways, "
                                   f"slices concatenated by one NCCL all-gather per result tensor",
                       parity_merged=h["parity_merged"])
        elif world > 1:
            cfg.update(exchange="fused peer stores over NVLink + flag barrier (sdb_search_batch_gather_device)"
                       if h["exchange"] != "nccl" else "NCCL all-gather per result tensor",
                       exchange_pipelining=("barrier + merge of step e on a side stream under the search of step e+1 "
                                            "(three gather buffers); value is steady-state throughput, e2e is one "
                                            "synchronous call per step") if h["pipelined"] and h["exchange"] != "nccl" else "none",
                       parity_merged=h["parity_merged"])
        cfg.update(user_qps=h["user_qps"], recall_at_10=h["recall_at_10"],
                   recall_scope=("merged top-k of all shards vs exact top-k of the union"
                                 if world > 1 and args.mode != "replicated" else "single shard vs exact flat scan"),
                   mean_hops=h["mean_hops"], mean_ndist=h["mean_ndist"], bytes_per_query=h["bytes_q"],
                   parity=h["parity"], host_cores=os.cpu_count(), setup_build_s=h["build_s"])
        if w["integer"]:
            cfg["recall_at_10_tie_aware"] = h["recall_at_10_tie_aware"]
        for k_ in ("recall_at_10_vs_exhaustive_adc", "oracle_recall", "fit_s", "pq_fit"):
            if h.get(k_) is not None:
                cfg[k_] = h[k_]
        out = {
            "metric": "vamana_search_qps", "value": h["value"], "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": h["ms_step"], "higher_is_better": True,
            "scaling": "strong" if args.mode == "replicated" else "weak", "vs_baseline": None,
            "dtype": "u64" if w["integer"] else "f32",
            "data": "synthetic" if name == "c2" else "synthetic (device-generated)", "config": cfg,
            "roofline": {"bound": "hbm", "achieved": h["achieved"], "peak": h["peak"], "unit": "GB/s",
                         "frac": h["achieved"] / h["peak"],
                         "traffic": measured_traffic() if (name == "c2" and n == 1_000_000 and B == 10_000) else None,
                         "algorithmic_bytes_per_launch": h["bytes_q"] * h["launch_queries"], "peak_kind": h["peak_kind"],
                         "kernel": "beam_search_kernel", "kernel_ms": h["kern_ms"],
                         "kernel_ms_how": "CUDA events around the kernel inside the timed loop, mean over its steps, max over ranks"},
            "cpu_baseline": cpu,
            "e2e": {"value": h["e2e_value"], "unit": "queries/s", "h2d_bytes_per_step": B * w["dim"] * 4,
                    "d2h_bytes_per_step": B * K * 12 + B * 4, "ms_per_step": h["e2e_s"] * 1e3},
            "gpu_launches": h["n_launch"],
            "clocks": h["clocks"],
            "extra_configs": extras,
            "wall_s": round(time.time() - _T0, 1),
        }
        print(json.dumps(out), file=_OUT, flush=True)
    if world > 1:
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
