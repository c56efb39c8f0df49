"""Shared helpers for parity tests: build a graph with the oracle, mirror it onto the GPU, compare
searches and graphs with the oracle's, and bound f32 distances against a float64 reference."""
from __future__ import annotations

import numpy as np

from oracle import oraclelib as O
from semadb_b200 import synth
from semadb_b200.vamana import IndexVamana, IndexVectorVamanaParameters, Quantizer


def oracle_graph(X, metric="euclidean", L=75, R=64, alpha=1.2, start_seed=99, threads=8, **okw):
    """Oracle index with ids 2..n+1 inserted (sequential if threads == 1)."""
    n, dim = X.shape
    ix = O.OracleIndex(dim, metric, L, R, alpha, **okw)
    start = synth.start_vector(dim, start_seed)
    ix.set_start(start)
    ids = np.arange(2, n + 2, dtype=np.uint32)
    ix.insert(ids, X, threads=threads)
    return ix, ids, start


def mirror_to_gpu(oix, X, ids, start, metric="euclidean", L=75, R=64, alpha=1.2, quantizer=None, relaxed=False):
    """GPU IndexVamana holding the same vectors and the oracle-built edges."""
    params = IndexVectorVamanaParameters(X.shape[1], metric, L, R, alpha, quantizer)
    g = IndexVamana("parity", params, start_vector=start, relaxed=relaxed)
    g.set_vectors(ids.astype(np.uint64), X)
    adj, deg = oix.get_graph()
    g.set_graph_dense(adj[1:], deg[1:], first_id=1)
    return g


def recall_at_k(ids, gt_ids):
    B, k = gt_ids.shape
    return float(np.mean([len(set(ids[b].tolist()) & set(gt_ids[b].tolist())) / k for b in range(B)]))


def check_search(oix, g, Q, k=10, L=75):
    """GPU beam search equal to the oracle's: counts, ids, distance bytes, hops and evaluations."""
    ref = oix.search(Q, k=k, search_size=L, threads=8, diagnostics=True)
    ids, d, cnt = g.search_batch(Q, k, L)
    hops, nd = g.last_search_stats(len(Q))
    assert (cnt == ref["counts"]).all()
    assert (ids == ref["ids"].astype(np.uint64)).all()
    assert d.tobytes() == ref["dists"].tobytes()
    assert (hops == ref["hops"]).all()
    assert (nd == ref["ndist"]).all()
    return ref


def check_graph_equal(oix, g, n):
    """GPU graph over nodes 1..n+1 equal to the oracle's edge for edge, in order."""
    adj, odeg = oix.get_graph()
    deg, e = g.get_edges(np.arange(1, n + 2, dtype=np.uint64))
    assert (deg == odeg[1:n + 2]).all()
    for r in range(n + 1):
        assert e[r, :deg[r]].tolist() == adj[r + 1, :odeg[r + 1]].tolist(), f"node {r + 1}"


def f64_dists(metric, X, Y):
    """float64 distances between the rows of X and the rows of Y ([len(X)][len(Y)]) and, for each,
    a bound on how far an f32 evaluation of it may lie: |fl(d) - d| <= gamma_n * sum|terms|,
    gamma_n = n u / (1 - n u), u = 2^-24 (Higham, Accuracy and Stability of Numerical Algorithms,
    §3.1), whatever the summation order. n counts the roundings a term goes through on its way into
    the result: dim for the sum, one for the metric's epilogue (1 - dot) and, for squared L2, two
    more: the rounded difference x - y enters its own square. The float64 evaluation's own error
    (squared L2 here is |x|^2 + |y|^2 - 2 x.y) is added to the bound."""
    X = np.asarray(X, np.float64)
    Y = np.asarray(Y, np.float64)
    dim = X.shape[1]
    n = dim + (3 if metric == "euclidean" else 1)
    gamma = n * 2.0 ** -24 / (1 - n * 2.0 ** -24)
    gamma64 = (dim + 2) * 2.0 ** -53 / (1 - (dim + 2) * 2.0 ** -53)
    dot = X @ Y.T
    if metric == "euclidean":
        nx, ny = (X * X).sum(1)[:, None], (Y * Y).sum(1)[None, :]
        d = np.maximum(nx + ny - 2.0 * dot, 0.0)
        return d, gamma * d + 4 * gamma64 * (nx + ny)
    mag = np.abs(X) @ np.abs(Y).T
    if metric == "dot":
        return -dot, (gamma + gamma64) * mag
    if metric == "cosine":
        return 1.0 - dot, (gamma + gamma64) * (1.0 + mag)
    raise ValueError(metric)
