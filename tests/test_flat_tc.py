"""K5 on tensor cores (csrc/flat_tc.cu): bf16 GEMM candidate pass + exact re-score must return
exactly what the exact CUDA-core scan (csrc/flat.cu) and the oracle's brute force return —
ids and distances bit for bit, ties by ascending id (flat.go:99,117 with ascending-id order)."""
import os

import numpy as np
import pytest

from semadb_b200 import synth
from semadb_b200.vamana import IndexFlat, IndexVectorFlatParameters

pytestmark = pytest.mark.gpu


def _both(g, Q, k):
    os.environ.pop("SDB_FLAT_EXACT", None)
    a = g.flat_search_batch(Q, k)
    os.environ["SDB_FLAT_EXACT"] = "1"
    try:
        b = g.flat_search_batch(Q, k)
    finally:
        os.environ.pop("SDB_FLAT_EXACT", None)
    return a, b


@pytest.mark.parametrize("metric,dim,kind", [("euclidean", 128, "sift"), ("euclidean", 100, "gauss"), ("dot", 96, "gauss"),
                                             ("cosine", 384, "unit"), ("euclidean", 2, "uniform")])
def test_flat_tc_equals_exact_scan(metric, dim, kind):
    n = 70_000  # above the tensor-core path's threshold (4 x 16384 sample points)
    if kind == "sift":
        X, Q = synth.sift_shaped(n, dim, 3), synth.sift_shaped(300, dim, 4, w_seed=3)
    elif kind == "uniform":
        X, Q = synth.uniform(n, dim, 1), synth.uniform(300, dim, 2)
    else:
        X = synth.latent_gaussian(n, dim, seed=dim, latent=8, normalize=(kind == "unit"))
        Q = synth.latent_gaussian(300, dim, seed=dim + 1, w_seed=dim, latent=8, normalize=(kind == "unit"))
    X[5000:5100] = X[:100]  # exact duplicates: ties must resolve by ascending id
    g = IndexFlat(IndexVectorFlatParameters(dim, metric))
    ids = np.arange(2, n + 2, dtype=np.uint64)
    g.set_vectors(ids, X)
    for k in (10, 1, 75):
        (ti, td, tc), (ei, ed, ec) = _both(g, Q, k)
        assert (tc == ec).all() and (ti == ei).all()
        assert td.tobytes() == ed.tobytes()
    # queries that are stored points: distance 0 (L2) and the duplicate with the lower id first
    (ti, td, tc), (ei, ed, ec) = _both(g, X[:100], 10)
    assert (ti == ei).all() and td.tobytes() == ed.tobytes()
    if metric == "euclidean":
        assert (ti[:, 0] == ids[:100]).all() and (ti[:, 1] == ids[5000:5100]).all() and (td[:, :2] == 0).all()
    # deleted rows never come back
    g.delete_rows(ids[:50])
    (ti, td, tc), (ei, ed, ec) = _both(g, X[:100], 10)
    assert (ti == ei).all() and td.tobytes() == ed.tobytes() and not np.isin(ti, ids[:50]).any()


def test_flat_tc_matches_oracle():
    from oracle import oraclelib as O
    n, dim = 70_000, 64
    X = synth.latent_gaussian(n, dim, seed=9, latent=8)
    Q = synth.latent_gaussian(100, dim, seed=10, w_seed=9, latent=8)
    oix = O.OracleIndex(dim, "euclidean")
    ids = np.arange(2, n + 2, dtype=np.uint32)
    oix.set_vectors(ids, X)
    gt = oix.flat_search(Q, k=10, threads=8)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(ids.astype(np.uint64), X)
    fi, fd, fc = g.flat_search_batch(Q, 10)
    assert (fi == gt["ids"].astype(np.uint64)).all() and fd.tobytes() == gt["dists"].tobytes()


@pytest.mark.parametrize("metric,dim", [("euclidean", 128), ("dot", 96), ("euclidean", 200), ("cosine", 384)])
def test_tcgen05_candidate_pass_matches_mma_sync_pass(metric, dim):
    """The tcgen05 + TMA candidate pass (default for dim <= 512) and the mma.sync pass compute the
    same bf16 GEMM: the candidate sets they keep must have (almost) the same size — only the fp32
    accumulation order differs — nobody may fall back to the exact scan, and the results are
    bit-identical. A wrong descriptor / swizzle would either flood the candidate lists (overflow
    -> exact scan) or starve them (wrong results); both are caught here."""
    n = 70_000
    X = synth.latent_gaussian(n, dim, seed=dim, latent=8, normalize=(metric == "cosine"))
    Q = synth.latent_gaussian(500, dim, seed=dim + 1, w_seed=dim, latent=8, normalize=(metric == "cosine"))
    g = IndexFlat(IndexVectorFlatParameters(dim, metric))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    os.environ.pop("SDB_FLAT_MMA_SYNC", None)
    d = g.flat_search_batch(Q, 10)  # the default: two-pass form of the tcgen05 path
    pd, cd, od = g.flat_last_stats()
    os.environ["SDB_FLAT_LEVELS"] = "1"  # the level scheme on both kernels: same algorithm, same candidate sets
    try:
        a = g.flat_search_batch(Q, 10)
        pa, ca, oa = g.flat_last_stats()
        os.environ["SDB_FLAT_MMA_SYNC"] = "1"
        b = g.flat_search_batch(Q, 10)
        pb, cb, ob = g.flat_last_stats()
    finally:
        os.environ.pop("SDB_FLAT_MMA_SYNC", None)
        os.environ.pop("SDB_FLAT_LEVELS", None)
    assert pa == 2 and pb == 1 and pd == 2
    assert oa == 0 and ob == 0 and od == 0
    assert ca >= 10 * len(Q) and abs(ca - cb) <= 0.01 * cb + 5
    assert cd >= 10 * len(Q)
    assert (a[0] == b[0]).all() and a[1].tobytes() == b[1].tobytes()
    assert (d[0] == b[0]).all() and d[1].tobytes() == b[1].tobytes()


@pytest.mark.parametrize("variant", ["levels", "sample_all", "sample_small"])
def test_flat_tc_variants_equal_exact_scan(variant, monkeypatch):
    """Every form of the candidate generation returns the exact scan's lists: the level scheme
    (SDB_FLAT_LEVELS=1), the two-pass form with the whole store as the sample and with a sample so
    small that the bound is loose."""
    env = {"levels": ("SDB_FLAT_LEVELS", "1"), "sample_all": ("SDB_FLAT_SAMPLE_DIV", "1"),
           "sample_small": ("SDB_FLAT_SAMPLE_DIV", "64")}[variant]
    n, dim = 70_000, 128
    X, Q = synth.sift_shaped(n, dim, 3), synth.sift_shaped(400, dim, 4, w_seed=3)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    monkeypatch.setenv(*env)
    for k in (10, 75):
        ti, td, tc = g.flat_search_batch(Q, k)
        path, cand, ovf = g.flat_last_stats()
        assert path == 2 and ovf == 0 and cand >= k * len(Q)
        monkeypatch.setenv("SDB_FLAT_EXACT", "1")
        ei, ed, ec = g.flat_search_batch(Q, k)
        monkeypatch.delenv("SDB_FLAT_EXACT")
        assert (tc == ec).all() and (ti == ei).all() and td.tobytes() == ed.tobytes()


def test_flat_tc_clustered_insertion_order():
    """Points stored in an order that follows their position (sorted along one coordinate, as a
    collection filled region by region would be): the sample of the minimum-mode pass is spread
    over the whole id range, so the bound stays useful — nobody overflows into the exact scan —
    and the lists are the exact scan's."""
    n, dim = 80_000, 64
    X = synth.latent_gaussian(n, dim, seed=21, latent=8)
    X = np.ascontiguousarray(X[np.argsort(X[:, 0], kind="stable")])
    Q = synth.latent_gaussian(300, dim, seed=22, w_seed=21, latent=8)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    a = g.flat_search_batch(Q, 10)
    path, cand, ovf = g.flat_last_stats()
    assert path == 2 and ovf == 0 and cand < 2000 * len(Q)
    os.environ["SDB_FLAT_EXACT"] = "1"
    try:
        b = g.flat_search_batch(Q, 10)
    finally:
        os.environ.pop("SDB_FLAT_EXACT", None)
    assert (a[0] == b[0]).all() and a[1].tobytes() == b[1].tobytes()


def test_flat_tc_overflow_falls_back_to_exact_scan():
    """10 000 near-copies of each of seven vectors: every query has thousands of points within the
    bf16 error bound of its k-th distance, the candidate lists overflow (cap 4 096) and those
    queries are answered by the exact scan — same lists, through the host-buffer call."""
    n, dim = 70_000, 96
    rng = np.random.default_rng(11)
    base = rng.normal(size=(7, dim)).astype(np.float32)
    X = (base[np.arange(n) % 7] + rng.normal(size=(n, dim)).astype(np.float32) * np.float32(1e-4)).astype(np.float32)
    Q = (base[rng.integers(0, 7, 200)] + rng.normal(size=(200, dim)).astype(np.float32) * np.float32(1e-3)).astype(np.float32)
    g = IndexFlat(IndexVectorFlatParameters(dim, "euclidean"))
    g.set_vectors(np.arange(2, n + 2, dtype=np.uint64), X)
    a = g.flat_search_batch(Q, 10)
    path, cand, ovf = g.flat_last_stats()
    assert path == 2 and ovf > 0
    os.environ["SDB_FLAT_EXACT"] = "1"
    try:
        b = g.flat_search_batch(Q, 10)
    finally:
        os.environ.pop("SDB_FLAT_EXACT", None)
    assert (a[2] == b[2]).all() and (a[0] == b[0]).all() and a[1].tobytes() == b[1].tobytes()
