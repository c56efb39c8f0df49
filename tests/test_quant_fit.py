"""K7/K9: the quantizer fit (VectorStore.Fit) and the encoders that run after it, on every
kernel path of `fit_locked` (quant.cu) and on degenerate training data.

Each PQ case fits an oracle index and a GPU index holding the same rows (ids with gaps, a few
deleted before the fit) from the same first row, then requires, bit for bit: flatCentroids,
centroidDists, the codes of every stored row, the rows the k-means wrote through
(kmeans.go:144), ADC tables, and the codes of rows set after the fit (pq_encode_kernel) --
among them rows equal to a centroid and rows at the same distance from two centroids.
Because the oracle computes in f32 in the same order, a mistake the two share would pass that
comparison; the float64 checks below do not trust the oracle: centroidDists and ADC tables lie
within the gamma_n bound of tests/helpers.f64_dists, every code is a float64 argmin up to that
bound, and the BQ threshold lies within the summation bound of the float64 column mean."""
from __future__ import annotations

from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import oraclelib as O
from semadb_b200 import synth
from semadb_b200._capi import ERR_INVALID, ERR_STATE, SdbError
from semadb_b200.vamana import (BinaryQuantizerParameters, IndexVamana, IndexVectorVamanaParameters,
                                ProductQuantizerParameters, Quantizer)
from tests.helpers import f64_dists

FLT_MAX = float(np.finfo(np.float32).max)
U32 = 2.0 ** -24

# ---------------------------------------------------------------- kernel selection of fit_locked
KM_TILE = 256  # rows per assign CTA
KM_MAX_TILES = 64  # the assign grid is capped at 64 row tiles: beyond 64 * 256 rows its loop strides
KM_STAGE_BYTES = 96 * 1024  # the K centres of a sub-space are staged in shared memory up to this size
MAX_ITER = 100  # product.go:209


def assign_path(dim, M, K, rows):
    """(km_assign_kernel template argument, centres staged in shared memory, row loop strides)."""
    sub = dim // M
    return (sub if sub in (4, 8, 16) else 0, K * sub * 4 <= KM_STAGE_BYTES, rows > KM_TILE * KM_MAX_TILES)


def reachable_paths():
    """Every combination that some (dim, M, K <= 256, rows) selects: a register form holds at most
    16 floats per centre, so its centres always fit shared memory."""
    out = set()
    for form in (4, 8, 16, 0):
        for staged in (True, False):
            if form and not staged:
                continue
            for strided in (False, True):
                out.add((form, staged, strided))
    return out


# ---------------------------------------------------------------- data
def _rows(kind, n, dim, seed, metric):
    rng = np.random.Generator(np.random.PCG64(seed))
    if kind == "gauss":
        X = synth.latent_gaussian(n, dim, seed=seed, latent=8)
    elif kind == "clusters":  # 200 tight clusters: k-means settles in a few rounds even at n = 20 000
        C = rng.normal(size=(200, dim)).astype(np.float32) * np.float32(4)
        X = C[rng.integers(0, 200, n)] + rng.normal(size=(n, dim)).astype(np.float32) * np.float32(0.05)
    elif kind == "dup40":  # 40 distinct rows repeated: fewer distinct sub-vectors than K everywhere
        X = synth.latent_gaussian(40, dim, seed=seed, latent=8)[rng.integers(0, 40, n)]
    elif kind == "const_sub":  # one sub-space constant across the rows
        X = synth.latent_gaussian(n, dim, seed=seed, latent=8)
        X[:, 8:12] = np.float32(0.75)
    elif kind == "int3":  # integer values {0, 1, 2}: exact distance ties everywhere
        X = rng.integers(0, 3, size=(n, dim)).astype(np.float32)
    elif kind == "huge":  # |x| up to ~4e19: most squared distances overflow f32 to +inf, not all
        X = synth.latent_gaussian(n, dim, seed=seed, latent=8) * np.float32(2e18)
    else:
        raise ValueError(kind)
    X = np.ascontiguousarray(X, dtype=np.float32)
    if metric == "cosine":
        X /= np.sqrt((X.astype(np.float64) ** 2).sum(1, keepdims=True)).astype(np.float32)
    return X


class PQCase:
    def __init__(self, name, metric, dim, M, K, n, kind, first):
        self.name, self.metric, self.dim, self.M, self.K, self.n, self.kind = name, metric, dim, M, K, n, kind
        self.sub = dim // M
        self.pq_metric = "euclidean" if metric == "cosine" else metric  # product.go:52-61
        seed = dim * 1000 + M * 10 + K
        rng = np.random.Generator(np.random.PCG64(seed))
        # ids with gaps: a sorted random sample of [2, 4n); a few deleted before the fit
        self.ids = np.sort(rng.choice(np.arange(2, 4 * n, dtype=np.uint32), size=n, replace=False))
        self.X = _rows(kind, n, dim, seed, metric)
        self.deleted = np.sort(rng.choice(self.ids, size=3 if n < 1000 else 7, replace=False))
        self.start = synth.start_vector(dim, seed + 1)
        keep = ~np.isin(self.ids, self.deleted)
        self.rows = np.concatenate([[1], self.ids[keep]]).astype(np.uint32)  # ascending id order, start node first
        self.Xfit = np.concatenate([self.start[None, :], self.X[keep]])  # what the fit reads
        self.first = len(self.rows) - 1 if first == "last" else first
        self.trigger = min(1000, len(self.rows))
        self.relaxed = self.trigger < 1000 or M < 2

    def __repr__(self):
        return self.name

    def path(self):
        return assign_path(self.dim, self.M, self.K, len(self.rows))

    def degenerate_init(self):
        """Some sub-space has fewer distinct sub-vectors than K, so the farthest-first init runs out
        of rows at a positive distance and falls back to row 0 (km_init_kernel)."""
        s = self.sub
        return any(len(np.unique(self.Xfit[:, m * s:(m + 1) * s], axis=0)) < self.K for m in range(self.M))


PQ_CASES = [
    # name                 metric      dim    M    K      n   data        first row
    PQCase("sub1",        "euclidean",    8,   8,  17,  1500, "gauss",     5),
    PQCase("sub2",        "dot",         16,   8, 255,  2000, "gauss",     "last"),
    PQCase("sub3",        "cosine",      24,   8,   3,  1200, "gauss",     0),
    PQCase("sub5",        "euclidean",   40,   8,   2,  1200, "gauss",     11),
    PQCase("sub4",        "dot",         64,  16,  64,  1500, "gauss",     7),
    PQCase("sub8",        "cosine",      64,   8,  32,  1500, "gauss",     "last"),
    PQCase("sub16",       "euclidean",   64,   4, 256,  3000, "gauss",     3),
    PQCase("staged96KB",  "euclidean",  192,   2, 256,  3000, "gauss",     9),  # K*sub*4 = 96 KB exactly
    PQCase("global100KB", "dot",        200,   2, 256,  3000, "gauss",     "last"),  # 100 KB: centres from global
    PQCase("wide512",     "cosine",    1024,   2,  64,  2000, "gauss",     1),
    PQCase("strided8",    "euclidean",   64,   8, 256, 20000, "clusters",  "last"),
    PQCase("strided4",    "dot",         32,   8,  64, 17000, "clusters",  "last"),
    PQCase("strided16",   "cosine",      64,   4, 128, 17000, "clusters",  "last"),
    PQCase("strided32",   "euclidean",   96,   3, 256, 20000, "clusters",  "last"),
    PQCase("strided100",  "euclidean",  100,   1, 256, 17000, "clusters",  "last"),
    PQCase("dup40",       "euclidean",   64,   8, 256,  3000, "dup40",     13),
    PQCase("const_sub",   "dot",         64,  16, 256,  3000, "const_sub", 21),
    PQCase("n_lt_K",      "cosine",      32,   4, 256,   100, "gauss",     50),
    PQCase("int3",        "euclidean",   48,  16, 256,  3000, "int3",      2),
    PQCase("huge",        "euclidean",   64,   8, 256,  3000, "huge",      17),
]


def test_case_table_reaches_every_fit_path():
    """CPU-only: the case table runs every assign form, staged and global centres, the strided
    row loop and the degenerate init branch, so the coverage below cannot erode silently."""
    paths = {c.path() for c in PQ_CASES}
    assert paths == reachable_paths(), sorted(reachable_paths() - paths)
    assert {c.sub for c in PQ_CASES} >= {1, 2, 3, 4, 5, 8, 16}
    assert {c.K for c in PQ_CASES} >= {2, 3, 17, 255, 256}
    assert {c.metric for c in PQ_CASES} == {"euclidean", "dot", "cosine"}
    # the register form and the generic form each stride with the last row as first centre
    strided = [c for c in PQ_CASES if c.path()[2]]
    assert {c.path()[0] != 0 for c in strided if c.first == len(c.rows) - 1} == {True, False}
    # the exact 96 KB boundary on both sides
    assert any(c.K * c.sub * 4 == KM_STAGE_BYTES for c in PQ_CASES)
    assert any(KM_STAGE_BYTES < c.K * c.sub * 4 <= KM_STAGE_BYTES + 4096 for c in PQ_CASES)
    # the degenerate init runs with a first row other than 0, so a fallback to it would show
    degenerate = [c for c in PQ_CASES if c.degenerate_init()]
    assert {c.kind for c in degenerate} >= {"dup40", "const_sub", "int3"} and any(c.n < c.K for c in degenerate)
    assert all(c.first != 0 for c in degenerate)
    for c in PQ_CASES:
        assert 0 <= c.first < len(c.rows)


# ---------------------------------------------------------------- helpers
def _same(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


def _pq_params(c, trigger=None):
    return IndexVectorVamanaParameters(c.dim, c.metric, quantizer=Quantizer(
        "product", product=ProductQuantizerParameters(c.K, c.M, c.trigger if trigger is None else trigger)))


def _pq_pair(c, trigger=None):
    """Oracle and GPU index holding the case's rows, the deleted ids gone."""
    oix = O.OracleIndex(c.dim, c.metric, quantizer="product", pq_m=c.M, pq_k=c.K,
                        pq_trigger=c.trigger if trigger is None else trigger)
    oix.set_start(c.start)
    oix.set_vectors(c.ids, c.X)
    oix.update_delete(c.deleted, np.zeros((len(c.deleted), c.dim), np.float32), np.zeros(len(c.deleted), np.uint8))
    g = IndexVamana("fit", _pq_params(c, trigger), start_vector=c.start, relaxed=c.relaxed)
    g.set_vectors(c.ids.astype(np.uint64), c.X)
    g.delete_rows(c.deleted.astype(np.uint64))
    assert oix.count == g.count == len(c.rows)
    return oix, g


def _check_table(metric, X, C, got, what):
    """got[i][j] is an f32 evaluation of the distance between X[i] and C[j]: within the gamma_n bound
    of the float64 value, +inf where that value is certainly above FLT_MAX."""
    d, b = f64_dists(metric, X, C)
    got = np.asarray(got, np.float64)
    over = d - b > FLT_MAX
    assert np.isposinf(got[over]).all(), what
    fin = d + b < FLT_MAX
    assert np.isfinite(got[fin]).all(), what
    err = np.abs(got[fin] - d[fin])
    assert (err <= b[fin]).all(), f"{what}: max excess {np.max(err - b[fin])}"


def _check_argmin(metric, X, C, codes, what):
    """codes[i] is an argmin over C of an f32 evaluation of the distance to X[i]: no centroid is
    certainly nearer (d64 + bound below the chosen one's d64 - bound). Distances that may exceed
    FLT_MAX may all be +inf in f32, and a chosen +inf means no candidate beat the first: code 0."""
    d, b = f64_dists(metric, X, C)
    lo, hi = d - b, d + b
    lo = np.where(lo > FLT_MAX, np.inf, lo)
    hi = np.where(hi > FLT_MAX, np.inf, hi)
    lo_c = lo[np.arange(len(X)), codes]
    bad = lo_c > hi.min(1)
    assert not bad.any(), f"{what}: rows {np.flatnonzero(bad)[:8]} codes {codes[bad][:8]}"
    assert (codes[np.isinf(lo_c)] == 0).all(), what


def _training_convergence(c, first):
    """Rounds the oracle's k-means runs per sub-space on the fit's input (kmeans.go:34-150) and its
    labels: converged when it stopped before the cap of 100 rounds."""
    X = np.ascontiguousarray(c.Xfit.copy())
    with ThreadPoolExecutor(8) as ex:  # the sub-spaces write disjoint columns of X
        res = list(ex.map(lambda m: O.kmeans_fit(X, c.K, MAX_ITER, m * c.sub, c.sub, first, alias=True)[1:3],
                          range(c.M)))
    return [it < MAX_ITER for _, it in res], np.stack([lab for lab, _ in res], 1)


def _f32_dists(metric, x, C):
    return np.array([O.float_dist(metric, x, c) for c in C], np.float32)


def _tied_midpoint(metric, a, b, C):
    """A sub-vector at the same f32 distance from centroids a and b and nearer to no other: the
    midpoint, its first element moved by up to 24 ulps until the two f32 distances are equal."""
    x = ((a.astype(np.float64) + b) / 2).astype(np.float32)
    for k in range(49):
        y = x.copy()
        step = np.float32(np.inf if k % 2 else -np.inf)
        for _ in range((k + 1) // 2):
            y[0] = np.nextafter(y[0], step)
        d = _f32_dists(metric, y, C)
        if O.float_dist(metric, y, a) == O.float_dist(metric, y, b) == d.min():
            return y
    return x


def _post_fit_rows(c, fc):
    """Rows to set after the fit: rows equal to a centroid in every sub-space, rows at the same
    distance from a centroid and its nearest distinct neighbour, a zero row, and rows of the
    training distribution."""
    rng = np.random.Generator(np.random.PCG64(c.dim + 7))
    M, K, s = c.M, c.K, c.sub
    eq = np.stack([np.concatenate([fc[m, rng.integers(0, K)] for m in range(M)]) for _ in range(8)])
    mid = []
    for _ in range(4):
        parts = []
        for m in range(M):
            a = fc[m, rng.integers(0, K)]
            d = f64_dists("euclidean", a[None, :], fc[m])[0][0]
            d[(fc[m] == a).all(1)] = np.inf
            parts.append(_tied_midpoint(c.pq_metric, a, fc[m, np.argmin(d)], fc[m]) if np.isfinite(d).any() else a)
        mid.append(np.concatenate(parts))
    fresh = _rows(c.kind, 16, c.dim, c.dim + 8, c.metric)
    return np.ascontiguousarray(np.concatenate([eq, np.stack(mid), np.zeros((1, c.dim), np.float32), fresh]))


def _exact_ties(c, fc, P):
    """(row, sub-space) pairs of P whose minimum f32 distance (the oracle's) is reached by two
    distinct centroids: the strict '<' of the encoder decides those."""
    ties = 0
    for p in P:
        for m in range(c.M):
            d = _f32_dists(c.pq_metric, p[m * c.sub:(m + 1) * c.sub], fc[m])
            at = np.flatnonzero(d == d.min())
            ties += len(at) > 1 and len(np.unique(fc[m, at], axis=0)) > 1
    return ties


# ---------------------------------------------------------------- 1 + 2: PQ fit parity and float64 bounds
@pytest.mark.gpu
@pytest.mark.parametrize("c", PQ_CASES, ids=repr)
def test_pq_fit_matches_oracle_and_float64(c):
    oix, g = _pq_pair(c)
    assert oix.fit(pq_first=c.first, pq_alias=True, threads=8) == 1
    assert g.fit(c.first) is True
    ofc, ocd = oix.get_pq()
    gfc, gcd = g.get_pq()
    assert _same(gfc, ofc), "flatCentroids"
    assert _same(gcd, ocd), "centroidDists"
    rows64 = c.rows.astype(np.uint64)
    codes = g.get_codes(rows64)
    assert _same(codes, oix.get_codes(c.rows)), "codes of the training rows"
    after = g.get_vectors(rows64)
    assert _same(after, oix.get_vectors(c.rows)), "written-through rows"
    Q = _rows(c.kind, 4, c.dim, c.dim + 9, c.metric)
    tabs = g.adc_tables(Q)
    for b in range(len(Q)):
        assert _same(tabs[b], oix.adc_table(Q[b])), f"ADC table {b}"

    # rows set after the fit go through pq_encode_kernel with the index metric (product.go:136-159)
    P = _post_fit_rows(c, gfc)
    pids = np.arange(4 * c.n, 4 * c.n + len(P), dtype=np.uint32)
    oix.set_vectors(pids, P)
    g.set_vectors(pids.astype(np.uint64), P)
    pcodes = g.get_codes(pids.astype(np.uint64))
    assert _same(pcodes, oix.get_codes(pids)), "codes of rows set after the fit"

    # float64: tables within the bound, codes an argmin up to it
    s = c.sub
    for m in range(c.M):
        _check_table(c.pq_metric, gfc[m], gfc[m], gcd[m], f"centroidDists[{m}]")
        _check_table(c.pq_metric, Q[:, m * s:(m + 1) * s], gfc[m], tabs[:, m], f"ADC[{m}]")
        _check_argmin(c.pq_metric, P[:, m * s:(m + 1) * s], gfc[m], pcodes[:, m], f"post-fit codes[{m}]")
    converged, labels = _training_convergence(c, c.first)
    assert _same(labels, codes), "oracle k-means labels on the fit's input"
    for m in np.flatnonzero(converged):
        # k-means assigns with squared L2 whatever the index metric (kmeans.go:100-115)
        _check_argmin("euclidean", after[:, m * s:(m + 1) * s], gfc[m], codes[:, m], f"training codes[{m}]")
    if c.kind not in ("huge",):
        assert _exact_ties(c, gfc, P) > 0 or c.K < 3, "no post-fit row ties two distinct centroids"


# ---------------------------------------------------------------- 3: the fit contract
@pytest.mark.gpu
def test_pq_fit_contract():
    """Below the trigger Fit does nothing; an out-of-range first row is rejected and leaves the
    store unfitted; a second Fit is a no-op (product.go:177-183)."""
    c = PQCase("contract", "euclidean", 64, 8, 32, 1500, "gauss", 0)
    n = len(c.rows)
    oix, g = _pq_pair(c, trigger=n + 1)
    assert oix.fit(pq_first=0, pq_alias=True) == 0
    assert g.fit(0) is False
    assert oix.get_pq() is None
    with pytest.raises(SdbError) as e:
        g.get_pq()
    assert e.value.code == ERR_STATE
    # one more row reaches the trigger; first row n is one past the last
    extra = _rows("gauss", 1, c.dim, 99, c.metric)
    xid = np.array([4 * c.n + 1], np.uint32)
    oix.set_vectors(xid, extra)
    g.set_vectors(xid.astype(np.uint64), extra)
    rows = np.concatenate([c.rows, xid])
    before = g.get_vectors(rows.astype(np.uint64))
    with pytest.raises(SdbError) as e:
        g.fit(n + 1)
    assert e.value.code == ERR_INVALID
    with pytest.raises(SdbError) as e:
        g.get_pq()
    assert e.value.code == ERR_STATE
    assert _same(g.get_vectors(rows.astype(np.uint64)), before)
    # a valid fit afterwards: the oracle's result
    assert oix.fit(pq_first=n, pq_alias=True, threads=8) == 1
    assert g.fit(n) is True
    ofc, ocd = oix.get_pq()
    gfc, gcd = g.get_pq()
    assert _same(gfc, ofc) and _same(gcd, ocd)
    codes = g.get_codes(rows.astype(np.uint64))
    vecs = g.get_vectors(rows.astype(np.uint64))
    assert _same(codes, oix.get_codes(rows)) and _same(vecs, oix.get_vectors(rows))
    # a second fit changes nothing
    assert g.fit(3) is False
    gfc2, gcd2 = g.get_pq()
    assert _same(gfc2, gfc) and _same(gcd2, gcd)
    assert _same(g.get_codes(rows.astype(np.uint64)), codes)
    assert _same(g.get_vectors(rows.astype(np.uint64)), vecs)


# ---------------------------------------------------------------- 4: BQ fit
def _bq_data(n, dim, seed):
    """Ids with gaps, a few deleted; one column constant and one of {0, 1, 2} with mean exactly 1 over
    the rows that stay, so values equal to the threshold meet the strict '>' (binary.go:123-127)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ids = np.sort(rng.choice(np.arange(2, 4 * n, dtype=np.uint32), size=n, replace=False))
    deleted = np.sort(rng.choice(ids, size=7, replace=False))
    keep = ~np.isin(ids, deleted)
    X = synth.latent_gaussian(n, dim, seed=seed, latent=8)
    start = synth.start_vector(dim, seed + 1)
    tri, R = dim - 1, int(keep.sum()) + 1
    s = rng.choice([-1.0, 0.0, 1.0], size=R // 2)
    dev = rng.permutation(np.concatenate([s, -s, np.zeros(R % 2)]))  # sums to 0 exactly
    start[tri] = np.float32(1 + dev[0])
    X[np.flatnonzero(keep), tri] = (1 + dev[1:]).astype(np.float32)
    if dim > 1:
        X[:, 0] = np.float32(0.25)
        start[0] = np.float32(0.25)
    return ids, deleted, X, start, np.concatenate([[1], ids[keep]]).astype(np.uint32)


def _bq_pair(dim, metric, ids, deleted, X, start, trigger, relaxed=False):
    oix = O.OracleIndex(dim, "euclidean", quantizer="binary", bq_metric=metric, bq_trigger=trigger)
    oix.set_start(start)
    oix.set_vectors(ids, X)
    oix.update_delete(deleted, np.zeros((len(deleted), dim), np.float32), np.zeros(len(deleted), np.uint8))
    params = IndexVectorVamanaParameters(dim, "euclidean", quantizer=Quantizer(
        "binary", binary=BinaryQuantizerParameters(None, trigger, metric)))
    g = IndexVamana("bq", params, start_vector=start, relaxed=relaxed)
    g.set_vectors(ids.astype(np.uint64), X)
    g.delete_rows(deleted.astype(np.uint64))
    return oix, g


def _check_bq_threshold(thr, Xfit):
    """Sequential f32 sum then one division (binary.go:161-173): within gamma_n * sum|x| / n plus one
    rounding of the float64 column mean."""
    n = len(Xfit)
    X64 = Xfit.astype(np.float64)
    mean = X64.sum(0) / n
    gamma = n * U32 / (1 - n * U32)
    bound = gamma * np.abs(X64).sum(0) / n * (1 + U32) + U32 * np.abs(mean) + 2.0 ** -50 * np.abs(X64).sum(0) / n
    assert (np.abs(thr.astype(np.float64) - mean) <= bound).all()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["hamming", "jaccard"])
@pytest.mark.parametrize("dim,n", [(1, 2500), (63, 2500), (64, 2500), (65, 2500), (100, 2500), (1000, 2500),
                                   (4096, 2500), (200, 20000)])
def test_bq_fit_matches_oracle(dim, n, metric):
    ids, deleted, X, start, rows = _bq_data(n, dim, dim * 7 + n)
    oix, g = _bq_pair(dim, metric, ids, deleted, X, start, trigger=2000)
    assert oix.fit() == 1
    assert g.fit() is True
    thr = g.get_bq_threshold()
    assert _same(thr, oix.get_bq_threshold())
    Xfit = oix.get_vectors(rows)
    _check_bq_threshold(thr, Xfit)
    if dim > 1:
        assert thr[0] == np.float32(0.25)
    assert thr[dim - 1] == np.float32(1.0)
    codes = g.get_codes(rows.astype(np.uint64))
    assert _same(codes, oix.get_codes(rows))
    # the codes against a plain restatement: bit i%64 of word i/64 set iff x[i] > thr[i]
    bits = np.packbits(Xfit > thr[None, :], axis=1, bitorder="little")
    ref = np.zeros_like(codes)
    ref[:, :bits.shape[1]] = bits
    assert _same(codes, ref)
    Q = synth.latent_gaussian(16, dim, seed=dim + 3, w_seed=dim * 7 + n, latent=8)
    gt = oix.flat_search(Q, k=10, threads=8)
    fi, fd, fc = g.flat_search_batch(Q, 10)
    assert (fi == gt["ids"].astype(np.uint64)).all() and _same(fd, gt["dists"]) and (fc == gt["counts"]).all()
    assert g.fit() is False
    assert _same(g.get_bq_threshold(), thr)


# ---------------------------------------------------------------- 5: hydrate
@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["euclidean", "dot"])
def test_set_pq_reencodes_like_the_oracle(metric):
    """sdb_index_set_pq on a fresh index of raw rows re-encodes every row with the index metric like
    the oracle's set_pq(reencode=True); for euclidean, where k-means and the encoder take the same
    argmin, the codes are those the converged fit produced."""
    c = PQCase("hydrate", metric, 64, 8, 32, 1500, "clusters", 4)
    oix, g = _pq_pair(c)
    assert oix.fit(pq_first=c.first, pq_alias=True, threads=8) == 1
    assert g.fit(c.first) is True
    fc, cd = g.get_pq()
    R = g.get_vectors(c.rows.astype(np.uint64))  # the rows as the fit left them
    users = c.rows[1:]
    o2 = O.OracleIndex(c.dim, metric, quantizer="product", pq_m=c.M, pq_k=c.K, pq_trigger=c.trigger)
    o2.set_start(R[0])
    o2.set_vectors(users, R[1:])
    o2.set_pq(fc, cd, reencode=True)
    g2 = IndexVamana("hydrate", _pq_params(c), start_vector=R[0], relaxed=c.relaxed)
    g2.set_vectors(users.astype(np.uint64), R[1:])
    g2.set_pq(fc, cd)
    codes = g2.get_codes(c.rows.astype(np.uint64))
    assert _same(codes, o2.get_codes(c.rows))
    if metric == "euclidean":
        converged, _ = _training_convergence(c, c.first)
        assert all(converged)
        assert _same(codes, g.get_codes(c.rows.astype(np.uint64)))
    Q = _rows(c.kind, 8, c.dim, 77, metric)
    for q in Q[:3]:
        assert _same(g2.query_dists(q, users.astype(np.uint64)), o2.query_dists(q, users))
    assert _same(g2.point_dists(int(users[5]), users.astype(np.uint64)),
                 np.array([o2.point_dist(int(users[5]), int(i)) for i in users], np.float32))
    gt = o2.flat_search(Q, k=10, threads=8)
    fi, fd, fcnt = g2.flat_search_batch(Q, 10)
    assert (fi == gt["ids"].astype(np.uint64)).all() and _same(fd, gt["dists"]) and (fcnt == gt["counts"]).all()
    assert g2.fit(0) is False  # installed state counts as fitted


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["hamming", "jaccard"])
def test_set_bq_threshold_reencodes_like_the_fit(metric):
    dim, n = 130, 3000
    ids, deleted, X, start, rows = _bq_data(n, dim, 5)
    oix, g = _bq_pair(dim, metric, ids, deleted, X, start, trigger=2000)
    assert oix.fit() == 1 and g.fit() is True
    thr = g.get_bq_threshold()
    users = rows[1:]
    params = IndexVectorVamanaParameters(dim, "euclidean", quantizer=Quantizer(
        "binary", binary=BinaryQuantizerParameters(None, 2000, metric)))
    g2 = IndexVamana("bq2", params, start_vector=start)
    g2.set_vectors(users.astype(np.uint64), oix.get_vectors(users))
    g2.set_bq_threshold(thr)
    assert _same(g2.get_bq_threshold(), thr)
    codes = g2.get_codes(rows.astype(np.uint64))
    assert _same(codes, oix.get_codes(rows)) and _same(codes, g.get_codes(rows.astype(np.uint64)))
    Q = synth.latent_gaussian(8, dim, seed=6, w_seed=5, latent=8)
    for q in Q[:3]:
        assert _same(g2.query_dists(q, users.astype(np.uint64)), oix.query_dists(q, users))
    assert _same(g2.point_dists(int(users[5]), users.astype(np.uint64)),
                 np.array([oix.point_dist(int(users[5]), int(i)) for i in users], np.float32))
    gt = oix.flat_search(Q, k=10, threads=8)
    fi, fd, fcnt = g2.flat_search_batch(Q, 10)
    assert (fi == gt["ids"].astype(np.uint64)).all() and _same(fd, gt["dists"]) and (fcnt == gt["counts"]).all()
    assert g2.fit() is False
