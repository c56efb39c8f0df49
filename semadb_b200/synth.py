"""Synthetic inputs for the BASELINE.json configs (BASELINE.md §4, SURVEY.md §8d).

All generators are numpy.random.Generator(PCG64(seed)), float32, deterministic.
Shared by tests/ and bench.py; no oracle or CUDA dependency.
"""
from __future__ import annotations

import numpy as np


def uniform(n: int, dim: int, seed: int) -> np.ndarray:
    """C1: iid U[0,1) like internal/loadrand/loadrand.go:17-23."""
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.random((n, dim), dtype=np.float32)


def _latent_w(latent: int, dim: int, seed: int) -> np.ndarray:
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.standard_normal((latent, dim), dtype=np.float32)


def _latent_points(n: int, latent: int, dim: int, w: np.ndarray, seed: int, chunk: int = 1 << 18) -> np.ndarray:
    rng = np.random.Generator(np.random.PCG64(seed + 7919))
    out = np.empty((n, dim), dtype=np.float32)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        z = rng.standard_normal((m, latent), dtype=np.float32)
        eps = rng.standard_normal((m, dim), dtype=np.float32)
        out[s:s + m] = z @ w + np.float32(0.1) * eps
    return out


def sift_shaped(n: int, dim: int = 128, seed: int = 3, w_seed: int | None = None, latent: int = 16) -> np.ndarray:
    """C2 "SIFT-shaped": z~N(0,I_16), x = clip(round(32*(zW+0.1e)+64), 0, 255).
    Queries use their own seed but the data's W (w_seed = data seed)."""
    w = _latent_w(latent, dim, seed if w_seed is None else w_seed)
    x = _latent_points(n, latent, dim, w, seed)
    np.multiply(x, np.float32(32), out=x)
    np.add(x, np.float32(64), out=x)
    np.rint(x, out=x)
    np.clip(x, 0, 255, out=x)
    return x


def latent_gaussian(n: int, dim: int, seed: int, w_seed: int | None = None, latent: int = 16,
                    normalize: bool = False) -> np.ndarray:
    """C3 (latent-16, L2-normalised, cosine) / C4 (latent-64, raw, dot)."""
    w = _latent_w(latent, dim, seed if w_seed is None else w_seed)
    x = _latent_points(n, latent, dim, w, seed)
    if normalize:
        nrm = np.sqrt((x.astype(np.float64) ** 2).sum(axis=1, keepdims=True)).astype(np.float32)
        x /= np.maximum(nrm, np.float32(1e-30))
    return x


def planted_bits(n: int, dim: int = 1024, seed: int = 7, n_proto: int = 65536, flip: float = 0.1,
                 proto_seed: int | None = None, chunk: int = 1 << 16) -> np.ndarray:
    """C5b: prototypes Bernoulli(0.5); each point = a random prototype with `flip` of its
    bits flipped; returned as 0.0/1.0 float32 (binarised with threshold 0.5,
    shard/vectorstore/vectorstore.go:56-66)."""
    prng = np.random.Generator(np.random.PCG64(seed if proto_seed is None else proto_seed))
    protos = prng.random((n_proto, dim), dtype=np.float32) < 0.5
    rng = np.random.Generator(np.random.PCG64(seed + 104729))
    out = np.empty((n, dim), dtype=np.float32)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        pick = rng.integers(0, n_proto, size=m)
        flips = rng.random((m, dim), dtype=np.float32) < flip
        out[s:s + m] = np.logical_xor(protos[pick], flips)
    return out


def start_vector(dim: int, seed: int) -> np.ndarray:
    """setupStartNode (shard/index/vamana/vamana.go:100-110): U(-1,1)^dim, L2-normalised,
    sum accumulated in f32 in index order like the reference loop."""
    rng = np.random.Generator(np.random.PCG64(seed))
    v = (rng.random(dim, dtype=np.float32) * np.float32(2) - np.float32(1)).astype(np.float32)
    s = np.float32(0)
    for x in v:
        s = np.float32(s + np.float32(x * x))
    norm = np.float32(1) / np.float32(np.sqrt(np.float64(s)))
    return (v * norm).astype(np.float32)


# ---- device-side generators (bench.py at shard sizes: 6.25M x 1024 floats do not fit a host
# generator's time budget). Same distributions as above drawn with torch.Generator on the CUDA
# device: deterministic for a given (seed, GPU model, torch build), NOT bit-equal to the numpy ones.
# Tests use the numpy generators; the bench states "synthetic (device-generated)".

def _torch_w(latent: int, dim: int, seed: int, device):
    import torch
    return torch.from_numpy(_latent_w(latent, dim, seed)).to(device)


def latent_gaussian_torch(n: int, dim: int, seed: int, device, w_seed: int | None = None, latent: int = 16,
                          normalize: bool = False, centres: int = 0, spread: float = 0.3, centre_seed: int = 1234,
                          chunk: int = 1 << 18):
    """Yields (start, X) chunks on `device`: x = zW + 0.1e with z ~ N(0, I_latent) — or, with
    centres > 0, z = c_j + spread * N(0, I) for a random one of `centres` fixed centres
    c_j ~ N(0, I) (clustered embedding data, C4) — optionally L2-normalised."""
    import torch
    w = _torch_w(latent, dim, seed if w_seed is None else w_seed, device)
    g = torch.Generator(device=device)
    g.manual_seed(int(seed) * 7919 + 17)
    cent = None
    if centres:
        gc = torch.Generator(device=device)
        gc.manual_seed(int(centre_seed))
        cent = torch.randn((centres, latent), generator=gc, device=device, dtype=torch.float32)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        z = torch.randn((m, latent), generator=g, device=device, dtype=torch.float32)
        if cent is not None:
            pick = torch.randint(0, centres, (m,), generator=g, device=device)
            z = cent[pick] + spread * z
        x = z @ w
        x.add_(torch.randn((m, dim), generator=g, device=device, dtype=torch.float32), alpha=0.1)
        if normalize:
            x /= x.norm(dim=1, keepdim=True).clamp_min(1e-30)
        yield s, x


def sign_bits_torch(n: int, dim: int, seed: int, device, w_seed: int | None = None, latent: int = 16,
                    chunk: int = 1 << 18):
    """C5b (BASELINE.md §4, amended): what binary quantisation of embedding vectors produces —
    bit i = (x_i > 0) of a latent-Gaussian embedding, supplied as 0.0/1.0 floats so the forced
    0.5 threshold of hamming/jaccard indexes (shard/vectorstore/vectorstore.go:56-66) recovers it."""
    for s, x in latent_gaussian_torch(n, dim, seed, device, w_seed=w_seed, latent=latent, chunk=chunk):
        yield s, (x > 0).to(x.dtype)


def sign_bits(n: int, dim: int, seed: int, w_seed: int | None = None, latent: int = 16) -> np.ndarray:
    """numpy twin of sign_bits_torch (tests, small sizes)."""
    return (latent_gaussian(n, dim, seed, w_seed=w_seed, latent=latent) > 0).astype(np.float32)


def clustered_latent(n: int, dim: int, seed: int, w_seed: int | None = None, latent: int = 16, centres: int = 2048,
                     spread: float = 0.3, centre_seed: int = 1234, normalize: bool = True) -> np.ndarray:
    """numpy twin of latent_gaussian_torch(centres=...) (tests, small sizes)."""
    w = _latent_w(latent, dim, seed if w_seed is None else w_seed)
    cent = np.random.Generator(np.random.PCG64(centre_seed)).standard_normal((centres, latent), dtype=np.float32)
    rng = np.random.Generator(np.random.PCG64(seed + 7919))
    pick = rng.integers(0, centres, size=n)
    z = cent[pick] + np.float32(spread) * rng.standard_normal((n, latent), dtype=np.float32)
    x = z @ w + np.float32(0.1) * rng.standard_normal((n, dim), dtype=np.float32)
    if normalize:
        x /= np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-30)
    return x.astype(np.float32)


# ---- geo (haversine, dim 2): rows are (latitude, longitude) in degrees, x[0] = latitude like the
# reference's KAT [-34.83333, -58.5166646] (Buenos Aires).

def _geo_centres(centres: int, seed: int) -> tuple[np.ndarray, np.ndarray]:
    """City centres uniform on the sphere (lat = asin(U[-1,1])); centre 0 sits on the north pole,
    centre 1 on the south pole and centre 2 on the antimeridian, so those cases always occur."""
    rng = np.random.Generator(np.random.PCG64(seed))
    clat = np.degrees(np.arcsin(rng.uniform(-1.0, 1.0, centres)))
    clon = rng.uniform(-180.0, 180.0, centres)
    if centres > 0:
        clat[0] = 90.0
    if centres > 1:
        clat[1] = -90.0
    if centres > 2:
        clon[2] = 180.0
    return clat, clon


def _geo_draw(n: int, rng, clat, clon, spread_deg: float, background: float) -> np.ndarray:
    lat = np.empty(n, dtype=np.float64)
    lon = np.empty(n, dtype=np.float64)
    bg = rng.random(n) < background if len(clat) else np.ones(n, dtype=bool)
    nb = int(bg.sum())
    lat[bg] = np.degrees(np.arcsin(rng.uniform(-1.0, 1.0, nb)))
    lon[bg] = rng.uniform(-180.0, 180.0, nb)
    nc = n - nb
    if nc:
        k = rng.integers(0, len(clat), nc)
        lat[~bg] = clat[k] + rng.normal(0.0, spread_deg, nc)
        lon[~bg] = clon[k] + rng.normal(0.0, spread_deg, nc)
    np.clip(lat, -90.0, 90.0, out=lat)
    lon = (lon + 180.0) % 360.0 - 180.0  # wrap into [-180, 180)
    return _geo_f32(lat, lon)


def _geo_f32(lat, lon) -> np.ndarray:
    out = np.stack([lat, lon], 1).astype(np.float32)
    out[out[:, 1] >= 180.0, 1] = -180.0  # a longitude just below 180 can round up to it in float32
    return out


def geo_points(n: int, seed: int, centres: int = 200, spread_deg: float = 0.5, background: float = 0.1) -> np.ndarray:
    """float32 [n, 2] (lat, lon) in degrees: a `background` fraction uniform on the sphere, the rest
    clustered around `centres` "cities" (normal, `spread_deg` per coordinate). Longitudes wrap into
    [-180, 180), so the antimeridian city straddles it; latitudes are clipped at +-90, so the polar
    cities pile up on the poles."""
    clat, clon = _geo_centres(centres, seed)
    return _geo_draw(n, np.random.Generator(np.random.PCG64(seed + 7919)), clat, clon, spread_deg, background)


def geo_queries(n: int, seed: int, centres: int = 200, spread_deg: float = 0.5, background: float = 0.1,
                jitter_deg: float = 0.01, query_seed: int = 1) -> np.ndarray:
    """Queries for geo_points(..., seed, centres, spread_deg, background): fresh draws from the same
    cities and background (own stream, query_seed), each jittered by N(0, jitter_deg)."""
    clat, clon = _geo_centres(centres, seed)
    rng = np.random.Generator(np.random.PCG64(seed + 15485863 * query_seed))
    q = _geo_draw(n, rng, clat, clon, spread_deg, background).astype(np.float64)
    q += rng.normal(0.0, jitter_deg, q.shape)
    np.clip(q[:, 0], -90.0, 90.0, out=q[:, 0])
    q[:, 1] = (q[:, 1] + 180.0) % 360.0 - 180.0
    return _geo_f32(q[:, 0], q[:, 1])
