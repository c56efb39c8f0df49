// prune.cuh — shared pieces of the graph-mutation kernels (insert.cu, delete.cu): the store
// view for DistanceFromPoint (plain.go:87-97, binary.go:213-234, product.go:279-305), the
// stable candidate sort (distset.go:223-238) and robustPrune (search.go:106-138) run by one
// CTA over a candidate list held in shared memory.
#pragma once
#include "common.cuh"
#include "index.cuh"

namespace sdb {

constexpr int PRUNE_THREADS = 256;
constexpr int PRUNE_GROUPS = PRUNE_THREADS / 8;
constexpr int MAX_CAND = 512;  // visited-list capacity handed to robustPrune (hamming shards of 6M points expand > 256 nodes for some inserts)

struct StoreView {
  int mode;  // 0 float rows, 1 bit rows, 2 PQ codes (SDC)
  int metric;
  const float* vec; uint32_t vec_pitch; uint32_t dim;
  const uint64_t* bits; uint32_t bits_pitch; uint32_t words;
  const uint8_t* codes; uint32_t codes_pitch; uint32_t pqM, pqK;
  const float* cdist;
  uint32_t row_bytes;  // bytes staged per candidate row
};

// Candidate list of one CTA, carved out of dynamic shared memory (capacity chosen per launch).
struct PruneShared {
  uint32_t* id;      // [cap] arrival order
  float* dist;       // [cap]
  uint32_t* sid;     // [cap] sorted by distance (stable)
  float* sdist;      // [cap]
  uint8_t* removed;  // [cap]
  uint32_t* edges;   // [64] result
  uint32_t* kill;    // [MATRIX_MAX][MATRIX_MAX/32] bit (i, j): accepting candidate i removes candidate j;
                     // overlays id/dist, which are dead once the candidates are sorted (nullptr if they are too small)
  int n;             // candidates (same value in every thread)
  int* cnt;          // shared: edges written so far
  static constexpr int MATRIX_MAX = 128;
  static __host__ __device__ size_t bytes(int cap) {
    return ((size_t(cap) * 17 + 15) / 16) * 16 + 64 * 4 + 16;
  }
  // returns the first byte after the carved area (16-byte aligned)
  __device__ __forceinline__ unsigned char* carve(unsigned char* base, int cap) {
    id = reinterpret_cast<uint32_t*>(base);
    dist = reinterpret_cast<float*>(base + size_t(cap) * 4);
    sid = reinterpret_cast<uint32_t*>(base + size_t(cap) * 8);
    sdist = reinterpret_cast<float*>(base + size_t(cap) * 12);
    removed = base + size_t(cap) * 16;
    unsigned char* p = base + ((size_t(cap) * 17 + 15) / 16) * 16;
    edges = reinterpret_cast<uint32_t*>(p);
    cnt = reinterpret_cast<int*>(p + 64 * 4);
    kill = size_t(cap) * 8 >= size_t(MATRIX_MAX) * (MATRIX_MAX / 32) * 4 ? reinterpret_cast<uint32_t*>(base) : nullptr;
    n = 0;
    return p + 64 * 4 + 16;
  }
};

// distance between two staged rows by an 8-lane group; result valid in the group's lane 0.
// All 32 lanes of the warp must call it together.
template <int METRIC>
__device__ __forceinline__ float group_float_dist(const float* x, const float* y, uint32_t dim, int g) {
  constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
  const int trips = dim >> 5;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int t = 0; t < trips; ++t) {
    float4 a = *reinterpret_cast<const float4*>(x + 32 * t + 4 * g);
    float4 b = *reinterpret_cast<const float4*>(y + 32 * t + 4 * g);
    trip_accum<L2>(a, b, acc);
  }
  float tail = 0.0f;
  if (g == 0)
    for (uint32_t i = trips << 5; i < dim; ++i) tail = tail_accum<L2>(x[i], y[i], tail);
  return metric_epilogue<METRIC>(group_reduce(acc, tail));
}

// same for two rows known to sit in shared memory, dim = 32 * TRIPS
template <int METRIC, int TRIPS>
__device__ __forceinline__ float smem_float_dist(const float* x, const float* y, int g) {
  constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
  const uint32_t xa = uint32_t(__cvta_generic_to_shared(x)) + 16u * g, ya = uint32_t(__cvta_generic_to_shared(y)) + 16u * g;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int t = 0; t < TRIPS; ++t) {
    float4 a, b;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(xa + 128u * t));
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(ya + 128u * t));
    trip_accum<L2>(a, b, acc);
  }
  return metric_epilogue<METRIC>(group_reduce(acc, 0.0f));
}

__device__ __forceinline__ float row_dist(const StoreView& s, const unsigned char* x, const unsigned char* y, int g) {
  if (s.mode == 0) {
    const float* a = reinterpret_cast<const float*>(x);
    const float* b = reinterpret_cast<const float*>(y);
    switch (s.metric) {
      case METRIC_EUCLIDEAN: return group_float_dist<METRIC_EUCLIDEAN>(a, b, s.dim, g);
      case METRIC_DOT: return group_float_dist<METRIC_DOT>(a, b, s.dim, g);
      case METRIC_COSINE: return group_float_dist<METRIC_COSINE>(a, b, s.dim, g);
      default: {
        // haversine: float64 math in lane 0; keep the warp's shuffle count consistent
        float r = (g == 0) ? haversine_thread(a, b) : 0.0f;
        return r;
      }
    }
  }
  float r = 0.0f;
  if (s.mode == 1) {
    // bit rows: the 8 lanes split the words (integer sums: order-free)
    const uint64_t* a = reinterpret_cast<const uint64_t*>(x);
    const uint64_t* b = reinterpret_cast<const uint64_t*>(y);
    int c = 0, u = 0;
    for (uint32_t w = g; w < s.words; w += 8) {
      if (s.metric == METRIC_JACCARD) { c += __popcll(a[w] & b[w]); u += __popcll(a[w] | b[w]); }
      else c += __popcll(a[w] ^ b[w]);
    }
#pragma unroll
    for (int o = 4; o >= 1; o >>= 1) {
      c += __shfl_down_sync(SDB_FULL, c, o, 8);
      u += __shfl_down_sync(SDB_FULL, u, o, 8);
    }
    r = bits_finish(s.metric, c, u);
  } else {
    // SDC: sum_i centroidDists[i][cx[i]][cy[i]], added sequentially in f32 (product.go:299-303).
    // The M table reads are independent: the group's 8 lanes fetch 32 of them at a time (4 each, all
    // in flight together), then the terms are added in sub-vector order through shuffles — the same
    // chain of additions, without M dependent L2 round trips in one lane.
    for (uint32_t m0 = 0; m0 < s.pqM; m0 += 32) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t m = m0 + 8 * u + g;
        v[u] = m < s.pqM ? __ldg(s.cdist + (size_t(m) * s.pqK + x[m]) * s.pqK + y[m]) : 0.0f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int l = 0; l < 8; ++l) {
          const float t = __shfl_sync(SDB_FULL, v[u], l, 8);
          if (m0 + 8 * u + l < s.pqM) r = __fadd_rn(r, t);  // warp-uniform
        }
      }
    }
  }
  return r;
}

__device__ __forceinline__ const unsigned char* global_row(const StoreView& s, uint32_t id) {
  if (s.mode == 0) return reinterpret_cast<const unsigned char*>(s.vec + size_t(id) * s.vec_pitch);
  if (s.mode == 1) return reinterpret_cast<const unsigned char*>(s.bits + size_t(id) * s.bits_pitch);
  return s.codes + size_t(id) * s.codes_pitch;
}

// Stable sort of (id, dist)[0..n) by distance into (sid, sdist): equals the reference's
// insertion sort (distset.go:223-238, strict '<' swaps => stable).
__device__ inline void stable_sort_by_dist(PruneShared& sh) {
  const int n = sh.n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float di = sh.dist[i];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      float dj = sh.dist[j];
      rank += (dj < di) || (dj == di && j < i);
    }
    sh.sid[rank] = sh.id[i];
    sh.sdist[rank] = di;
  }
  __syncthreads();
}

// Stage rows of the sorted candidates into shared memory (as many as fit).
__device__ inline void stage_rows(const StoreView& s, PruneShared& sh, unsigned char* rows, int staged) {
  const uint32_t vec16 = s.row_bytes / 16;
  const uint32_t total = uint32_t(staged) * vec16;
  for (uint32_t t = threadIdx.x; t < total; t += blockDim.x) {
    const uint32_t c = t / vec16, i = t % vec16;
    const uint4* src = reinterpret_cast<const uint4*>(global_row(s, sh.sid[c]));
    reinterpret_cast<uint4*>(rows + size_t(c) * s.row_bytes)[i] = __ldg(src + i);
  }
  __syncthreads();
}

// robustPrune (search.go:106-138) over the sorted candidates in sh.sid/sdist; node = id of
// the node being pruned (skipped if it appears, search.go:116). Fills sh.edges/sh.cnt.
//
// The reference walks the candidates in ascending order; an accepted candidate p* removes every
// later candidate c with alpha * d(p*, c) < d(node, c) (search.go:132, strict). Whether p* removes
// c does not depend on the walk, only on the pair — so for lists of up to MATRIX_MAX candidates
// (back-edge prunes have R+1 = 65) all pairs (i < j) are evaluated first, in parallel by the CTA's
// 8-lane groups with no barrier in the loop, into a bit matrix kill[i] = {j : alpha * d(i, j) <
// sdist[j]}; one warp then replays the walk with bit operations: skip removed / self, accept, stop
// at R, removed |= kill[i]. Same distances, same comparisons, same edges as the sequential form
// (kept below for longer lists, and for a new point's ~80-100 candidates, insert.cu), which spent
// its time in one block-wide barrier per accepted candidate (profiles/r01_ab_insert.txt: 30 %
// barrier stalls in backedge_kernel).
__device__ inline void robust_prune_cta_seq(const StoreView& s, PruneShared& sh, const unsigned char* rows, int staged,
                                            uint32_t node, int R, float alpha) {
  const int n = sh.n;
  const int lane = threadIdx.x & 31;
  const int g = lane & 7;
  const int grp = threadIdx.x >> 3;  // 0..PRUNE_GROUPS-1
  for (int i = threadIdx.x; i < n; i += blockDim.x) sh.removed[i] = 0;
  __syncthreads();
  // every thread tracks the edge count in a register (the decisions below are block-uniform):
  // one barrier per accepted candidate — after its removal marks — instead of three
  int cnt = 0;
  for (int i = 0; i < n; ++i) {
    if (sh.removed[i] || sh.sid[i] == node) continue;  // block-uniform
    if (threadIdx.x == 0) sh.edges[cnt] = sh.sid[i];
    ++cnt;
    if (cnt >= R) break;
    const unsigned char* xi = i < staged ? rows + size_t(i) * s.row_bytes : global_row(s, sh.sid[i]);
    for (int j0 = i + 1; j0 < n; j0 += PRUNE_GROUPS) {
      int j = j0 + grp;
      bool act = (j < n) && !sh.removed[j];
      // warp-uniform skip when none of this warp's 4 groups has work
      if (!__any_sync(SDB_FULL, act)) continue;
      int jj = act ? j : i;
      const unsigned char* yj = jj < staged ? rows + size_t(jj) * s.row_bytes : global_row(s, sh.sid[jj]);
      float d = row_dist(s, xi, yj, g);
      if (act && g == 0 && __fmul_rn(alpha, d) < sh.sdist[j]) sh.removed[j] = 1;  // search.go:132
    }
    __syncthreads();  // removal marks of this round are visible before the next candidate is read
  }
  if (threadIdx.x == 0) *sh.cnt = cnt;
  __syncthreads();
}

// All pairs (i < j) of the sorted candidates into the kill matrix. Rows are handed out in mirrored
// pairs (u, n-2-u) — n-1-u and u+1 columns, n steps together — so every 8-lane group runs the same
// number of steps and no index arithmetic beyond a compare is needed; a middle row (odd number of
// rows) forms a unit of its own. DIST(xi, yj, g) = DistanceFromPoint of the store, valid in lane 0
// of the group.
template <bool ALLSTAGED, class Dist>
__device__ __forceinline__ void prune_fill_kill(const StoreView& s, PruneShared& sh, const unsigned char* rows, int staged,
                                                float alpha, Dist&& dist) {
  constexpr int KW = PruneShared::MATRIX_MAX / 32;
  const int n = sh.n;
  const int lane = threadIdx.x & 31;
  const int g = lane & 7;
  const int grp = threadIdx.x >> 3;
  const int nrows = n - 1;          // rows 0 .. n-2 have at least one column
  const int P = nrows / 2;          // mirrored pairs
  const int U = P + (nrows & 1);    // + the middle row
  for (int u0 = 0; u0 < U; u0 += PRUNE_GROUPS) {
    const int u = u0 + grp;
    const bool has = u < U;
    const int ra = has ? u : 0;                      // first row of the unit
    const int la = has ? n - 1 - ra : 0;             // its columns
    const int rb = n - 2 - u;                        // mirrored row (none for the middle unit)
    const int lb = (has && u < P) ? u + 1 : 0;
    for (int step = 0; step < n; ++step) {           // la + lb <= n
      const bool first = step < la;
      const bool act = first || step - la < lb;
      if (!__any_sync(SDB_FULL, act)) continue;      // warp-uniform
      const int i = act ? (first ? ra : rb) : 0;
      const int j = act ? (first ? ra + 1 + step : rb + 1 + (step - la)) : 1;
      const unsigned char* xi = (ALLSTAGED || i < staged) ? rows + uint32_t(i) * s.row_bytes : global_row(s, sh.sid[i]);
      const unsigned char* yj = (ALLSTAGED || j < staged) ? rows + uint32_t(j) * s.row_bytes : global_row(s, sh.sid[j]);
      const float d = dist(xi, yj, g);
      if (act && g == 0 && __fmul_rn(alpha, d) < sh.sdist[j]) atomicOr(&sh.kill[i * KW + (j >> 5)], 1u << (j & 31));  // search.go:132
    }
  }
}

__device__ inline void robust_prune_cta(const StoreView& s, PruneShared& sh, const unsigned char* rows, int staged,
                                        uint32_t node, int R, float alpha) {
  const int n = sh.n;
  if (n > PruneShared::MATRIX_MAX || sh.kill == nullptr) {
    robust_prune_cta_seq(s, sh, rows, staged, node, R, alpha);
    return;
  }
  constexpr int KW = PruneShared::MATRIX_MAX / 32;
  for (int t = threadIdx.x; t < n * KW; t += blockDim.x) sh.kill[t] = 0;
  __syncthreads();
  // the store's DistanceFromPoint, resolved once per prune rather than per pair. Fast path: f32 rows
  // of 32*TRIPS floats, every candidate staged in shared memory (the back-edge prune of a dim-128
  // store): compile-time trip count, shared-memory loads only.
  const bool all_staged = s.mode == 0 && staged >= n && (s.dim & 31u) == 0;
  const int trips = int(s.dim >> 5);
#define SDB_PRUNE_FAST(M, T)                                                                                     \
  prune_fill_kill<true>(s, sh, rows, staged, alpha, [&](const unsigned char* x, const unsigned char* y, int g) { \
    return smem_float_dist<M, T>(reinterpret_cast<const float*>(x), reinterpret_cast<const float*>(y), g);      \
  })
  if (all_staged && s.metric == METRIC_EUCLIDEAN && trips == 4) {
    SDB_PRUNE_FAST(METRIC_EUCLIDEAN, 4);
  } else if (all_staged && s.metric == METRIC_EUCLIDEAN && trips == 12) {
    SDB_PRUNE_FAST(METRIC_EUCLIDEAN, 12);
  } else if (all_staged && s.metric == METRIC_COSINE && trips == 12) {
    SDB_PRUNE_FAST(METRIC_COSINE, 12);
  } else if (all_staged && s.metric == METRIC_DOT && trips == 24) {
    SDB_PRUNE_FAST(METRIC_DOT, 24);
  } else
#undef SDB_PRUNE_FAST
  if (s.mode == 0 && s.metric == METRIC_EUCLIDEAN) {
    prune_fill_kill<false>(s, sh, rows, staged, alpha, [&](const unsigned char* x, const unsigned char* y, int g) {
      return group_float_dist<METRIC_EUCLIDEAN>(reinterpret_cast<const float*>(x), reinterpret_cast<const float*>(y), s.dim, g);
    });
  } else if (s.mode == 0 && s.metric == METRIC_DOT) {
    prune_fill_kill<false>(s, sh, rows, staged, alpha, [&](const unsigned char* x, const unsigned char* y, int g) {
      return group_float_dist<METRIC_DOT>(reinterpret_cast<const float*>(x), reinterpret_cast<const float*>(y), s.dim, g);
    });
  } else if (s.mode == 0 && s.metric == METRIC_COSINE) {
    prune_fill_kill<false>(s, sh, rows, staged, alpha, [&](const unsigned char* x, const unsigned char* y, int g) {
      return group_float_dist<METRIC_COSINE>(reinterpret_cast<const float*>(x), reinterpret_cast<const float*>(y), s.dim, g);
    });
  } else {
    prune_fill_kill<false>(s, sh, rows, staged, alpha,
                    [&](const unsigned char* x, const unsigned char* y, int g) { return row_dist(s, x, y, g); });
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // the walk (search.go:113-137) by one thread: the removed set lives in KW registers and the
    // next candidate still alive is found with a find-first-set over ~removed, so the loop runs
    // once per ACCEPTED candidate (~35 of 65); a kill row is one 128-bit shared-memory load
    static_assert(KW == 4, "the walk keeps the removed set in four registers");
    uint32_t rem[KW] = {0u, 0u, 0u, 0u};
    int cnt = 0;
    const uint4* krow = reinterpret_cast<const uint4*>(sh.kill);
    bool done = false;
#pragma unroll
    for (int w = 0; w < KW; ++w) {
      if (done || 32 * w >= n) break;
      const uint32_t valid = n - 32 * w >= 32 ? 0xFFFFFFFFu : ((1u << (n - 32 * w)) - 1u);
      uint32_t todo = valid;  // candidates of this word not yet looked at
      while (true) {
        const uint32_t avail = ~rem[w] & todo;
        if (!avail) break;
        const int b = __ffs(avail) - 1;
        todo = b == 31 ? 0u : (todo & ~((2u << b) - 1u));
        const int i = 32 * w + b;
        const uint32_t id = sh.sid[i];
        if (id == node) continue;
        sh.edges[cnt] = id;
        ++cnt;
        if (cnt >= R) { done = true; break; }
        const uint4 k = krow[i];
        rem[0] |= k.x; rem[1] |= k.y; rem[2] |= k.z; rem[3] |= k.w;
      }
    }
    *sh.cnt = cnt;
  }
  __syncthreads();
}

inline StoreView make_view(const sdb_index* ix) {
  StoreView s{};
  s.vec = ix->d_vec; s.vec_pitch = ix->vec_pitch; s.dim = ix->p.dim;
  s.bits = ix->d_bits; s.bits_pitch = ix->bits_pitch; s.words = ix->words;
  s.codes = ix->d_codes; s.codes_pitch = ix->codes_pitch; s.pqM = ix->pqM; s.pqK = ix->pqK;
  s.cdist = ix->d_pq_cdist;
  if (ix->p.quantizer == SDB_QUANT_BINARY && ix->bq_fitted) {
    s.mode = 1; s.metric = ix->bq_metric; s.row_bytes = ix->bits_pitch * 8;
  } else if (ix->p.quantizer == SDB_QUANT_PRODUCT && ix->pq_fitted) {
    s.mode = 2; s.metric = ix->store_metric; s.row_bytes = ix->codes_pitch;
  } else {
    s.mode = 0; s.metric = ix->store_metric; s.row_bytes = ix->vec_pitch * 4;
  }
  return s;
}


}  // namespace sdb
