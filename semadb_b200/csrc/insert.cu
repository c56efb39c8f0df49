// insert.cu — K8: batched graph build, restating insertSinglePoint (shard/index/vamana/
// insert.go:16-68) + robustPrune (search.go:106-138) for mini-batches of new points.
//
// Per mini-batch (all on one stream, no host round trip):
//   1. beam search (search.cuh) of every new point against the current graph, emitting the
//      visited (expanded) list in expansion order — greedySearch(vec, 1, L) (insert.go:22);
//   2. prune_new_kernel, one CTA per new point A: stable sort of the visited list by
//      distance (search.go:100), robustPrune(A) with candidate rows staged in shared
//      memory, write A's adjacency row, emit (B <- A) back-edge pairs;
//   3. stable radix sort of the pairs by target B (cub), segment heads;
//   4. backedge_kernel, one CTA per distinct target B: apply its new in-edges in batch
//      order: append, or — when deg(B)+1 > R — candidates = N(B) ∪ {A} by distance from B,
//      stable sort, robustPrune(B) (insert.go:37-65).
// With a mini-batch of 1 this is exactly the reference's sequential (1-worker) schedule
// and reproduces the oracle's graph edge for edge; larger batches search a slightly stale
// snapshot, like the reference's concurrent insert workers (vamana.go:190-195).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "prune.cuh"

namespace sdb {

namespace {

// running totals behind sdb_insert_stats (the terms of the build's algorithmic-bytes figure)
enum : int { INS_POINTS = 0, INS_HOPS, INS_NDIST, INS_EDGES, INS_TARGETS, INS_PRUNES, INS_PRUNE_CAND, INS_NSTATS = 8 };

struct InsertArgs {
  StoreView s;
  uint32_t* adj; uint32_t* deg; uint8_t* dirty; uint32_t R; float alpha;
  const uint32_t* new_ids;   // [m]
  const uint32_t* vis_ids;   // [m][vis_cap] expansion order
  const float* vis_dists;
  const uint32_t* vis_len;
  uint32_t vis_cap;
  uint32_t m;
  uint32_t* pair_key;        // [m*R] target B (INVALID_ID = none)
  uint32_t* pair_val;        // [m*R] pair index (batch order)
  int staged_max;            // rows that fit in shared memory
  uint32_t* error_flag;
  const uint32_t* ndist;     // [m] distance evaluations of each point's search
  unsigned long long* stats; // running totals for sdb_insert_stats
};

__global__ void __launch_bounds__(PRUNE_THREADS) prune_new_kernel(InsertArgs a) {
  extern __shared__ __align__(16) unsigned char dyn_raw[];
  PruneShared sh;
  unsigned char* dyn = sh.carve(dyn_raw, MAX_CAND + 1);
  const uint32_t b = blockIdx.x;
  const uint32_t A = a.new_ids[b];
  uint32_t n = a.vis_len[b];
  if (n > a.vis_cap || n > MAX_CAND) {
    if (threadIdx.x == 0) atomicAdd(a.error_flag, 1u);
    n = min(min(n, a.vis_cap), uint32_t(MAX_CAND));
  }
  sh.n = int(n);
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    sh.id[i] = a.vis_ids[size_t(b) * a.vis_cap + i];
    sh.dist[i] = a.vis_dists[size_t(b) * a.vis_cap + i];
  }
  __syncthreads();
  stable_sort_by_dist(sh);
  int staged = min(int(n), a.staged_max);
  stage_rows(a.s, sh, dyn, staged);
  // the sequential robustPrune: a new point's ~80-100 candidates end the walk of search.go:106-138
  // at R accepted edges with removed candidates skipped, about a third of the pairs — 0.127 s against
  // 0.218 s for the all-pairs matrix per 1M-point build (a back-edge target's R+1: the matrix wins)
  robust_prune_cta_seq(a.s, sh, dyn, staged, A, int(a.R), a.alpha);
  const int cnt = *sh.cnt;
  for (uint32_t t = threadIdx.x; t < a.R; t += blockDim.x) {
    uint32_t e = t < uint32_t(cnt) ? sh.edges[t] : INVALID_ID;
    a.adj[size_t(A) * a.R + t] = e;
    a.pair_key[size_t(b) * a.R + t] = e;
    a.pair_val[size_t(b) * a.R + t] = b * a.R + t;
  }
  if (threadIdx.x == 0) {
    a.deg[A] = uint32_t(cnt);
    a.dirty[A] = 1;
    atomicAdd(a.stats + INS_POINTS, 1ull);
    atomicAdd(a.stats + INS_HOPS, (unsigned long long)a.vis_len[b]);
    atomicAdd(a.stats + INS_NDIST, (unsigned long long)a.ndist[b]);
    atomicAdd(a.stats + INS_EDGES, (unsigned long long)cnt);
  }
}

__global__ void segment_heads_kernel(const uint32_t* keys, uint32_t n, uint32_t* seg_start, uint32_t* seg_count) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t k = keys[i];
  if (k == INVALID_ID) return;
  if (i == 0 || keys[i - 1] != k) seg_start[atomicAdd(seg_count, 1u)] = i;
}

__global__ void iota_segments_kernel(const uint32_t* keys, uint32_t n, uint32_t* seg_start, uint32_t* seg_count) {
  if (threadIdx.x == 0) {
    uint32_t c = 0;
    for (uint32_t i = 0; i < n; ++i)
      if (keys[i] != INVALID_ID) seg_start[c++] = i;
    *seg_count = c;
  }
}

struct BackArgs {
  StoreView s;
  uint32_t* adj; uint32_t* deg; uint8_t* dirty; uint32_t R; float alpha;
  const uint32_t* new_ids;     // [m]
  const uint32_t* keys;        // sorted targets
  const uint32_t* vals;        // sorted pair indices (A index = val / R)
  uint32_t n_pairs;
  const uint32_t* seg_start;
  const uint32_t* seg_count;
  uint32_t* prune_list;        // segments whose target overflows (written by backedge_append_kernel)
  uint32_t* prune_count;
  int staged_max;
  unsigned long long* stats;
};

// nodeB.AddNeighbour(vecA) (insert.go:62): a target with room for all its new in-edges takes them
// by one warp — the common case by far (16 of 18.6 M targets of a 1 M-point build) and a 256-byte
// row update that does not need a CTA. Targets that overflow the degree bound go to the list the
// CTA kernel below works through (robustPrune(B), insert.go:44-59).
__global__ void __launch_bounds__(256) backedge_append_kernel(BackArgs a) {
  const uint32_t seg = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (seg >= *a.seg_count) return;
  const uint32_t p0 = a.seg_start[seg];
  const uint32_t B = a.keys[p0];
  // segment length: the run of equal keys from p0 (sorted by target); longer than a warp => CTA path
  const bool same = p0 + lane < a.n_pairs && a.keys[p0 + lane] == B;
  const uint32_t run = __ballot_sync(SDB_FULL, same);
  const uint32_t len = run == 0xFFFFFFFFu ? 33u : uint32_t(__ffs(~run) - 1);
  const uint32_t d = a.deg[B];
  if (len <= 32 && d + len <= a.R) {
    if (uint32_t(lane) < len) a.adj[size_t(B) * a.R + d + lane] = a.new_ids[a.vals[p0 + lane] / a.R];
    if (lane == 0) {
      a.deg[B] = d + len;
      a.dirty[B] = 1;
      atomicAdd(a.stats + INS_TARGETS, 1ull);
    }
  } else if (lane == 0) {
    a.prune_list[atomicAdd(a.prune_count, 1u)] = seg;
  }
}

__global__ void __launch_bounds__(PRUNE_THREADS) backedge_kernel(BackArgs a) {
  extern __shared__ __align__(16) unsigned char dyn_raw[];
  PruneShared sh;
  unsigned char* dyn = sh.carve(dyn_raw, MAX_CAND + 1);
  __shared__ uint32_t cur[64 + 1];
  const int lane = threadIdx.x & 31;
  const int g = lane & 7;
  const int grp = threadIdx.x >> 3;
  const uint32_t nseg = *a.prune_count;
  // The per-target chain list -> seg_start -> keys -> deg / adj is dependent global loads in front
  // of the prune: the next target's head of the chain is fetched while this one is processed.
  uint32_t nx_p0 = 0, nx_B = 0;
  if (blockIdx.x < nseg) {
    nx_p0 = a.seg_start[a.prune_list[blockIdx.x]];
    nx_B = a.keys[nx_p0];
  }
  for (uint32_t seg = blockIdx.x; seg < nseg; seg += gridDim.x) {
    const uint32_t p0 = nx_p0;
    const uint32_t B = nx_B;
    __syncthreads();
    // every thread tracks the degree in a register (a shared counter bumped by one thread
    // would race with the other warps' branch on it)
    int cur_n = int(a.deg[B]);
    for (uint32_t t = threadIdx.x; t < a.R; t += blockDim.x) cur[t] = a.adj[size_t(B) * a.R + t];
    if (seg + gridDim.x < nseg) {
      nx_p0 = a.seg_start[a.prune_list[seg + gridDim.x]];
      nx_B = a.keys[nx_p0];
    }
    __syncthreads();
    const unsigned char* xb = global_row(a.s, B);
    uint32_t p_end = p0;
    while (p_end < a.n_pairs && a.keys[p_end] == B) ++p_end;
    uint32_t p = p0;
    while (p < p_end) {
      if (cur_n + 1 <= int(a.R)) {
        // nodeB.AddNeighbour(vecA) (insert.go:62) for as many in-edges as fit, one barrier
        const uint32_t take = min(uint32_t(int(a.R) - cur_n), p_end - p);
        for (uint32_t t = threadIdx.x; t < take; t += blockDim.x) cur[cur_n + t] = a.new_ids[a.vals[p + t] / a.R];
        cur_n += int(take);
        p += take;
        __syncthreads();
        continue;
      }
      // deg(B)+1 > R: candidateSet.Add(nodeB.neighbours...), Add(vecA), distances from B, Sort,
      // robustPrune(B) (insert.go:44-59). A target that receives several new in-edges from one
      // mini-batch takes them in one prune (with one new point per mini-batch — the reference's
      // sequential schedule — this is exactly insert.go): hubs would otherwise serialise
      // hundreds of prunes in one CTA.
      const int c = int(min(p_end - p, uint32_t(MAX_CAND - cur_n)));
      const int n = cur_n + c;
      sh.n = n;
      for (int i = threadIdx.x; i < n; i += blockDim.x)
        sh.id[i] = i < cur_n ? cur[i] : a.new_ids[a.vals[p + (i - cur_n)] / a.R];
      __syncthreads();
      for (int j0 = 0; j0 < n; j0 += PRUNE_GROUPS) {
        int j = j0 + grp;
        bool act = j < n;
        if (!__any_sync(SDB_FULL, act)) continue;
        const unsigned char* yj = global_row(a.s, sh.id[act ? j : 0]);
        float d = row_dist(a.s, xb, yj, g);
        if (act && g == 0) sh.dist[j] = d;
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        atomicAdd(a.stats + INS_PRUNES, 1ull);
        atomicAdd(a.stats + INS_PRUNE_CAND, (unsigned long long)n);
      }
      stable_sort_by_dist(sh);  // candidateSet.Sort() (insert.go:58)
      int staged = min(n, a.staged_max);
      stage_rows(a.s, sh, dyn, staged);
      robust_prune_cta(a.s, sh, dyn, staged, B, int(a.R), a.alpha);
      cur_n = *sh.cnt;
      for (int t = threadIdx.x; t < cur_n; t += blockDim.x) cur[t] = sh.edges[t];
      p += uint32_t(c);
      __syncthreads();
    }
    for (uint32_t t = threadIdx.x; t < a.R; t += blockDim.x)
      a.adj[size_t(B) * a.R + t] = t < uint32_t(cur_n) ? cur[t] : INVALID_ID;
    if (threadIdx.x == 0) {
      a.deg[B] = uint32_t(cur_n);
      a.dirty[B] = 1;
      atomicAdd(a.stats + INS_TARGETS, 1ull);
    }
  }
}

// A new point none of whose out-neighbours kept the back-edge has no inbound edge at all: a
// mini-batch searches a snapshot, so mutually close new points cannot link to each other and
// robustPrune(B) may drop all of them from the few old nodes they share. One CTA per new point
// A: unlinked[b] = 1 iff no row adj[B], B in N(A), contains A.
__global__ void unlinked_flag_kernel(const uint32_t* new_ids, uint32_t m, uint32_t R, const uint32_t* adj,
                                     const uint32_t* deg, uint8_t* unlinked) {
  const uint32_t b = blockIdx.x;
  if (b >= m) return;
  const uint32_t A = new_ids[b];
  const uint32_t dA = deg[A];
  int found = 0;
  for (uint32_t j = 0; j < dA; ++j) {
    const uint32_t B = adj[size_t(A) * R + j];
    for (uint32_t t = threadIdx.x; t < R; t += blockDim.x) found |= adj[size_t(B) * R + t] == A;
  }
  found = __syncthreads_or(found);
  if (threadIdx.x == 0) unlinked[b] = (found || dA == 0) ? 0 : 1;
}

__global__ void gather_retry_kernel(const uint32_t* sel, uint32_t n, const uint32_t* src_ids, const float* src_vecs,
                                    uint32_t dim, uint32_t* dst_ids, float* dst_vecs) {
  const uint32_t i = blockIdx.x;
  if (i >= n) return;
  const uint32_t s = sel[i];
  if (threadIdx.x == 0) dst_ids[i] = src_ids[s];
  for (uint32_t t = threadIdx.x; t < dim; t += blockDim.x) dst_vecs[size_t(i) * dim + t] = src_vecs[size_t(s) * dim + t];
}

// debug aid (SDB_DEBUG_INSERT=1): adjacency rows must hold deg valid ids then padding
__global__ void check_rows_kernel(const uint32_t* adj, const uint32_t* deg, const uint8_t* exists, uint32_t rows,
                                  uint32_t R, uint32_t* report) {
  uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= rows || !exists[id]) return;
  uint32_t d = deg[id];
  bool bad = d > R;
  for (uint32_t t = 0; t < R && !bad; ++t) {
    uint32_t e = adj[size_t(id) * R + t];
    if (t < d) bad = (e == INVALID_ID) || e >= rows || !exists[e] || e == id;
    else bad = e != INVALID_ID;
  }
  if (bad && atomicAdd(report, 1u) == 0) { report[1] = id; report[2] = d; }
}

}  // namespace

int insert_batch_locked(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors, bool reinsert,
                        bool vectors_on_device) {
  // classify like insertUpdateDelete (vamana.go:149-185): only fresh inserts are handled here
  std::vector<uint32_t> h32(n);
  uint64_t mx = 0;
  for (uint64_t i = 0; i < n; ++i) {
    if (ids[i] == START_ID) return fail(SDB_ERR_RESERVED_ID, "cannot modify point with start id: 1");
    if (ids[i] == 0) return fail(SDB_ERR_RESERVED_ID, "invalid point id: 0");
    if (ids[i] >= (uint64_t(1) << 31) - 1) return fail(SDB_ERR_INVALID, "node id too large for a device index");
    if (!reinsert && ids[i] < ix->rows && ix->h_exists[ids[i]]) return fail(SDB_ERR_STATE, "point already exists (updates go through sdb_insert_update_delete): " + std::to_string(ids[i]));
    mx = std::max(mx, ids[i]);
    h32[i] = uint32_t(ids[i]);
  }
  if (ix->rows <= START_ID || !ix->h_exists[START_ID]) return fail(SDB_ERR_STATE, "failed to get start point");
  int rc = index_reserve_locked(ix, mx);
  if (rc) return rc;
  cudaStream_t st = ix->stream;
  if (!ix->d_ins_stats) {
    SDB_CUDA(cudaMalloc(reinterpret_cast<void**>(&ix->d_ins_stats), INS_NSTATS * sizeof(unsigned long long)));
    SDB_CUDA(cudaMemsetAsync(ix->d_ins_stats, 0, INS_NSTATS * sizeof(unsigned long long), st));
  }
  const uint32_t R = ix->p.degree_bound, L = ix->p.search_size, dim = ix->p.dim;
  const uint32_t vis_cap = MAX_CAND;
  // updated points are re-inserted one by one (vamana.go:249-253) unless the index is relaxed
  const bool one_by_one = reinsert && !ix->p.relaxed;
  // mini-batch schedule: explicit (sdb_insert_config) or by the width of the distance rows (index.cuh)
  const bool narrow_rows = ix->distance_row_bytes() <= 512;
  const uint32_t cfg_max_batch = ix->ins_max_batch ? ix->ins_max_batch : (narrow_rows ? 32768u : 16384u);
  const uint32_t cfg_growth_div = ix->ins_growth_div ? ix->ins_growth_div : (narrow_rows ? 8u : 16u);
  const uint32_t max_batch = one_by_one ? 1u : std::max<uint32_t>(1, std::max(cfg_max_batch, ix->ins_min_batch));

  // device copies of ids and vectors for the whole call (chunked to bound staging)
  const uint64_t chunk_pts = std::max<uint64_t>(max_batch, (uint64_t(512) << 20) / (dim * sizeof(float)));
  sdb::DevBuf<uint32_t> d_ids;
  sdb::DevBuf<float> d_vecs;
  sdb::DevBuf<uint32_t> d_pair_key, d_pair_val, d_pair_key2, d_pair_val2, d_seg, d_misc, d_plist;
  sdb::DevBuf<unsigned char> d_cubtmp;
  sdb::DevBuf<uint8_t> d_unflag;
  sdb::DevBuf<uint32_t> d_sel, d_retry_ids[2];
  sdb::DevBuf<float> d_retry_vecs[2];
  auto release_all = [&]() {
    d_ids.release(); d_vecs.release(); d_pair_key.release(); d_pair_val.release(); d_pair_key2.release();
    d_pair_val2.release(); d_seg.release(); d_misc.release(); d_plist.release(); d_cubtmp.release(); d_unflag.release(); d_sel.release();
    for (int i = 0; i < 2; ++i) { d_retry_ids[i].release(); d_retry_vecs[i].release(); }
  };
#define INS_CHECK(expr)            \
  do {                             \
    int _rc = (expr);              \
    if (_rc) { release_all(); return _rc; } \
  } while (0)
#define INS_CUDA(expr)                                              \
  do {                                                              \
    cudaError_t _e = (expr);                                        \
    if (_e != cudaSuccess) { release_all(); return cuda_fail(_e, #expr); } \
  } while (0)

  const size_t max_pairs = size_t(max_batch) * R;
  INS_CHECK(d_pair_key.ensure(max_pairs));
  INS_CHECK(d_pair_val.ensure(max_pairs));
  INS_CHECK(d_pair_key2.ensure(max_pairs));
  INS_CHECK(d_pair_val2.ensure(max_pairs));
  INS_CHECK(d_seg.ensure(max_pairs));
  INS_CHECK(d_plist.ensure(max_pairs));
  INS_CHECK(d_misc.ensure(8));
  INS_CHECK(ix->d_vis_ids.ensure(size_t(max_batch) * vis_cap));
  INS_CHECK(ix->d_vis_d.ensure(size_t(max_batch) * vis_cap));
  INS_CHECK(ix->d_vis_len.ensure(max_batch));
  INS_CHECK(ix->d_oid.ensure(max_batch));
  INS_CHECK(ix->d_od.ensure(max_batch));
  INS_CHECK(ix->d_oc.ensure(max_batch));
  size_t cub_bytes = 0, sel_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, d_pair_key.p, d_pair_key2.p, d_pair_val.p, d_pair_val2.p, int(max_pairs), 0, 32, st);
  // repair pass for new points left without an inbound edge (batched schedule only)
  const bool repair = max_batch > 1;
  if (repair) {
    INS_CHECK(d_unflag.ensure(max_batch));
    INS_CHECK(d_sel.ensure(max_batch));
    for (int i = 0; i < 2; ++i) {
      INS_CHECK(d_retry_ids[i].ensure(max_batch));
      INS_CHECK(d_retry_vecs[i].ensure(size_t(max_batch) * dim));
    }
    cub::DeviceSelect::Flagged(nullptr, sel_bytes, thrust::counting_iterator<uint32_t>(0), d_unflag.p, d_sel.p, d_misc.p,
                               int(max_batch), st);
  }
  INS_CHECK(d_cubtmp.ensure(std::max(cub_bytes, sel_bytes) + 16));
  INS_CUDA(cudaMemsetAsync(d_misc.p, 0, 8 * sizeof(uint32_t), st));
  uint32_t* d_err = d_misc.p + 1;
  uint32_t* d_segcount = d_misc.p;

  // shared memory budget for staged candidate rows
  size_t static_smem = PruneShared::bytes(MAX_CAND + 1) + 512;
  cudaFuncAttributes fa;
  INS_CUDA(cudaFuncGetAttributes(&fa, prune_new_kernel));
  static_smem = std::max(static_smem, fa.sharedSizeBytes);
  INS_CUDA(cudaFuncGetAttributes(&fa, backedge_kernel));
  static_smem = std::max(static_smem, fa.sharedSizeBytes);

  const bool debug = getenv("SDB_DEBUG_INSERT") != nullptr;
  uint64_t inserted_before = ix->count > 0 ? ix->count - 1 : 0;  // user points already in the graph
  for (uint64_t c0 = 0; c0 < n; c0 += chunk_pts) {
    const uint64_t cn = std::min(chunk_pts, n - c0);
    INS_CHECK(d_ids.ensure(cn));
    INS_CUDA(cudaMemcpyAsync(d_ids.p, h32.data() + c0, cn * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    const float* chunk_vecs = vectors + c0 * dim;  // device-resident input is used where it lies
    if (!vectors_on_device) {
      INS_CHECK(d_vecs.ensure(size_t(cn) * dim));
      INS_CUDA(cudaMemcpyAsync(d_vecs.p, vectors + c0 * dim, size_t(cn) * dim * sizeof(float), cudaMemcpyHostToDevice, st));
      chunk_vecs = d_vecs.p;
    }
    // vecStore.Set for the chunk (insert.go:17): rows become visible, nothing points at them yet
    INS_CHECK(set_rows_device(ix, uint32_t(cn), d_ids.p, chunk_vecs, st));
    StoreView view = make_view(ix);
    // rows staged per CTA: aim for >= 2 CTAs/SM
    size_t budget = std::min<size_t>(ix->smem_optin, size_t(100) << 10);
    size_t dyn_budget = budget > static_smem ? budget - static_smem : 0;
    int staged_max = int(std::min<size_t>(MAX_CAND, dyn_budget / view.row_bytes));
    // ... but no more than 32 KB of rows (at least 32 rows if they fit): a back-edge prune has 65
    // candidates, and residency beats staging the long tail of a visited list — 1M x 128 builds in
    // 1.12 s with 64 staged rows, 1.19 s with 96, 1.26 s with 128, 1.35 s with 186 (profiles/r01_ab_insert.txt)
    staged_max = std::min(staged_max, std::max(int((size_t(32) << 10) / view.row_bytes), std::min(32, staged_max)));
    // ... and the R+1 candidates of a back-edge prune all of them when that costs one more row (dim 128:
    // 65 x 512 B): the all-pairs pass then runs on shared memory only
    if (staged_max == int(R) && size_t(R + 1) * view.row_bytes <= dyn_budget) staged_max = int(R) + 1;
    size_t dyn_smem = PruneShared::bytes(MAX_CAND + 1) + size_t(staged_max) * view.row_bytes;
    INS_CUDA(cudaFuncSetAttribute(prune_new_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(dyn_smem)));
    INS_CUDA(cudaFuncSetAttribute(backedge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(dyn_smem)));

    // SDB_DEBUG_INSERT_STATS: per-phase wall time (synchronises after every phase)
    const bool timing = getenv("SDB_DEBUG_INSERT_STATS") != nullptr;
    double t_phase[4] = {0, 0, 0, 0};
    auto tick = [&](int phase, std::chrono::steady_clock::time_point& t0) {
      if (!timing) return;
      cudaStreamSynchronize(st);
      auto t1 = std::chrono::steady_clock::now();
      t_phase[phase] += std::chrono::duration<double>(t1 - t0).count();
      t0 = t1;
    };
    // one mini-batch: search, prune, group back-edge pairs, apply them
    auto run_batch = [&](const uint32_t* b_ids, const float* b_vecs, uint32_t m, uint64_t at) -> int {
      auto t0 = std::chrono::steady_clock::now();
      if (timing) cudaStreamSynchronize(st);
      // 1. greedySearch(vec, 1, L) with the visited list
      INS_CHECK(launch_search(ix, m, b_vecs, 1, L, ix->d_oid.p, ix->d_od.p, ix->d_oc.p, ix->d_vis_ids.p, ix->d_vis_d.p,
                              ix->d_vis_len.p, vis_cap, nullptr, st));
      tick(0, t0);
      // 2. robustPrune(A) + emit back-edge pairs
      InsertArgs ia{};
      ia.s = view; ia.adj = ix->d_adj; ia.deg = ix->d_deg; ia.dirty = ix->d_dirty; ia.R = R; ia.alpha = ix->p.alpha;
      ia.new_ids = b_ids; ia.vis_ids = ix->d_vis_ids.p; ia.vis_dists = ix->d_vis_d.p; ia.vis_len = ix->d_vis_len.p;
      ia.vis_cap = vis_cap; ia.m = m; ia.pair_key = d_pair_key.p; ia.pair_val = d_pair_val.p;
      ia.staged_max = staged_max; ia.error_flag = d_err;
      ia.ndist = ix->d_ndist.p; ia.stats = ix->d_ins_stats;
      prune_new_kernel<<<m, PRUNE_THREADS, dyn_smem, st>>>(ia);
      ix->launches++;
      INS_CUDA(cudaGetLastError());
      tick(1, t0);
      // 3. group pairs by target (stable => batch order within a target)
      const uint32_t np = m * R;
      const uint32_t* skeys = d_pair_key.p;
      const uint32_t* svals = d_pair_val.p;
      if (m > 1) {
        size_t tb = cub_bytes;
        INS_CUDA(cub::DeviceRadixSort::SortPairs(d_cubtmp.p, tb, d_pair_key.p, d_pair_key2.p, d_pair_val.p, d_pair_val2.p, int(np), 0, 32, st));
        ix->launches += 4;
        skeys = d_pair_key2.p;
        svals = d_pair_val2.p;
      }
      INS_CUDA(cudaMemsetAsync(d_segcount, 0, sizeof(uint32_t), st));
      if (m > 1) {
        segment_heads_kernel<<<(np + 255) / 256, 256, 0, st>>>(skeys, np, d_seg.p, d_segcount);
        ix->launches++;
        INS_CUDA(cudaGetLastError());
      }
      tick(2, t0);
      // 4. back-edges
      BackArgs ba{};
      ba.s = view; ba.adj = ix->d_adj; ba.deg = ix->d_deg; ba.dirty = ix->d_dirty; ba.R = R; ba.alpha = ix->p.alpha;
      ba.new_ids = b_ids; ba.keys = skeys; ba.vals = svals; ba.n_pairs = np; ba.seg_start = d_seg.p;
      ba.seg_count = d_segcount; ba.staged_max = staged_max; ba.stats = ix->d_ins_stats;
      ba.prune_list = d_plist.p; ba.prune_count = d_misc.p + 2;
      if (m == 1) {
        // a single new point: every target is its own segment, in edge order — no sort needed
        iota_segments_kernel<<<1, 64, 0, st>>>(skeys, np, d_seg.p, d_segcount);
        ix->launches++;
      }
      INS_CUDA(cudaMemsetAsync(d_misc.p + 2, 0, sizeof(uint32_t), st));
      backedge_append_kernel<<<(np + 7) / 8, 256, 0, st>>>(ba);  // np >= number of segments
      uint32_t grid = std::min<uint32_t>(np, uint32_t(ix->sm_count) * 8);
      backedge_kernel<<<grid, PRUNE_THREADS, dyn_smem, st>>>(ba);
      ix->launches += 2;
      INS_CUDA(cudaGetLastError());
      tick(3, t0);
      if (debug) {
        INS_CUDA(cudaMemsetAsync(d_misc.p + 4, 0, 3 * sizeof(uint32_t), st));
        check_rows_kernel<<<(ix->rows + 255) / 256, 256, 0, st>>>(ix->d_adj, ix->d_deg, ix->d_exists, ix->rows, R, d_misc.p + 4);
        uint32_t rep[3];
        INS_CUDA(cudaMemcpyAsync(rep, d_misc.p + 4, sizeof(rep), cudaMemcpyDeviceToHost, st));
        INS_CUDA(cudaStreamSynchronize(st));
        if (rep[0]) {
          release_all();
          return fail(SDB_ERR_INTERNAL, "insert debug: " + std::to_string(rep[0]) + " inconsistent rows after a batch of " + std::to_string(m) + " at offset " + std::to_string(at) + ", first node " + std::to_string(rep[1]) + " deg " + std::to_string(rep[2]));
        }
      }
      return SDB_OK;
    };
    // how many of a mini-batch's points ended up without any inbound edge (ascending list in d_sel)
    auto count_unlinked = [&](const uint32_t* b_ids, uint32_t m, uint32_t* out) -> int {
      unlinked_flag_kernel<<<m, 64, 0, st>>>(b_ids, m, R, ix->d_adj, ix->d_deg, d_unflag.p);
      ix->launches++;
      INS_CUDA(cudaGetLastError());
      size_t tb = sel_bytes;
      INS_CUDA(cub::DeviceSelect::Flagged(d_cubtmp.p, tb, thrust::counting_iterator<uint32_t>(0), d_unflag.p, d_sel.p,
                                          d_misc.p + 3, int(m), st));
      ix->launches++;
      INS_CUDA(cudaMemcpyAsync(out, d_misc.p + 3, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      INS_CUDA(cudaStreamSynchronize(st));
      return SDB_OK;
    };

    uint64_t done = 0;
    uint64_t stat_unlinked[2] = {0, 0};
    while (done < cn) {
      uint64_t total_in = inserted_before + c0 + done;
      uint64_t want = std::max<uint64_t>(ix->ins_min_batch, total_in / cfg_growth_div);
      uint32_t m = uint32_t(std::min<uint64_t>(std::min<uint64_t>(want, max_batch), cn - done));
      if (m == 0) m = 1;
      const uint32_t* b_ids = d_ids.p + done;
      const float* b_vecs = chunk_vecs + done * dim;
      INS_CHECK(run_batch(b_ids, b_vecs, m, c0 + done));
      if (repair && m > 1) {
        // Re-insert the points nobody points at, in quarter-size mini-batches: mutually close
        // new points then find each other. At most two rounds — a point every neighbour prunes
        // away again is an orphan the sequential schedule produces too (robustPrune(B) drops it).
        const uint32_t* cur_ids = b_ids;
        const float* cur_vecs = b_vecs;
        uint32_t cur_m = m;
        for (int round = 0; cur_m > 1 && round < 2; ++round) {
          uint32_t un = 0;
          INS_CHECK(count_unlinked(cur_ids, cur_m, &un));
          stat_unlinked[round] += un;
          if (un == 0) break;
          const int w = round & 1;
          gather_retry_kernel<<<un, 128, 0, st>>>(d_sel.p, un, cur_ids, cur_vecs, dim, d_retry_ids[w].p, d_retry_vecs[w].p);
          ix->launches++;
          INS_CUDA(cudaGetLastError());
          const uint32_t sub = std::max<uint32_t>(1, std::min<uint32_t>(un, cur_m) / 4);
          for (uint32_t off = 0; off < un; off += sub)
            INS_CHECK(run_batch(d_retry_ids[w].p + off, d_retry_vecs[w].p + size_t(off) * dim, std::min(sub, un - off), c0 + done));
          cur_ids = d_retry_ids[w].p;
          cur_vecs = d_retry_vecs[w].p;
          cur_m = sub > 1 ? un : 1;
        }
      }
      done += m;
    }
    if (debug || getenv("SDB_DEBUG_INSERT_STATS"))
      fprintf(stderr, "[sdb] insert chunk of %llu: %llu points without an inbound edge after their mini-batch, %llu after one repair round\n",
              (unsigned long long)cn, (unsigned long long)stat_unlinked[0], (unsigned long long)stat_unlinked[1]);
    if (timing)
      fprintf(stderr, "[sdb] insert phases: search %.3fs, prune_new %.3fs, pair sort %.3fs, backedge %.3fs\n", t_phase[0],
              t_phase[1], t_phase[2], t_phase[3]);
    INS_CUDA(cudaStreamSynchronize(st));
  }
  uint32_t h_misc[2] = {0, 0};
  INS_CUDA(cudaMemcpy(h_misc, d_misc.p, sizeof(h_misc), cudaMemcpyDeviceToHost));
  release_all();
#undef INS_CHECK
#undef INS_CUDA
  for (uint64_t i = 0; i < n; ++i) {
    if (!ix->h_exists[h32[i]]) {
      ix->h_exists[h32[i]] = 1;
      ix->count++;
    }
    if (h32[i] > ix->max_node_id) ix->max_node_id = h32[i];
  }
  // A visited list longer than MAX_CAND was cut to its first MAX_CAND expansions before robustPrune
  // (the reference's list is unbounded; never observed below 6M-point hamming shards at 512). The
  // graph is valid and the index state is committed, so this is counted, not an error: failing
  // here would leave host and device state apart (the points exist on the device).
  ix->insert_truncated += h_misc[1];
  return SDB_OK;
}

}  // namespace sdb
