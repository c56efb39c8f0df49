// flat.cu — K5: brute-force scan + top-k, restating IndexFlat.Search
// (shard/index/flat/flat.go:76-132) for a batch of queries.
//
// The reference scans every stored point (Go-map order), keeps a Limit-sized sorted
// slice, skips when full and d >= worst (flat.go:99) and bubbles while strictly smaller
// (flat.go:117). With ascending-id iteration that is exactly "top-k by (distance asc,
// id asc)", which decomposes over point chunks: each (query, chunk) keeps a local top-k,
// a second kernel merges the chunks in chunk order with the same rule.
// Distances use the reference's exact f32 summation order (common.cuh), one thread per
// (query, point) pair; the query tile sits transposed in shared memory (conflict-free),
// the point rows are read through a broadcast shared tile of up to FP rows (fewer when FP rows
// of a wide store do not fit next to the query tile).
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "index.cuh"

namespace sdb {

namespace {

constexpr int FQ = 128;      // queries per CTA (one per thread)
constexpr int FP = 16;       // points per shared tile (at most; FlatArgs::tile_pts)
constexpr int FMAXK = 75;    // models/search.go:329

struct FlatArgs {
  const float* vec; uint32_t vec_pitch;
  const uint64_t* bits; uint32_t bits_pitch; uint32_t words;
  const uint8_t* codes; uint32_t codes_pitch;
  const float* adc; uint32_t pqM, pqK;
  const float* bq_thr; int bit_metric;
  const uint8_t* exists;
  const uint32_t* filter_bits;
  const float* queries;
  uint32_t dim, B, k;
  uint32_t first_id, end_id;  // scan [first_id, end_id)
  uint32_t chunk;             // points per chunk (a multiple of tile_pts)
  uint32_t tile_pts;          // f32 rows per shared point tile, 1..FP
  uint32_t n_chunks;
  uint32_t* part_ids;         // [B][n_chunks][k]
  float* part_d;
  uint32_t* part_cnt;         // [B][n_chunks]
  // query list on the device (launch_flat_exact_list): slot s < min(*qcount, B) is batch row
  // qlist[s]; the split into chunks is derived from the count on the device
  const uint32_t* qlist;
  const uint32_t* qcount;
  uint32_t sm_count;
};

struct FlatSplit {
  uint32_t n_chunks, chunk;
};

// (query block x point chunk) split of a scan of nq queries over npts points: about 4 CTAs per SM,
// chunks of at least 256 points, whole shared point tiles. The host (launch_flat_exact) and the
// device (a list whose count only the device knows) derive the same split from the same count.
__host__ __device__ inline FlatSplit flat_split(uint32_t nq, uint32_t npts, uint32_t tile_pts, uint32_t sm_count) {
  const uint32_t qblocks = (nq + FQ - 1) / FQ;
  uint32_t want = (sm_count * 4 + qblocks - 1) / qblocks;
  if (want < 1) want = 1;
  uint32_t max_chunks = (npts + 255) / 256;
  if (max_chunks < 1) max_chunks = 1;
  uint32_t n = want < max_chunks ? want : max_chunks;
  if (n > 1024) n = 1024;
  uint32_t chunk = (npts + n - 1) / n;
  if (chunk == 0) chunk = 1;
  chunk = (chunk + tile_pts - 1) / tile_pts * tile_pts;
  return {npts == 0 ? 1 : (npts + chunk - 1) / chunk, chunk};
}

struct TopK {
  float d[FMAXK];
  uint32_t id[FMAXK];
  int n = 0;
  // flat.go:99-119
  __device__ __forceinline__ void offer(uint32_t pid, float dist, int k) {
    if (n == k && dist >= d[n - 1]) return;
    int i;
    if (n < k) i = n++;
    else i = n - 1;
    while (i > 0 && dist < d[i - 1]) {
      d[i] = d[i - 1];
      id[i] = id[i - 1];
      --i;
    }
    d[i] = dist;
    id[i] = pid;
  }
};

// One work item: query block qb (slots qb*FQ .. of nq) against point chunk c.
// mode 0: f32 rows (METRIC template), 1: bits, 2: PQ codes via ADC table
// QSMEM: the query tile fits transposed in shared memory; otherwise (large dim) each thread
// streams its query row through L1.
template <int MODE, int METRIC, bool QSMEM, bool LIST>
__device__ __forceinline__ void scan_item(const FlatArgs& a, unsigned char* sm, uint32_t qb, uint32_t c, uint32_t nq,
                                          uint32_t chunk, uint32_t n_chunks) {
  const int tid = threadIdx.x;
  const uint32_t slot = qb * FQ + tid;
  const bool qvalid = slot < nq;
  const uint32_t q = qvalid ? (LIST ? a.qlist[slot] : slot) : 0;  // batch row
  uint32_t lo = a.first_id + c * chunk;
  uint32_t hi = min(a.end_id, lo + chunk);
  TopK top;

  if (MODE == 0) {
    // shared: qT[dim][FQ] floats, pt[FP][dim] floats
    float* qT = reinterpret_cast<float*>(sm);
    float* pt = qT + (QSMEM ? size_t(a.dim) * FQ : 0);
    const float* qrow = a.queries + size_t(q) * a.dim;
    if (QSMEM) {
      for (uint32_t i = tid; i < a.dim * FQ; i += FQ) {
        uint32_t qq = i / a.dim, dd = i % a.dim;  // coalesced read of query rows
        uint32_t gs = qb * FQ + qq;
        qT[dd * FQ + qq] = gs < nq ? a.queries[size_t(LIST ? a.qlist[gs] : gs) * a.dim + dd] : 0.0f;
      }
    }
    auto qat = [&](uint32_t i) -> float { return QSMEM ? qT[i * FQ + tid] : __ldg(qrow + i); };
    __syncthreads();
    constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
    const int blocks = a.dim >> 5;
    for (uint32_t p0 = lo; p0 < hi; p0 += a.tile_pts) {
      uint32_t np = min(a.tile_pts, hi - p0);
      for (uint32_t i = tid; i < np * a.dim; i += FQ) {
        uint32_t pp = i / a.dim, dd = i % a.dim;
        pt[pp * a.dim + dd] = a.vec[size_t(p0 + pp) * a.vec_pitch + dd];
      }
      __syncthreads();
      for (uint32_t pp = 0; pp < np; ++pp) {
        uint32_t pid = p0 + pp;
        bool ok = a.exists[pid] && (!a.filter_bits || ((a.filter_bits[pid >> 5] >> (pid & 31)) & 1u));
        if (!ok) continue;  // block-uniform
        const float* y = pt + pp * a.dim;
        float dist;
        if (METRIC == METRIC_HAVERSINE) {
          float xq[2] = {qat(0), qat(1)};
          dist = haversine_thread(xq, y);
        } else {
          float acc[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = 0.0f;
          for (int t = 0; t < blocks; ++t) {
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] = tail_accum<L2>(qat(t * 32 + i), y[t * 32 + i], acc[i]);
          }
          float tail = 0.0f;
          for (uint32_t i = blocks << 5; i < a.dim; ++i) tail = tail_accum<L2>(qat(i), y[i], tail);
          float w[4];
#pragma unroll
          for (int l = 0; l < 4; ++l) {
            float v0 = __fadd_rn(__fadd_rn(__fadd_rn(acc[l], acc[8 + l]), acc[16 + l]), acc[24 + l]);
            float v1 = __fadd_rn(__fadd_rn(__fadd_rn(acc[4 + l], acc[12 + l]), acc[20 + l]), acc[28 + l]);
            w[l] = __fadd_rn(v0, v1);
          }
          w[0] = __fadd_rn(w[0], tail);
          dist = metric_epilogue<METRIC>(__fadd_rn(__fadd_rn(w[0], w[1]), __fadd_rn(w[2], w[3])));
        }
        if (qvalid) top.offer(pid, dist, a.k);
      }
      __syncthreads();
    }
  } else if (MODE == 1) {
    // shared: qb[FQ][words] (thread-private rows, stride words+1 to spread banks)
    uint64_t* qb = reinterpret_cast<uint64_t*>(sm) + size_t(tid) * (a.words | 1);
    if (qvalid) {
      const float* qv = a.queries + size_t(q) * a.dim;
      for (uint32_t w = 0; w < a.words; ++w) {
        uint64_t word = 0;
        for (uint32_t b = 0; b < 64; ++b) {
          uint32_t i = w * 64 + b;
          if (i < a.dim && qv[i] > a.bq_thr[i]) word |= uint64_t(1) << b;
        }
        qb[w] = word;
      }
    }
    for (uint32_t pid = lo; pid < hi; ++pid) {
      bool ok = a.exists[pid] && (!a.filter_bits || ((a.filter_bits[pid >> 5] >> (pid & 31)) & 1u));
      if (!ok || !qvalid) continue;
      const uint64_t* y = a.bits + size_t(pid) * a.bits_pitch;
      int x = 0, u = 0;
      for (uint32_t w = 0; w < a.words; ++w) {
        uint64_t yw = __ldg(y + w);
        if (a.bit_metric == METRIC_JACCARD) { x += __popcll(qb[w] & yw); u += __popcll(qb[w] | yw); }
        else x += __popcll(qb[w] ^ yw);
      }
      top.offer(pid, bits_finish(a.bit_metric, x, u), a.k);
    }
  } else {
    const float* table = a.adc + size_t(q) * a.pqM * a.pqK;
    for (uint32_t pid = lo; pid < hi; ++pid) {
      bool ok = a.exists[pid] && (!a.filter_bits || ((a.filter_bits[pid >> 5] >> (pid & 31)) & 1u));
      if (!ok || !qvalid) continue;
      const uint8_t* code = a.codes + size_t(pid) * a.codes_pitch;
      float d = 0.0f;
      for (uint32_t i = 0; i < a.pqM; ++i) d = __fadd_rn(d, __ldg(table + i * a.pqK + __ldg(code + i)));
      top.offer(pid, d, a.k);
    }
  }
  if (qvalid) {
    size_t o = (size_t(slot) * n_chunks + c) * a.k;
    for (int i = 0; i < top.n; ++i) { a.part_ids[o + i] = top.id[i]; a.part_d[o + i] = top.d[i]; }
    a.part_cnt[size_t(slot) * n_chunks + c] = top.n;
  }
}

// LIST = false: one work item per CTA, grid (query blocks, chunks) split on the host.
// LIST = true: a fixed grid loops over the items of the split of min(*qcount, B) listed queries.
template <int MODE, int METRIC, bool QSMEM, bool LIST>
__global__ void __launch_bounds__(FQ) flat_scan_kernel(FlatArgs a) {
  extern __shared__ __align__(16) unsigned char sm[];
  if (!LIST) {
    scan_item<MODE, METRIC, QSMEM, false>(a, sm, blockIdx.x, blockIdx.y, a.B, a.chunk, a.n_chunks);
    return;
  }
  const uint32_t nq = min(*a.qcount, a.B);
  if (nq == 0) return;
  const FlatSplit s = flat_split(nq, a.end_id - a.first_id, a.tile_pts, a.sm_count);
  const uint32_t items = (nq + FQ - 1) / FQ * s.n_chunks;
  for (uint32_t w = blockIdx.x; w < items; w += gridDim.x) {
    scan_item<MODE, METRIC, QSMEM, true>(a, sm, w / s.n_chunks, w % s.n_chunks, nq, s.chunk, s.n_chunks);
    __syncthreads();  // the next item refills the shared query tile
  }
}

// merges slot q's chunk lists in chunk order (= ascending id order) into output row q, or, with a
// query list, into row qlist[q]
__global__ void flat_merge_kernel(FlatArgs a, uint64_t* out_ids, float* out_d, uint32_t* out_cnt) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t nq = a.qlist ? min(*a.qcount, a.B) : a.B;
  if (s >= nq) return;
  const uint32_t n_chunks = a.qlist ? flat_split(nq, a.end_id - a.first_id, a.tile_pts, a.sm_count).n_chunks : a.n_chunks;
  const uint32_t q = a.qlist ? a.qlist[s] : s, k = a.k;
  TopK top;
  for (uint32_t c = 0; c < n_chunks; ++c) {
    size_t o = (size_t(s) * n_chunks + c) * k;
    uint32_t n = a.part_cnt[size_t(s) * n_chunks + c];
    for (uint32_t i = 0; i < n; ++i) top.offer(a.part_ids[o + i], a.part_d[o + i], k);
  }
  for (uint32_t i = 0; i < k; ++i) {
    out_ids[size_t(q) * k + i] = i < uint32_t(top.n) ? uint64_t(top.id[i]) : 0;
    out_d[size_t(q) * k + i] = i < uint32_t(top.n) ? top.d[i] : __int_as_float(0x7f800000);
  }
  out_cnt[q] = top.n;
}

template <int MODE, int METRIC, bool QSMEM = true, bool LIST = false>
int launch_scan(sdb_index* ix, const FlatArgs& a, size_t smem, uint32_t list_grid, cudaStream_t stream) {
  auto kern = flat_scan_kernel<MODE, METRIC, QSMEM, LIST>;
  if (smem > 48 * 1024) SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  dim3 grid = LIST ? dim3(list_grid) : dim3((a.B + FQ - 1) / FQ, a.n_chunks);
  kern<<<grid, FQ, smem, stream>>>(a);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

// store and query fields of a scan over [first_id, end_id), and the rows of its shared point tile
int flat_args(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_filter_bits,
              uint32_t first_id, uint32_t end_id, FlatArgs& a, bool& qsmem) {
  a = FlatArgs{};
  a.vec = ix->d_vec; a.vec_pitch = ix->vec_pitch;
  a.bits = ix->d_bits; a.bits_pitch = ix->bits_pitch; a.words = ix->words;
  a.codes = ix->d_codes; a.codes_pitch = ix->codes_pitch;
  a.pqM = ix->pqM; a.pqK = ix->pqK;
  a.bq_thr = ix->d_bq_thr; a.bit_metric = ix->bq_metric;
  a.exists = ix->d_exists;
  a.filter_bits = d_filter_bits;
  a.queries = d_queries;
  a.dim = ix->p.dim; a.B = B; a.k = k;
  a.first_id = first_id;  // from 2: the start node is not a flat-index point
  a.end_id = std::min(std::max(end_id, first_id), std::max<uint32_t>(2, ix->max_node_id + 1));
  a.sm_count = uint32_t(ix->sm_count);
  // f32 rows: the query tile in shared memory when it fits next to FP point rows; otherwise the
  // queries are read through L1 and the point tile takes as many rows as fit (14 at dim 4096)
  const size_t row_bytes = size_t(a.dim) * sizeof(float);
  qsmem = (size_t(FQ) + FP) * row_bytes <= ix->smem_optin;
  a.tile_pts = uint32_t(std::min<size_t>(FP, ix->smem_optin / row_bytes));
  if (a.tile_pts == 0) return fail(SDB_ERR_INVALID, "flat scan: one vector does not fit in shared memory");
  return SDB_OK;
}

}  // namespace

int launch_flat(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_filter_bits,
                uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, cudaStream_t stream) {
  // f32 stores above a few sample sizes: tensor-core candidate pass + exact re-score (flat_tc.cu),
  // bit-identical to the exact scan below
  if (flat_tc_eligible(ix, k, d_filter_bits != nullptr))
    return launch_flat_tc(ix, B, d_queries, k, d_out_ids, d_out_dists, d_out_counts, stream);
  ix->flat_last_path = 0;
  ix->flat_stats_pending = false;
  return launch_flat_exact(ix, B, d_queries, k, d_filter_bits, d_out_ids, d_out_dists, d_out_counts, stream, 2,
                           std::max<uint32_t>(2, ix->max_node_id + 1));
}

// Unfiltered flat search of device-resident queries into device-resident outputs, all enqueued on
// `stream` with no host synchronisation (once a call of the same shape has run: growing scratch
// frees and allocates device memory). The host entry and both device entries run through it.
int flat_device_locked(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint64_t* d_out_ids, float* d_out_dists,
                       uint32_t* d_out_counts, cudaStream_t stream) {
  ix->flat_last_gathered = ix->flat_last_scanned = 0;
  ix->flat_last_pairs = 0;
  return launch_flat(ix, B, d_queries, k, nullptr, d_out_ids, d_out_dists, d_out_counts, stream);
}

int launch_flat_exact(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_filter_bits,
                      uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, cudaStream_t stream,
                      uint32_t first_id, uint32_t end_id) {
  FlatArgs a;
  bool qsmem;
  int rc;
  if ((rc = flat_args(ix, B, d_queries, k, d_filter_bits, first_id, end_id, a, qsmem))) return rc;
  const uint32_t npts = a.end_id - a.first_id;
  const FlatSplit sp = flat_split(B, npts, a.tile_pts, a.sm_count);
  a.n_chunks = sp.n_chunks;
  a.chunk = sp.chunk;
  size_t parts = size_t(B) * a.n_chunks * k;
  if ((rc = ix->d_tmp32.ensure(parts + size_t(B) * a.n_chunks))) return rc;
  if ((rc = ix->d_tmpf.ensure(parts))) return rc;
  a.part_ids = ix->d_tmp32.p;
  a.part_cnt = ix->d_tmp32.p + parts;
  a.part_d = ix->d_tmpf.p;

  const size_t row_bytes = size_t(a.dim) * sizeof(float);
  if (ix->p.quantizer == SDB_QUANT_BINARY && ix->bq_fitted) {
    size_t smem = size_t(FQ) * (a.words | 1) * 8;
    if ((rc = launch_scan<1, 0>(ix, a, smem, 0, stream))) return rc;
  } else if (ix->p.quantizer == SDB_QUANT_PRODUCT && ix->pq_fitted) {
    if ((rc = ix->d_adc.ensure(size_t(B) * ix->pqM * ix->pqK))) return rc;
    if ((rc = launch_adc_tables(ix, B, d_queries, ix->d_adc.p, stream))) return rc;
    a.adc = ix->d_adc.p;
    if ((rc = launch_scan<2, 0>(ix, a, 0, 0, stream))) return rc;
  } else {
    const size_t smem = ((qsmem ? size_t(FQ) : 0) + a.tile_pts) * row_bytes;
    switch (ix->store_metric) {
      case SDB_METRIC_EUCLIDEAN:
        rc = qsmem ? launch_scan<0, METRIC_EUCLIDEAN, true>(ix, a, smem, 0, stream) : launch_scan<0, METRIC_EUCLIDEAN, false>(ix, a, smem, 0, stream);
        break;
      case SDB_METRIC_DOT:
        rc = qsmem ? launch_scan<0, METRIC_DOT, true>(ix, a, smem, 0, stream) : launch_scan<0, METRIC_DOT, false>(ix, a, smem, 0, stream);
        break;
      case SDB_METRIC_COSINE:
        rc = qsmem ? launch_scan<0, METRIC_COSINE, true>(ix, a, smem, 0, stream) : launch_scan<0, METRIC_COSINE, false>(ix, a, smem, 0, stream);
        break;
      case SDB_METRIC_HAVERSINE: rc = launch_scan<0, METRIC_HAVERSINE, true>(ix, a, smem, 0, stream); break;
      default: return fail(SDB_ERR_INVALID, "metric not supported by the flat scan");
    }
    if (rc) return rc;
  }
  flat_merge_kernel<<<(B + 127) / 128, 128, 0, stream>>>(a, d_out_ids, d_out_dists, d_out_counts);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

int launch_flat_exact_list(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_list,
                           const uint32_t* d_count, uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                           cudaStream_t stream, uint32_t first_id, uint32_t end_id) {
  if (ix->quant_active() || ix->store_metric == SDB_METRIC_HAVERSINE)
    return fail(SDB_ERR_INTERNAL, "flat scan of a query list: f32 squared-L2 / dot / cosine stores only");
  FlatArgs a;
  bool qsmem;
  int rc;
  if ((rc = flat_args(ix, B, d_queries, k, nullptr, first_id, end_id, a, qsmem))) return rc;
  a.qlist = d_list;
  a.qcount = d_count;
  // the count is only known on the device: size the partial lists and the grid for the largest
  // split any count 1..B can take (one CTA per work item at the worst count)
  const uint32_t npts = a.end_id - a.first_id;
  size_t parts = 0;
  uint32_t grid = 1;
  for (uint32_t qb = 1; qb <= (B + FQ - 1) / FQ; ++qb) {
    const uint32_t nq = std::min(B, qb * FQ);
    const FlatSplit sp = flat_split(nq, npts, a.tile_pts, a.sm_count);
    parts = std::max(parts, size_t(nq) * sp.n_chunks);
    grid = std::max(grid, qb * sp.n_chunks);
  }
  if ((rc = ix->d_tmp32.ensure(parts * (k + 1)))) return rc;
  if ((rc = ix->d_tmpf.ensure(parts * k))) return rc;
  a.part_ids = ix->d_tmp32.p;
  a.part_cnt = ix->d_tmp32.p + parts * k;
  a.part_d = ix->d_tmpf.p;
  const size_t smem = ((qsmem ? size_t(FQ) : 0) + a.tile_pts) * size_t(a.dim) * sizeof(float);
  switch (ix->store_metric) {
    case SDB_METRIC_EUCLIDEAN:
      rc = qsmem ? launch_scan<0, METRIC_EUCLIDEAN, true, true>(ix, a, smem, grid, stream) : launch_scan<0, METRIC_EUCLIDEAN, false, true>(ix, a, smem, grid, stream);
      break;
    case SDB_METRIC_DOT:
      rc = qsmem ? launch_scan<0, METRIC_DOT, true, true>(ix, a, smem, grid, stream) : launch_scan<0, METRIC_DOT, false, true>(ix, a, smem, grid, stream);
      break;
    default:
      rc = qsmem ? launch_scan<0, METRIC_COSINE, true, true>(ix, a, smem, grid, stream) : launch_scan<0, METRIC_COSINE, false, true>(ix, a, smem, grid, stream);
      break;
  }
  if (rc) return rc;
  flat_merge_kernel<<<(B + 127) / 128, 128, 0, stream>>>(a, d_out_ids, d_out_dists, d_out_counts);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

// ---- filtered requests ------------------------------------------------------------------
// Per-filter route. A filter f used by n_f requests that names m_f rows costs n_f * m_f gathered
// (request, row) pairs on the gather route (flat_filter.cu), and ceil(n_f / FQ) passes of the
// range scan over all npts points on the scan route (flat_scan_kernel with f's bitmap, one CTA row
// of FQ query slots per pass). FLAT_GATHER_PAIRS_PER_POINT gathered pairs cost as much as one
// point of one scan pass: gather iff n_f * m_f < FLAT_GATHER_PAIRS_PER_POINT * ceil(n_f / FQ) * npts.
// Measured (scripts/bench_flat_filters.py, profiles/r03_flat_filters.json, B200 at 1 000 W): one
// filter of 16 384 ids on 1M x 128 f32 L2, kernel time of both routes — a scanned point-pass costs
// 14.9 gathered pairs at 1 024 requests (0.083 ns per pair, 1.23 ns per point-pass) and 29.3 at 128.
// The full-batch figure is the one used; a filter near the boundary costs about the same either way.
constexpr double FLAT_GATHER_PAIRS_PER_POINT = 15.0;
constexpr uint32_t FLAT_GATHER_CHUNK = 1024;  // ids per gather work item (one warp)

namespace {

// rows d_list[0..n) of the batch through `run` on a compacted copy of their queries, results
// scattered back into the batch's outputs
template <class Run>
int run_subset(sdb_index* ix, const uint32_t* d_list, uint32_t n, const float* d_queries, uint32_t k, uint64_t* d_out_ids,
               float* d_out_dists, uint32_t* d_out_counts, cudaStream_t stream, Run run) {
  const uint32_t dim = ix->p.dim;
  int rc;
  if ((rc = ix->d_fsub_q.ensure(size_t(n) * dim)) || (rc = ix->d_fsub_ids.ensure(size_t(n) * k)) ||
      (rc = ix->d_fsub_d.ensure(size_t(n) * k)) || (rc = ix->d_fsub_cnt.ensure(n)))
    return rc;
  gather_queries_kernel<<<n, 128, 0, stream>>>(d_list, n, d_queries, dim, ix->d_fsub_q.p);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  if ((rc = run(n, ix->d_fsub_q.p, ix->d_fsub_ids.p, ix->d_fsub_d.p, ix->d_fsub_cnt.p))) return rc;
  scatter_results_kernel<<<n, 128, 0, stream>>>(d_list, n, k, ix->d_fsub_ids.p, ix->d_fsub_d.p, ix->d_fsub_cnt.p,
                                                d_out_ids, d_out_dists, d_out_counts);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

}  // namespace

int flat_plan(sdb_index* ix, uint32_t s, uint32_t B, uint32_t n_filters, const uint32_t* h_off, const int32_t* query_filter,
              uint32_t npts, uint8_t* slot, size_t at, FlatFilterPlan* p) {
  auto filter_of = [&](uint32_t b) -> int32_t { return query_filter ? query_filter[b] : 0; };
  // requests per filter, grouped by filter (counting sort, batch order within a filter)
  auto& first = p->first;
  first.assign(size_t(n_filters) + 1, 0);
  for (uint32_t b = 0; b < B; ++b)
    if (filter_of(b) >= 0) first[filter_of(b) + 1]++;
  for (uint32_t f = 0; f < n_filters; ++f) first[f + 1] += first[f];
  const bool scan_all = getenv("SDB_FLAT_EXACT") != nullptr;  // tests: every filter through the range scan
  p->gather.assign(n_filters, 0);
  p->n_scanned = 0;
  p->pairs = 0;
  for (uint32_t f = 0; f < n_filters; ++f) {
    const uint64_t nf = first[f + 1] - first[f], mf = h_off[f + 1] - h_off[f];
    if (nf == 0) continue;
    p->gather[f] = !scan_all && double(nf) * double(mf) < FLAT_GATHER_PAIRS_PER_POINT * double((nf + FQ - 1) / FQ) * npts;
    if (p->gather[f]) p->pairs += nf * mf;
    else p->n_scanned++;
  }
  // ---- gather route: work items (request, chunk of its filter's ids) in batch order
  uint64_t n_items = 0;
  uint32_t n_req = 0;
  for (uint32_t b = 0; b < B; ++b) {
    const int32_t f = filter_of(b);
    if (f < 0 || !p->gather[f]) continue;
    n_req++;
    n_items += (h_off[f + 1] - h_off[f] + FLAT_GATHER_CHUNK - 1) / FLAT_GATHER_CHUNK;
  }
  if (n_items >= (uint64_t(1) << 32)) return fail(SDB_ERR_INVALID, "filters: too many ids in one batch");
  p->n_items = uint32_t(n_items);
  p->n_req = n_req;
  p->req_at = at;
  p->rows_at = p->req_at + align16((size_t(n_req) * 2 + 1) * 4);
  p->items_at = p->rows_at + align16(size_t(B) * 4);
  int rc;
  if ((rc = ix->h_stage_items[s].ensure(n_items))) return rc;
  uint4* items = ix->h_stage_items[s].p;
  uint32_t* req = reinterpret_cast<uint32_t*>(slot + p->req_at);  // [n_req] batch rows, then [n_req + 1] first items
  uint32_t* rows = reinterpret_cast<uint32_t*>(slot + p->rows_at);
  uint32_t it = 0, r = 0, plain = first[n_filters];
  for (uint32_t b = 0; b < B; ++b) {
    const int32_t f = filter_of(b);
    if (f < 0) { rows[plain++] = b; continue; }
    rows[first[f]++] = b;  // first[f] becomes the end of f's requests: restored below
    if (!p->gather[f]) continue;
    req[r] = b;
    req[n_req + r++] = it;
    for (uint32_t s = h_off[f]; s < h_off[f + 1]; s += FLAT_GATHER_CHUNK)
      items[it++] = make_uint4(b, s, std::min(h_off[f + 1], s + FLAT_GATHER_CHUNK), 0);
  }
  req[2 * n_req] = it;
  for (uint32_t f = n_filters; f > 0; --f) first[f] = first[f - 1];
  first[0] = 0;
  p->n_plain = plain - first[n_filters];
  return SDB_OK;
}

int launch_flat_filtered(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const FilterStage& fs,
                         uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, cudaStream_t stream) {
  const uint32_t end_id = std::max<uint32_t>(2, ix->max_node_id + 1);
  const FlatFilterPlan& p = fs.flat;
  const uint32_t n_filters = uint32_t(p.gather.size());
  const uint32_t* h_off = fs.h_off;
  const uint32_t* d_ids = fs.sf.ids;
  const uint8_t* d = ix->d_fstage.p;
  const uint32_t* d_rows = reinterpret_cast<const uint32_t*>(d + p.rows_at);
  ix->flat_last_scanned = p.n_scanned;
  ix->flat_last_gathered = 0;
  for (uint32_t f = 0; f < n_filters; ++f) ix->flat_last_gathered += p.gather[f];
  ix->flat_last_pairs = p.pairs;
  ix->flat_last_path = 0;
  ix->flat_last_candidates = 0;
  ix->flat_last_overflow = 0;
  ix->flat_stats_pending = false;
  int rc;
  // ---- gather route
  if (p.n_req) {
    const uint32_t* d_req = reinterpret_cast<const uint32_t*>(d + p.req_at);
    if ((rc = launch_flat_gather(ix, B, d_queries, k, d_ids, p.n_items, reinterpret_cast<const uint4*>(d + p.items_at), p.n_req,
                                 d_req, d_req + p.n_req, d_out_ids, d_out_dists, d_out_counts, stream)))
      return rc;
  }
  // ---- scan route: the range scan with the filter's bitmap over the filter's requests
  for (uint32_t f = 0; f < n_filters; ++f) {
    if (p.first[f + 1] == p.first[f] || p.gather[f]) continue;
    if ((rc = ix->d_filter_bits.ensure((size_t(ix->rows) + 31) / 32 + 1))) return rc;
    if ((rc = launch_filter_bits(ix, d_ids + h_off[f], h_off[f + 1] - h_off[f], ix->d_filter_bits.p, stream))) return rc;
    rc = run_subset(ix, d_rows + p.first[f], p.first[f + 1] - p.first[f], d_queries, k, d_out_ids, d_out_dists, d_out_counts,
                    stream, [&](uint32_t n, const float* q, uint64_t* oi, float* od, uint32_t* oc) {
                      return launch_flat_exact(ix, n, q, k, ix->d_filter_bits.p, oi, od, oc, stream, 2, end_id);
                    });
    if (rc) return rc;
  }
  // ---- unfiltered requests: the unfiltered pass (tensor-core form where eligible) over their subset
  if (p.n_plain == B) return launch_flat(ix, B, d_queries, k, nullptr, d_out_ids, d_out_dists, d_out_counts, stream);
  if (p.n_plain)
    return run_subset(ix, d_rows + p.first[n_filters], p.n_plain, d_queries, k, d_out_ids, d_out_dists, d_out_counts, stream,
                      [&](uint32_t n, const float* q, uint64_t* oi, float* od, uint32_t* oc) {
                        return launch_flat(ix, n, q, k, nullptr, oi, od, oc, stream);
                      });
  return SDB_OK;
}

}  // namespace sdb
