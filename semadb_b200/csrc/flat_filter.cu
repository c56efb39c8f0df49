// flat_filter.cu — K5 under a per-request filter: score only the filter's rows.
//
// IndexFlat.Search checks filter membership while it iterates the store (flat.go:94-96); a
// request whose filter names m rows therefore has m candidates, and scoring those m rows is the
// whole job. Work item = (filtered request, chunk of at most FG_CHUNK ids of its filter), one WARP
// per item: the item's rows are gathered by id, scored with exactly the evaluator the range scan
// (flat.cu) uses for the store, and kept in a register top-k (WarpTopK) by (distance asc, id asc).
// A second kernel merges a request's chunk lists — the same total order, so the result is the
// scan's, bit for bit. Which filters take this route and which take the range scan is decided in
// flat.cu (launch_flat_filtered).
//
// Evaluators (chosen as launch_flat_exact chooses its mode):
//   f32 L2 / dot / cosine: an 8-lane group per row, query in shared memory, the reference's summation
//     order (trip_accum / tail_accum / group_reduce). 16 rows per warp step (4 per group); trips are
//     loaded four at a time, so a lane has 16 row loads in flight at any dim (dim <= 128: the whole
//     rows, as in rescore_warp_kernel's short form);
//   haversine: one lane per row, the query's terms once (haversine_terms), then haversine_from;
//   binary store (hamming / jaccard): the query encoded once per warp against bq_thr, one lane per row;
//   PQ: the request's ADC table (launch_adc_tables), one lane per row, M lookups in sub-vector order.
#include <algorithm>

#include "common.cuh"
#include "index.cuh"
#include "warp_topk.cuh"

namespace sdb {

namespace {

constexpr int FG_WARPS = 4;  // work items per CTA

struct GatherArgs {
  const float* vec; uint32_t vec_pitch;
  const uint64_t* bits; uint32_t bits_pitch; uint32_t words;
  const uint8_t* codes; uint32_t codes_pitch;
  const float* adc; uint32_t pqM, pqK;
  const float* bq_thr; int bit_metric;
  const uint8_t* exists;
  const float* queries; uint32_t dim, k;
  const uint32_t* ids;        // staged filter ids, ascending within each filter
  const uint4* items;         // x = batch row of the request, [y, z) = its ids in `ids`
  uint32_t n_items;
  uint32_t* part_ids;         // [n_items][k]
  float* part_d;
  uint32_t* part_cnt;         // [n_items]
};

// mode 0: f32 rows (METRIC), 1: bits, 2: PQ codes via the ADC table
template <int MODE, int METRIC, int NS>
__global__ void __launch_bounds__(32 * FG_WARPS) flat_gather_kernel(GatherArgs a) {
  extern __shared__ __align__(16) unsigned char fg_sm[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t it = blockIdx.x * FG_WARPS + wid;
  if (it >= a.n_items) return;
  const uint4 item = a.items[it];
  const uint32_t b = item.x, c_begin = item.y, c_end = item.z;
  SDB_WARP_TOPK_STATE(top, NS, a.k, lane);
  if (MODE == 0 && METRIC != METRIC_HAVERSINE) {
    const int g = lane & 7, grp = lane >> 3;
    const uint32_t dpad = (a.dim + 3) & ~3u;
    float* s_q = reinterpret_cast<float*>(fg_sm) + size_t(wid) * dpad;
    for (uint32_t i = lane; i < dpad; i += 32) s_q[i] = i < a.dim ? a.queries[size_t(b) * a.dim + i] : 0.0f;
    __syncwarp();
    constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
    const int trips = a.dim >> 5;
    for (uint32_t c0 = c_begin; c0 < c_end; c0 += 16) {
      uint32_t pid[4];
      float4 acc[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t c = c0 + u * 4 + grp;
        pid[u] = a.ids[c < c_end ? c : c_begin];
        acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      for (int t0 = 0; t0 < trips; t0 += 4) {
        float4 y[4][4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float* row = a.vec + size_t(pid[u]) * a.vec_pitch + 4 * g + 32 * t0;
#pragma unroll
          for (int t = 0; t < 4; ++t) y[u][t] = t0 + t < trips ? ldg_f4_stream(row + 32 * t) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int t = 0; t < 4; ++t)
            if (t0 + t < trips) trip_accum<L2>(*reinterpret_cast<const float4*>(s_q + 32 * (t0 + t) + 4 * g), y[u][t], acc[u]);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t c = c0 + u * 4 + grp;
        const float* row = a.vec + size_t(pid[u]) * a.vec_pitch;
        float tail = 0.0f;
        if (g == 0)
          for (uint32_t i = trips << 5; i < a.dim; ++i) tail = tail_accum<L2>(s_q[i], __ldg(row + i), tail);
        const float r = metric_epilogue<METRIC>(group_reduce(acc[u], tail));
        top.offer(r, pid[u], g == 0 && c < c_end && a.exists[pid[u]]);
      }
    }
  } else {
    // one lane per row
    const float* qv = a.queries + size_t(b) * a.dim;
    HaversineX hx{};
    if (MODE == 0) hx = haversine_terms(qv[0], qv[1]);
    uint64_t* qb = reinterpret_cast<uint64_t*>(fg_sm) + size_t(wid) * a.words;
    if (MODE == 1) {
      for (uint32_t w = lane; w < a.words; w += 32) {
        uint64_t word = 0;
        for (uint32_t bit = 0; bit < 64; ++bit) {
          const uint32_t i = w * 64 + bit;
          if (i < a.dim && qv[i] > a.bq_thr[i]) word |= uint64_t(1) << bit;
        }
        qb[w] = word;
      }
      __syncwarp();
    }
    const float* table = MODE == 2 ? a.adc + size_t(b) * a.pqM * a.pqK : nullptr;
    for (uint32_t c0 = c_begin; c0 < c_end; c0 += 32) {
      const uint32_t c = c0 + lane;
      const uint32_t pid = a.ids[c < c_end ? c : c_begin];
      const bool have = c < c_end && a.exists[pid];
      float d = 0.0f;
      if (have) {
        if (MODE == 0) {
          const float* y = a.vec + size_t(pid) * a.vec_pitch;
          d = haversine_from(hx, __ldg(y), __ldg(y + 1));
        } else if (MODE == 1) {
          const uint64_t* y = a.bits + size_t(pid) * a.bits_pitch;
          int x = 0, un = 0;
          for (uint32_t w = 0; w < a.words; ++w) {
            const uint64_t yw = __ldg(y + w);
            if (a.bit_metric == METRIC_JACCARD) { x += __popcll(qb[w] & yw); un += __popcll(qb[w] | yw); }
            else x += __popcll(qb[w] ^ yw);
          }
          d = bits_finish(a.bit_metric, x, un);
        } else {
          const uint8_t* code = a.codes + size_t(pid) * a.codes_pitch;
          for (uint32_t i = 0; i < a.pqM; ++i) d = __fadd_rn(d, __ldg(table + i * a.pqK + __ldg(code + i)));
        }
      }
      top.offer(d, pid, have);
    }
  }
  const size_t o = size_t(it) * a.k;
#pragma unroll
  for (int j = 0; j < NS; ++j) {
    const uint32_t p = lane + 32 * j;
    if (p < top_len) { a.part_ids[o + p] = top_ki[j]; a.part_d[o + p] = top_kd[j]; }
  }
  if (lane == 0) a.part_cnt[it] = top_len;
}

// One warp per gathered request: its chunk lists (items req_items[r] .. req_items[r+1]) into the
// request's output row req_rows[r]; empty slots id 0 / +inf like flat_merge_kernel.
template <int NS>
__global__ void __launch_bounds__(32 * FG_WARPS) flat_gather_merge_kernel(
    const uint32_t* req_rows, const uint32_t* req_items, uint32_t n_req, uint32_t k, const uint32_t* part_ids,
    const float* part_d, const uint32_t* part_cnt, uint64_t* out_ids, float* out_d, uint32_t* out_cnt) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t r = blockIdx.x * FG_WARPS + wid;
  if (r >= n_req) return;
  SDB_WARP_TOPK_STATE(top, NS, k, lane);
  for (uint32_t it = req_items[r]; it < req_items[r + 1]; ++it) {
    const uint32_t n = part_cnt[it];
    const size_t o = size_t(it) * k;
    for (uint32_t i0 = 0; i0 < n; i0 += 32) {
      const uint32_t i = i0 + lane;
      const bool have = i < n;
      top.offer(have ? part_d[o + i] : 0.0f, have ? part_ids[o + i] : 0u, have);
    }
  }
  const uint32_t b = req_rows[r];
#pragma unroll
  for (int j = 0; j < NS; ++j) {
    const uint32_t p = lane + 32 * j;
    if (p < k) {
      out_ids[size_t(b) * k + p] = p < top_len ? uint64_t(top_ki[j]) : 0;
      out_d[size_t(b) * k + p] = p < top_len ? top_kd[j] : __int_as_float(0x7f800000);
    }
  }
  if (lane == 0) out_cnt[b] = top_len;
}

__global__ void filter_bits_kernel(const uint32_t* ids, uint32_t n, uint32_t* bits) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicOr(&bits[ids[i] >> 5], 1u << (ids[i] & 31));
}

template <int MODE, int METRIC>
int launch_gather(sdb_index* ix, const GatherArgs& a, size_t smem, cudaStream_t stream) {
  auto kern = a.k <= 32 ? flat_gather_kernel<MODE, METRIC, 1> : flat_gather_kernel<MODE, METRIC, 3>;
  if (smem > 48 * 1024) SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  kern<<<(a.n_items + FG_WARPS - 1) / FG_WARPS, 32 * FG_WARPS, smem, stream>>>(a);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

}  // namespace

int launch_flat_gather(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_ids,
                       uint32_t n_items, const uint4* d_items, uint32_t n_req, const uint32_t* d_req_rows,
                       const uint32_t* d_req_items, uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                       cudaStream_t stream) {
  if (n_req == 0) return SDB_OK;
  int rc;
  const size_t parts = size_t(n_items) * k;
  if ((rc = ix->d_fg_part32.ensure(parts + n_items + 1))) return rc;
  if ((rc = ix->d_fg_partf.ensure(parts + 1))) return rc;
  GatherArgs a{};
  a.vec = ix->d_vec; a.vec_pitch = ix->vec_pitch;
  a.bits = ix->d_bits; a.bits_pitch = ix->bits_pitch; a.words = ix->words;
  a.codes = ix->d_codes; a.codes_pitch = ix->codes_pitch;
  a.pqM = ix->pqM; a.pqK = ix->pqK;
  a.bq_thr = ix->d_bq_thr; a.bit_metric = ix->bq_metric;
  a.exists = ix->d_exists;
  a.queries = d_queries; a.dim = ix->p.dim; a.k = k;
  a.ids = d_ids; a.items = d_items; a.n_items = n_items;
  a.part_ids = ix->d_fg_part32.p;
  a.part_cnt = ix->d_fg_part32.p + parts;
  a.part_d = ix->d_fg_partf.p;
  if (n_items) {
    if (ix->p.quantizer == SDB_QUANT_BINARY && ix->bq_fitted) {
      rc = launch_gather<1, 0>(ix, a, size_t(FG_WARPS) * a.words * 8, stream);
    } else if (ix->p.quantizer == SDB_QUANT_PRODUCT && ix->pq_fitted) {
      if ((rc = ix->d_adc.ensure(size_t(B) * ix->pqM * ix->pqK))) return rc;
      if ((rc = launch_adc_tables(ix, B, d_queries, ix->d_adc.p, stream))) return rc;
      a.adc = ix->d_adc.p;
      rc = launch_gather<2, 0>(ix, a, 0, stream);
    } else {
      const size_t smem = size_t(FG_WARPS) * ((a.dim + 3) & ~3u) * sizeof(float);
      switch (ix->store_metric) {
        case SDB_METRIC_EUCLIDEAN: rc = launch_gather<0, METRIC_EUCLIDEAN>(ix, a, smem, stream); break;
        case SDB_METRIC_DOT: rc = launch_gather<0, METRIC_DOT>(ix, a, smem, stream); break;
        case SDB_METRIC_COSINE: rc = launch_gather<0, METRIC_COSINE>(ix, a, smem, stream); break;
        case SDB_METRIC_HAVERSINE: rc = launch_gather<0, METRIC_HAVERSINE>(ix, a, 0, stream); break;
        default: return fail(SDB_ERR_INVALID, "metric not supported by the flat scan");
      }
    }
    if (rc) return rc;
  }
  const uint32_t grid = (n_req + FG_WARPS - 1) / FG_WARPS;
  if (k <= 32)
    flat_gather_merge_kernel<1><<<grid, 32 * FG_WARPS, 0, stream>>>(d_req_rows, d_req_items, n_req, k, a.part_ids, a.part_d,
                                                                    a.part_cnt, d_out_ids, d_out_dists, d_out_counts);
  else
    flat_gather_merge_kernel<3><<<grid, 32 * FG_WARPS, 0, stream>>>(d_req_rows, d_req_items, n_req, k, a.part_ids, a.part_d,
                                                                    a.part_cnt, d_out_ids, d_out_dists, d_out_counts);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

int launch_filter_bits(sdb_index* ix, const uint32_t* d_ids, uint32_t n, uint32_t* d_bits, cudaStream_t stream) {
  SDB_CUDA(cudaMemsetAsync(d_bits, 0, (size_t(ix->rows) + 31) / 32 * sizeof(uint32_t), stream));
  if (n) {
    filter_bits_kernel<<<(n + 255) / 256, 256, 0, stream>>>(d_ids, n, d_bits);
    ix->launches++;
    SDB_CUDA(cudaGetLastError());
  }
  return SDB_OK;
}

}  // namespace sdb
