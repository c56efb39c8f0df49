// search.cu — dispatch of the beam-search kernel variants (search.cuh), and the entries that search
// a shard and store its lists into every peer GPU's gather buffer (beam search and flat search).
#include "search_launch.cuh"

#include <algorithm>

namespace sdb {

namespace launch {
// one translation unit per f32 metric (search_l2.cu, search_dot.cu, search_cos.cu)
extern template int launch_float<METRIC_EUCLIDEAN>(sdb_index*, const SearchArgs&, bool, cudaStream_t);
extern template int launch_float<METRIC_DOT>(sdb_index*, const SearchArgs&, bool, cudaStream_t);
extern template int launch_float<METRIC_COSINE>(sdb_index*, const SearchArgs&, bool, cudaStream_t);
// search_bits.cu / search_pq.cu: the bit-row and PQ-code evaluators
int launch_bits(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream);
int launch_pq(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream);
// search_geo.cu: dim-2 haversine rows
int launch_geo(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream);
}  // namespace launch
using namespace launch;

// Visited-table slots of the geo kernel (profiles/r03_geo.json, B200 at 1000 W): a geo query evaluates
// ~590 rows on average at L = 75 (p99 920, max 1240 at 1 M points; p99 1130, max 3500 at 10 M). 1024
// slots (limit 896) send the tail to the RETRY launch: 3.8 M QPS at 1 M points against 6.0 M with 2048
// and 4.1 M with 4096 (why 4096 costs that much is not measured). A level is usable when the quotient
// span (VisitedCompactN::init) leaves a displacement of at least 2 buckets: at 10 M points 2048 slots
// have span 32768 and no displacement, every bucket collision spills (0.44 M QPS), 4096 slots 2.4 M.
// So: 2048 slots up to 2^23 rows, 4096 up to 2^24, ...; the retry step-up (vt_level) moves on from there.
static uint32_t geo_vt_slots(const sdb_index* ix) {
  static const uint32_t kGeoSlots[4] = {2048, 4096, 8192, 16384};
  uint32_t b = ix->rows <= 2 ? 1 : 32 - uint32_t(__builtin_clz(ix->rows - 1));
  if (b < 16) b = 16;
  int lvl = 0;
  auto span = [&](int l) { return ((uint64_t(1) << b) + kGeoSlots[l] / 4 - 1) / (kGeoSlots[l] / 4); };
  while (lvl < 3 && (65535u - std::min<uint64_t>(span(lvl), 65535u)) / span(lvl) < 2) ++lvl;
  return kGeoSlots[std::min(3, lvl + ix->vt_level)];
}

static int dispatch_search(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream);

int launch_search(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint32_t L, uint64_t* d_out_ids,
                  float* d_out_dists, uint32_t* d_out_counts, uint32_t* d_vis_ids, float* d_vis_dists,
                  uint32_t* d_vis_len, uint32_t vis_cap, const SearchFilters* filters, cudaStream_t stream) {
  // Visited-table size for this launch: start at 5888 slots; if the previous search on this
  // handle sent more than 0.1 % of its queries to the RETRY launch (they visited more nodes than
  // 87.5 % of the table), step up. Read only when the stream is idle: never adds a sync.
  if (ix->retry_check_pending && cudaStreamQuery(ix->last_search_stream) == cudaSuccess) {
    uint32_t h_retry = 0;
    SDB_CUDA(cudaMemcpy(&h_retry, ix->d_work.p + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    // A re-run query costs about as much as a whole first-pass wave (it walks its ~80 hops
    // alone on an SM), so a handful per batch already outweighs the ~5-10 % the bigger table
    // costs everybody: step up above 0.1 % of the batch (or any at all in a small batch).
    if ((uint64_t(h_retry) * 1000 > ix->last_B || (h_retry > 0 && ix->last_B <= 2000)) && ix->vt_level < 2) ix->vt_level++;
    ix->retry_check_pending = false;
  }
  int rc;
  if ((rc = ix->d_hops.ensure(B))) return rc;
  if ((rc = ix->d_ndist.ensure(B))) return rc;
  if ((rc = ix->d_work.ensure(4 + size_t(B)))) return rc;
  static const uint32_t kSlots[3] = {5888, 8192, 12288};
  SDB_CUDA(cudaMemsetAsync(ix->d_work.p, 0, 4 * sizeof(uint32_t), stream));
  SearchArgs a{};
  a.vt_slots = kSlots[ix->vt_level];
  if (ix->store_metric == SDB_METRIC_HAVERSINE && !ix->quant_active()) a.vt_slots = geo_vt_slots(ix);
  if (const char* e = getenv("SDB_VT_SLOTS")) a.vt_slots = uint32_t(atoi(e)) / 8 * 8;
  a.vec = ix->d_vec;
  a.vec_pitch = ix->vec_pitch;
  a.bits = ix->d_bits;
  a.bits_pitch = ix->bits_pitch;
  a.words = ix->words;
  a.codes = ix->d_codes;
  a.codes_pitch = ix->codes_pitch;
  a.pqM = ix->pqM;
  a.pqK = ix->pqK;
  a.bq_thr = ix->d_bq_thr;
  a.bit_metric = ix->bq_metric;
  a.adj = ix->d_adj;
  a.R = ix->p.degree_bound;
  a.start_extra = ix->d_start_extra.p;
  a.n_start_extra = uint32_t(ix->h_start_extra.size());
  a.rows = ix->rows;
  a.queries = d_queries;
  a.dim = ix->p.dim;
  a.B = B;
  a.L = L;
  a.k = k;
  a.out_ids = d_out_ids;
  a.out_dists = d_out_dists;
  a.out_counts = d_out_counts;
  a.out_hops = ix->d_hops.p;
  a.out_ndist = ix->d_ndist.p;
  a.vis_ids = d_vis_ids;
  a.vis_dists = d_vis_dists;
  a.vis_len = d_vis_len;
  a.vis_cap = vis_cap;
  a.n_work = B;
  // RETRY launch: one visited bitmap over all rows per resident CTA (at most 512 MB in total)
  {
    const uint32_t words = ((ix->rows + 31) / 32 + 3) / 4 * 4;
    uint32_t slots = uint32_t(std::min<uint64_t>(uint64_t(ix->sm_count), std::max<uint64_t>(1, (uint64_t(512) << 20) / (uint64_t(words) * 4))));
    if ((rc = ix->d_retry_bitmap.ensure(size_t(words) * slots))) return rc;
    a.retry_bitmap = ix->d_retry_bitmap.p;
    a.bitmap_words = words;
    ix->retry_slots = slots;
  }
  if (ix->gather) a.pg = *ix->gather;
  a.work_counter = ix->d_work.p;
  a.retry_count = ix->d_work.p + 1;
  a.retry_list = ix->d_work.p + 4;
  ix->last_B = B;
  ix->retry_check_pending = true;
  ix->last_search_stream = stream;
  if (ix->p.quantizer == SDB_QUANT_PRODUCT && ix->pq_fitted) {
    a.pq_cent = ix->d_pq_centroids;
    if (!adc_on_the_fly(ix)) {  // materialised per-query tables (product.go:255-263), K4
      if ((rc = ix->d_adc.ensure(size_t(B) * ix->pqM * ix->pqK))) return rc;
      if ((rc = launch_adc_tables(ix, B, d_queries, ix->d_adc.p, stream))) return rc;
      a.adc = ix->d_adc.p;
    }
  }
  if (filters == nullptr) return dispatch_search(ix, a, false, stream);
  // per-request filters: the unfiltered requests of the batch run through the fast kernels, the
  // filtered ones through the FILTER variant, each over its own subset of the batch
  if (filters->n_plain > 0) {
    SearchArgs u = a;
    u.qmap = filters->n_plain == B ? nullptr : filters->qmap_plain;
    u.n_work = filters->n_plain;
    if ((rc = dispatch_search(ix, u, false, stream))) return rc;
    if (filters->n_filtered > 0) SDB_CUDA(cudaMemsetAsync(ix->d_work.p, 0, 4 * sizeof(uint32_t), stream));
  }
  if (filters->n_filtered > 0) {
    a.filter_ids = filters->ids;
    a.filter_off = filters->off;
    a.query_filter = filters->query_filter;
    a.filter_bits = filters->bits;
    a.qmap = filters->n_filtered == B ? nullptr : filters->qmap_filtered;
    a.n_work = filters->n_filtered;
    return dispatch_search(ix, a, true, stream);
  }
  return SDB_OK;
}

static int dispatch_search(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream) {
  if (ix->p.quantizer == SDB_QUANT_BINARY && ix->bq_fitted) return launch_bits(ix, a, filtered, stream);
  if (ix->p.quantizer == SDB_QUANT_PRODUCT && ix->pq_fitted) return launch_pq(ix, a, filtered, stream);
  switch (ix->store_metric) {
    case SDB_METRIC_EUCLIDEAN: return launch_float<METRIC_EUCLIDEAN>(ix, a, filtered, stream);
    case SDB_METRIC_DOT: return launch_float<METRIC_DOT>(ix, a, filtered, stream);
    case SDB_METRIC_COSINE: return launch_float<METRIC_COSINE>(ix, a, filtered, stream);
    case SDB_METRIC_HAVERSINE: return launch_geo(ix, a, filtered, stream);
    default: return fail(SDB_ERR_INVALID, "metric not supported by the Vamana search kernel");
  }
}

// the caller's peer buffers (sdb_peer_gather) as the kernels take them, for a top-k of k slots
static int peer_gather_args(const sdb_peer_gather* pg, uint32_t k, PeerGather* g) {
  if (pg->n_peers == 0 || pg->n_peers > SDB_MAX_PEERS || pg->shard >= (1u << 24))
    return fail(SDB_ERR_INVALID, "peer gather: n_peers must be 1..16");
  *g = PeerGather{};
  g->n = pg->n_peers;
  g->shard = pg->shard;
  g->limit = pg->per_shard_limit == 0 || pg->per_shard_limit > k ? k : pg->per_shard_limit;
  g->tag = uint64_t(pg->shard) << 40;
  for (uint32_t p = 0; p < pg->n_peers; ++p) {
    if (!pg->ids[p] || !pg->dists[p] || !pg->counts[p]) return fail(SDB_ERR_INVALID, "peer gather: null peer buffer");
    g->ids[p] = pg->ids[p];
    g->dists[p] = pg->dists[p];
    g->counts[p] = pg->counts[p];
  }
  return SDB_OK;
}

// Flat shards: the flat search's last writer is known only once its whole sequence has run (the
// overflow fallback rewrites rows after the re-score), so a kernel of its own publishes the final
// lists. Slot [shard][q] of every peer's buffer gets the bytes the beam-search epilogue stores:
// tagged ids and the distances of the first count ranks, id 0 / +inf in the rest, count
// min(count, limit). One thread per (query, rank); rank 0's thread also writes the counts.
__global__ void flat_publish_kernel(PeerGather g, uint32_t B, uint32_t k, const uint64_t* ids, const float* dists,
                                    const uint32_t* counts) {
  const uint64_t t = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= uint64_t(B) * k) return;
  const uint32_t q = uint32_t(t / k), r = uint32_t(t % k);
  const uint32_t cnt = min(counts[q], k);
  const bool have = r < cnt;
  const uint64_t id = have ? (ids[t] | g.tag) : 0;
  const float d = have ? dists[t] : __int_as_float(0x7f800000);
  const size_t o = (size_t(g.shard) * B + q) * k + r;
  for (uint32_t s = 0; s < g.n; ++s) {
    g.ids[s][o] = id;
    g.dists[s][o] = d;
    if (r == 0) g.counts[s][size_t(g.shard) * B + q] = min(cnt, g.limit);
  }
}

}  // namespace sdb

using namespace sdb;

extern "C" int sdb_search_batch_gather_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k,
                                              uint32_t search_size, uint64_t* d_out_ids, float* d_out_dists,
                                              uint32_t* d_out_counts, const sdb_peer_gather* pg, void* stream) {
  if (!ix || !pg) return fail(SDB_ERR_INVALID, "null argument");
  if (B == 0) return SDB_OK;
  if (!d_queries || !d_out_ids || !d_out_dists || !d_out_counts) return fail(SDB_ERR_INVALID, "null argument");
  PeerGather g;
  if (int prc = peer_gather_args(pg, k, &g)) return prc;
  if (k == 0 || search_size < k) return fail(SDB_ERR_INVALID, "searchSize must be greater than or equal to k");
  std::lock_guard<std::mutex> lk(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (int prc = peer_barrier_poisoned(ix->device)) return prc;
  ix->gather = &g;
  int rc = launch_search(ix, B, d_queries, k, search_size, d_out_ids, d_out_dists, d_out_counts, nullptr, nullptr, nullptr, 0,
                         nullptr, static_cast<cudaStream_t>(stream));
  ix->gather = nullptr;
  return rc;
}

extern "C" int sdb_flat_search_batch_gather_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k,
                                                   uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                                                   const sdb_peer_gather* pg, void* stream) {
  if (!ix || !pg) return fail(SDB_ERR_INVALID, "null argument");
  if (B == 0) return SDB_OK;
  if (!d_queries || !d_out_ids || !d_out_dists || !d_out_counts) return fail(SDB_ERR_INVALID, "null argument");
  PeerGather g;
  if (int prc = peer_gather_args(pg, k, &g)) return prc;
  if (k < 1 || k > 75) return fail(SDB_ERR_INVALID, "invalid limit for vector query, expected 1-75");  // models/search.go:329
  std::lock_guard<std::mutex> lk(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (int prc = peer_barrier_poisoned(ix->device)) return prc;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = flat_device_locked(ix, B, d_queries, k, d_out_ids, d_out_dists, d_out_counts, st);
  if (rc) return rc;
  const uint64_t n = uint64_t(B) * k;
  flat_publish_kernel<<<uint32_t((n + 255) / 256), 256, 0, st>>>(g, B, k, d_out_ids, d_out_dists, d_out_counts);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}
