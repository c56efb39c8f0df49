// index.cuh — the device-resident index behind an sdb_index handle.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/semadb_b200.h"

namespace sdb {

constexpr uint32_t MAX_DIM = 4096;  // largest vector size an index accepts (models/index.go:285)

void set_error(const std::string& msg);
int fail(int code, const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);

#define SDB_CUDA(expr)                                         \
  do {                                                         \
    cudaError_t _e = (expr);                                   \
    if (_e != cudaSuccess) return ::sdb::cuda_fail(_e, #expr); \
  } while (0)

template <class T>
struct DevBuf {  // grow-only device scratch
  T* p = nullptr;
  size_t n = 0;
  int ensure(size_t want) {
    if (want <= n) return SDB_OK;
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
    size_t cap = want + want / 4 + 64;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), cap * sizeof(T));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(scratch)");
    n = cap;
    return SDB_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
};

template <class T>
struct PinBuf {  // grow-only pinned host staging
  T* p = nullptr;
  size_t n = 0;
  int ensure(size_t want) {
    if (want <= n) return SDB_OK;
    if (p) cudaFreeHost(p);
    p = nullptr;
    n = 0;
    size_t cap = want + want / 4 + 64;
    cudaError_t e = cudaMallocHost(reinterpret_cast<void**>(&p), cap * sizeof(T));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMallocHost(staging)");
    n = cap;
    return SDB_OK;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    n = 0;
  }
};

}  // namespace sdb

// Data layout in HBM (all row-indexed by node id; row 0 unused, row 1 = start node):
//   vec   [rows][vec_pitch]   f32, vec_pitch = dim rounded up to 4 floats (16-byte rows;
//                              512-byte aligned rows when dim = 128)
//   bits  [rows][bits_pitch]  u64, bits_pitch = ceil(dim/64) rounded up to 2 (binary store)
//   codes [rows][codes_pitch] u8,  codes_pitch = M rounded up to 16 (product store)
//   adj   [rows][R]           u32, unused slots = 0xFFFFFFFF
//   deg   [rows]              u32
//   exists[rows]              u8
namespace sdb { struct PeerGather; }

struct sdb_index {
  sdb_params p{};
  const sdb::PeerGather* gather = nullptr;  // set for the duration of sdb_search_batch_gather_device
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 148;
  size_t smem_optin = 0;
  size_t smem_per_sm = 233472;
  mutable std::mutex mu;

  uint32_t rows = 0;  // allocated rows
  uint32_t vec_pitch = 0, bits_pitch = 0, words = 0, codes_pitch = 0;
  float* d_vec = nullptr;
  uint64_t* d_bits = nullptr;
  uint8_t* d_codes = nullptr;
  uint32_t* d_adj = nullptr;
  uint32_t* d_deg = nullptr;
  uint8_t* d_exists = nullptr;
  uint8_t* d_dirty = nullptr;  // [rows] edge list changed since the last sdb_index_dirty_edges(clear)
  std::vector<uint8_t> h_exists;
  // edges of the start node beyond degree_bound: removeInboundEdges re-attaches orphaned nodes
  // with AddNeighbourIfNotExists, which is unbounded (prune.go:137-151, node.go:73-80)
  std::vector<uint32_t> h_start_extra;
  sdb::DevBuf<uint32_t> d_start_extra;
  uint64_t count = 0;
  uint32_t max_node_id = 0;

  // quantizer state
  int store_metric = 0;  // metric used by float distances of the store (PQ: cosine -> euclidean)
  bool bq_fitted = false;
  float* d_bq_thr = nullptr;
  int bq_metric = SDB_METRIC_HAMMING;
  uint32_t pqM = 0, pqK = 0, pqSub = 0;
  bool pq_fitted = false;
  float* d_pq_centroids = nullptr;  // [M][K][sub]
  float* d_pq_cdist = nullptr;      // [M][K][K]

  // scratch
  sdb::DevBuf<float> d_q;
  sdb::DevBuf<uint64_t> d_oid;
  sdb::DevBuf<float> d_od;
  sdb::DevBuf<uint32_t> d_oc, d_hops, d_ndist;
  sdb::DevBuf<uint32_t> d_work;
  sdb::DevBuf<uint32_t> d_retry_bitmap;  // RETRY launch: [retry_slots][rows/32] exact visited bitmaps
  uint32_t retry_slots = 1;
  sdb::DevBuf<float> d_adc;
  sdb::DevBuf<uint32_t> d_filter_ids, d_filter_off, d_filter_bits, d_qmap;
  sdb::DevBuf<int32_t> d_query_filter;
  sdb::DevBuf<uint32_t> d_vis_ids, d_vis_len;
  sdb::DevBuf<float> d_vis_d;
  sdb::DevBuf<uint64_t> d_ids64;
  sdb::DevBuf<uint32_t> d_tmp32;
  sdb::DevBuf<float> d_tmpf;
  sdb::DevBuf<uint8_t> d_tmp8;
  sdb::PinBuf<uint8_t> h_stage;
  // tensor-core flat scan (flat_tc.cu): bf16 shadow of the store + per-call scratch
  uint64_t flat_last_candidates = 0;  // tensor-core flat scan: candidates kept by the last level, all queries
  uint32_t flat_last_overflow = 0;    // ... and queries that fell back to the exact scan
  int flat_last_path = 0;             // 0 exact scan, 1 mma.sync candidate pass, 2 tcgen05 candidate pass
  // the two counters above as the last tensor-core call left them on the device: copied to h_flat_misc
  // behind its last kernel, event recorded after the copy; flat_stats_settle reads them when pending
  sdb::PinBuf<uint32_t> h_flat_misc;
  cudaEvent_t flat_stats_ev = nullptr;
  bool flat_stats_pending = false;
  // filtered flat search (flat.cu launch_flat_filtered, flat_filter.cu): routes of the last flat call
  // (sdb_flat_last_filter_stats), host staging of the gather route's work, device scratch of both routes
  uint32_t flat_last_gathered = 0, flat_last_scanned = 0;  // filters that took each route
  uint64_t flat_last_pairs = 0;                             // (request, id) pairs the gather route scored
  std::vector<uint4> h_fg_items;
  std::vector<uint32_t> h_fg_req;
  sdb::DevBuf<uint4> d_fg_items;
  sdb::DevBuf<uint32_t> d_fg_req, d_fg_part32, d_fsub_list, d_fsub_cnt;
  sdb::DevBuf<float> d_fg_partf, d_fsub_q, d_fsub_d;
  sdb::DevBuf<uint64_t> d_fsub_ids;
  uint64_t vec_epoch = 1, tc_epoch = 0;  // vec_epoch: bumped by every change to vec / exists
  sdb::DevBuf<uint16_t> d_x16, d_q16;
  sdb::DevBuf<float> d_xn, d_qn, d_thr, d_sample_d;
  sdb::DevBuf<float> d_bias;  // tcgen05 flat pass: per-point score bias (|x|^2 or 0; +inf = no such point)
  sdb::DevBuf<float> d_mu;    // squared-L2: translation applied to the bf16 shadow and the queries (+ partial sums)
  sdb::DevBuf<float> d_gmin;  // tcgen05 flat pass, minimum mode: [groups][B_pad] smallest approximate scores
  sdb::DevBuf<uint32_t> d_xmax;  // bits of the largest squared norm of a (centred) stored row
  sdb::DevBuf<uint32_t> d_cand, d_candcnt, d_sample_cnt;
  sdb::DevBuf<uint64_t> d_sample_ids;
  uint32_t last_B = 0;
  int vt_level = 0;                  // visited-table size step (search.cu)
  bool retry_check_pending = false;  // d_work holds the retry count of the last search
  cudaStream_t last_search_stream = nullptr;
  uint64_t launches = 0;
  // sdb_search_profile: CUDA events around the first-pass beam-search kernel of each search
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;  // [2 * PROF_RING]: start, stop pairs
  uint32_t prof_n = 0;               // searches recorded since enabling
  static constexpr uint32_t PROF_RING = 256;
  unsigned long long* d_ins_stats = nullptr;  // [8] running totals of the batched insert (insert.cu)
  uint64_t insert_truncated = 0;  // inserts whose visited list was cut to MAX_CAND candidates (insert.cu)

  // insert schedule
  // 1M x 128 build, same recall@10 (0.9992) at every setting: 1..4096 /16 2.39 s and 1..16384 /16 1.87 s with round 1's
  // kernels (profiles/r01_ab_insert.txt); with round 2's kernels 1..16384 /16 0.81 s, 1..32768 /8 0.70 s (profiles/r02_ab_insert.txt)
  // while the store's distance rows are wider than 512 bytes (C3: 384 floats) the larger batches cost more in the back-edge
  // prunes than they save: 1.25M x 384 builds in 2.8-3.7 s at 1..16384 /16 and 4.7-5.4 s at either larger setting. 0 = choose
  // by the width of the rows the searches read (insert.cu), sdb_insert_config overrides.
  uint32_t ins_min_batch = 1, ins_max_batch = 0, ins_growth_div = 0;
  uint32_t distance_row_bytes() const {
    if (p.quantizer == SDB_QUANT_BINARY && bq_fitted) return bits_pitch * 8;
    if (p.quantizer == SDB_QUANT_PRODUCT && pq_fitted) return codes_pitch;
    return vec_pitch * 4;
  }

  bool quant_active() const {
    return (p.quantizer == SDB_QUANT_BINARY && bq_fitted) || (p.quantizer == SDB_QUANT_PRODUCT && pq_fitted);
  }
};

namespace sdb {
int index_reserve_locked(sdb_index* ix, uint64_t max_node_id);
int peer_barrier_poisoned(int device);  // dist.cu: SDB_ERR_STATE once a cross-GPU barrier on the device has timed out
// Device-side description of a batch's filters (search.cuh SearchArgs): nullptr = no request is
// filtered. qmap_*: the batch positions of the filtered / unfiltered requests (either may be
// nullptr when its count is 0 or B).
struct SearchFilters {
  const uint32_t* ids = nullptr;          // concatenated ascending ids
  const uint32_t* off = nullptr;          // [n_filters + 1]
  const int32_t* query_filter = nullptr;  // [B], nullptr = every filtered query uses filter 0
  const uint32_t* bits = nullptr;         // optional bitmask over rows of filter 0
  const uint32_t* qmap_filtered = nullptr;
  uint32_t n_filtered = 0;
  const uint32_t* qmap_plain = nullptr;
  uint32_t n_plain = 0;
};
int launch_search(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint32_t L, uint64_t* d_out_ids,
                  float* d_out_dists, uint32_t* d_out_counts, uint32_t* d_vis_ids, float* d_vis_dists,
                  uint32_t* d_vis_len, uint32_t vis_cap, const SearchFilters* filters, cudaStream_t stream);
int launch_flat(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_filter_bits,
                uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, cudaStream_t stream);
int launch_flat_exact(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_filter_bits,
                      uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, cudaStream_t stream,
                      uint32_t first_id, uint32_t end_id);
// the exact scan of the batch rows d_list[0 .. min(*d_count, B)) (f32 stores without a filter): the
// count is read on the device, which splits the scan from it as launch_flat_exact does from B; each
// row's list goes to its row of the outputs, other rows are left as they are
int launch_flat_exact_list(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_list,
                           const uint32_t* d_count, uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                           cudaStream_t stream, uint32_t first_id, uint32_t end_id);
// completes flat_last_candidates / flat_last_overflow of the last tensor-core call (waits for it)
int flat_stats_settle(sdb_index* ix);
// unfiltered flat search, device queries and outputs, enqueued on `stream` (index.cu)
int flat_device_locked(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint64_t* d_out_ids, float* d_out_dists,
                       uint32_t* d_out_counts, cudaStream_t stream);
// Flat search of a batch whose requests carry filters (staged as by the Vamana search: ascending
// u32 ids in d_ids, filter f = [h_off[f], h_off[f+1]), ids 0 and 1 and ids >= rows dropped);
// query_filter[b] < 0 = request b unfiltered, nullptr = every request uses filter 0. Routes each
// filter to the gather kernel or to the range scan and the unfiltered requests to launch_flat.
int launch_flat_filtered(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint32_t n_filters,
                         const uint32_t* h_off, const int32_t* query_filter, const uint32_t* d_ids, uint64_t* d_out_ids,
                         float* d_out_dists, uint32_t* d_out_counts, cudaStream_t stream);
// flat_filter.cu: score each work item's ids (x = batch row, [y, z) = range of d_ids) and merge a
// request's items (d_req_items[r] .. d_req_items[r+1]) into output row d_req_rows[r]
int launch_flat_gather(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, const uint32_t* d_ids,
                       uint32_t n_items, const uint4* d_items, uint32_t n_req, const uint32_t* d_req_rows,
                       const uint32_t* d_req_items, uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                       cudaStream_t stream);
// the row bitmap of an id list (d_bits: rows/32 words, cleared first)
int launch_filter_bits(sdb_index* ix, const uint32_t* d_ids, uint32_t n, uint32_t* d_bits, cudaStream_t stream);
// flat_tc.cu: compact the rows list[0..n) of a batch, and scatter a compacted batch's results back
__global__ void gather_queries_kernel(const uint32_t* list, uint32_t n, const float* src, uint32_t dim, float* dst);
__global__ void scatter_results_kernel(const uint32_t* list, uint32_t n, uint32_t k, const uint64_t* ids, const float* d,
                                       const uint32_t* cnt, uint64_t* out_ids, float* out_d, uint32_t* out_cnt);
bool flat_tc_eligible(const sdb_index* ix, uint32_t k, bool filtered);
int launch_flat_tc(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint64_t* d_out_ids, float* d_out_dists,
                   uint32_t* d_out_counts, cudaStream_t stream);
int launch_encode_rows(sdb_index* ix, uint32_t n, const uint32_t* d_ids, cudaStream_t stream);
int launch_adc_tables(sdb_index* ix, uint32_t B, const float* d_queries, float* d_out, cudaStream_t stream);
int launch_merge(uint32_t S, uint32_t B, uint32_t k, const uint64_t* in_ids, const float* in_d, const uint32_t* in_c,
                 uint64_t* out_ids, float* out_d, uint32_t* out_c, cudaStream_t stream);
// reinsert: ids already exist (update path, vamana.go:249-253): rows are overwritten, one point per mini-batch
int insert_batch_locked(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors, bool reinsert = false,
                        bool vectors_on_device = false);
// VectorStore.Set on device-resident ids/vectors: scatter rows, mark exists, encode if fitted
int set_rows_device(sdb_index* ix, uint32_t n, const uint32_t* d_ids, const float* d_vecs, cudaStream_t stream);
int fit_locked(sdb_index* ix, uint64_t pq_first_row, int32_t* fitted);
// insertUpdateDelete (vamana.go:136-263) minus Fit/flush; has_vector[i] == 0 = nil vector
int insert_update_delete_locked(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors,
                                const uint8_t* has_vector);
int upload_start_extra(sdb_index* ix);
int dirty_edges_locked(sdb_index* ix, uint64_t cap, uint64_t* ids_out, uint64_t* n_out, int clear);
int edge_scan_locked(sdb_index* ix, uint64_t n_delete, const uint64_t* delete_ids, uint64_t* to_prune,
                     uint64_t* n_prune, uint64_t* to_save, uint64_t* n_save);
}  // namespace sdb
