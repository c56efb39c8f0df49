/* semadb_b200.h — C ABI of the B200-native vector-search hot path for SemaDB.
 *
 * This is the drop-in boundary: the entry points a Go shard binds through cgo in
 * place of its CPU implementation of shard/index/vamana (IndexVamana),
 * shard/index/flat (IndexFlat), shard/vectorstore (VectorStore + quantizers) and
 * distance (DistFunc family). Plain pointers and sizes only; no CUDA/torch types.
 * See INTEGRATION.md for the cgo stub. All reference citations are relative to
 * the semadb repository root.
 *
 * Conventions (precedent: internal/shardpy/shardpy.go:165-197)
 *  - caller allocates every output buffer, callee fills it;
 *  - no pointer is retained after a call returns (cgo pointer-passing rule):
 *    inputs are copied to pinned/device memory before return;
 *  - every function returns 0 on success or an SDB_ERR_* code; the message is
 *    available from sdb_last_error() on the calling thread. Nothing aborts or
 *    panics (CONTRIBUTING.md:150). There is NO CPU fallback: without a CUDA
 *    device every compute call fails with SDB_ERR_CUDA.
 *  - node ids are the reference's uint64 node ids (0 invalid, 1 = start node,
 *    user points from 2: vamana.go:28,150-157; idcounter.go:52-54). They must be
 *    dense small integers (< 2^31) because device rows are indexed by id.
 *  - a handle is internally serialised by a mutex; calls may come from any OS
 *    thread (cgo) and set the CUDA device on entry.
 *  - *_device variants take DEVICE pointers (same process, same device) and a
 *    cudaStream_t passed as void*; they enqueue work and do not synchronise.
 */
#ifndef SEMADB_B200_H
#define SEMADB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDB_ABI_VERSION 1

/* error codes */
#define SDB_OK 0
#define SDB_ERR_INVALID 1    /* bad argument / parameter out of the reference's range */
#define SDB_ERR_CUDA 2       /* CUDA runtime failure (incl. no device) */
#define SDB_ERR_OOM 3        /* host or device allocation failed */
#define SDB_ERR_STATE 4      /* call not valid in the current state (e.g. PQ not fitted) */
#define SDB_ERR_SEARCHSIZE 5 /* searchSize < k (search.go:23-25) */
#define SDB_ERR_RESERVED_ID 6 /* id 0 or 1 in an insert (vamana.go:150-157) */
#define SDB_ERR_NOTFOUND 7   /* a referenced node id does not exist */
#define SDB_ERR_INTERNAL 8

/* distance metrics — models/constants.go:7-14, distance/distance.go:70-97 */
#define SDB_METRIC_EUCLIDEAN 0 /* squared L2 (distance.go:14-16) */
#define SDB_METRIC_DOT 1       /* -dot (distance.go:19-21) */
#define SDB_METRIC_COSINE 2    /* 1-dot, caller normalises (distance.go:23-25) */
#define SDB_METRIC_HAMMING 3   /* distance.go:45-54, binary store forced on (vectorstore.go:56-66) */
#define SDB_METRIC_JACCARD 4   /* distance.go:56-67 */
#define SDB_METRIC_HAVERSINE 5 /* distance.go:33-43, dim must be 2 */

/* quantizers — models/quantizer.go:5-9 */
#define SDB_QUANT_NONE 0
#define SDB_QUANT_BINARY 1
#define SDB_QUANT_PRODUCT 2

/* Mirrors models.IndexVectorVamanaParameters (models/index.go:275-282) plus
 * models.Quantizer (models/quantizer.go:5-76). Ranges are validated like the
 * reference: searchSize 25..75, degreeBound 32..64, alpha 1.1..1.5, dim 1..4096,
 * PQ centroids 2..256, PQ subvectors >= 2 and dividing dim. Set `relaxed` to skip
 * the lower bounds (tests use tiny graphs; upper bounds always hold). */
typedef struct sdb_params {
  uint32_t dim;
  int32_t metric;
  uint32_t search_size;  /* L */
  uint32_t degree_bound; /* R */
  float alpha;
  int32_t quantizer;
  float bq_threshold;      /* NaN = unset: fit from the per-dimension mean (binary.go:145-185) */
  int32_t bq_metric;       /* SDB_METRIC_HAMMING or _JACCARD */
  uint32_t bq_trigger;     /* TriggerThreshold (models/quantizer.go:36) */
  uint32_t pq_subvectors;  /* M */
  uint32_t pq_centroids;   /* K */
  uint32_t pq_trigger;     /* TriggerThreshold (models/quantizer.go:62) */
  int32_t device;          /* CUDA ordinal */
  int32_t relaxed;         /* 0 = enforce the reference's parameter ranges */
} sdb_params;

typedef struct sdb_index sdb_index;

/* Thread-local message of the last failing call on this thread. */
const char* sdb_last_error(void);
int sdb_abi_version(void);
/* Number of visible CUDA devices (0 if none / driver missing). */
int sdb_device_count(void);

/* ---- lifecycle: replaces vamana.NewIndexVamana (vamana.go:54-81) / flat.NewIndexFlat
 * (flat.go:21-32). The index owns all device memory. ------------------------ */
int sdb_index_create(const sdb_params* params, sdb_index** out);
void sdb_index_destroy(sdb_index* ix);
/* cache.Cachable.SizeInMemory (vamana.go:83-85): device bytes held. */
int64_t sdb_index_size_bytes(const sdb_index* ix);
/* Pre-size device arrays for node ids <= max_node_id. */
int sdb_index_reserve(sdb_index* ix, uint64_t max_node_id);
uint64_t sdb_index_max_node_id(const sdb_index* ix); /* vamana.go:47 */
uint64_t sdb_index_count(const sdb_index* ix);       /* stored points incl. start node */

/* ---- hydrate / flush: the GPU index mirrors the bucket keys n<id>v / n<id>e
 * (node.go:85-135, plain.go:125-147); the diskstore stays in Go. -------------- */
/* setupStartNode (vamana.go:93-120): the caller supplies node 1's vector. */
int sdb_index_set_start(sdb_index* ix, const float* vec);
/* VectorStore.Set for n points (plain.go:58-66, binary.go:131-139, product.go:161-169):
 * stores raw vectors and, if the quantizer is fitted, their codes. No graph work. */
int sdb_index_set_vectors(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors);
/* Replace the edge lists of n nodes. edges = concatenated lists (the u64 payload of
 * n<id>e, conversion.go:110-124), degrees[i] = length of list i (<= degreeBound). */
int sdb_index_set_edges(sdb_index* ix, uint64_t n, const uint64_t* ids, const uint32_t* degrees,
                        const uint64_t* edges);
/* Read back edge lists; edges_out has n*degreeBound slots, list i at i*degreeBound. */
int sdb_index_get_edges(sdb_index* ix, uint64_t n, const uint64_t* ids, uint32_t* degrees_out,
                        uint64_t* edges_out);
/* Read back raw vectors (n x dim). */
int sdb_index_get_vectors(sdb_index* ix, uint64_t n, const uint64_t* ids, float* out);
/* VectorStore.Delete + nodeStore.Delete bookkeeping (vamana.go:233-238): marks ids absent
 * (edges pointing at them must already be gone). */
int sdb_index_delete(sdb_index* ix, uint64_t n, const uint64_t* ids);

/* ---- search: replaces IndexVamana.Search (vamana.go:278-310) for a batch of B queries.
 * queries: B x dim. k = Limit, search_size = SearchSize (error if < k).
 * filter_ids: optional ascending node ids shared by the batch (search.go:33-51,93-95);
 * filter_ids != NULL means "filtered" even when n_filter == 0 (see sdb_search_batch_filters).
 * out_ids/out_dists: B x k, row b holds out_counts[b] results (start node removed,
 * vamana.go:294-296), remaining slots id 0 / +inf. HybridScore = -dist*weight is left
 * to the caller (vamana.go:303). */
int sdb_search_batch(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, uint32_t search_size,
                     const uint64_t* filter_ids, uint64_t n_filter, uint64_t* out_ids, float* out_dists,
                     uint32_t* out_counts);
/* Per-request filters in one batch (the reference hands every request its own bitmap:
 * shard/index/search.go:59-85 -> vamana/search.go:33-51,93-95). filter f is the ascending id
 * list filter_ids[filter_offsets[f] .. filter_offsets[f+1]); request b uses filter
 * query_filter[b], or none if query_filter[b] < 0 (query_filter == NULL: every request uses
 * filter 0). An EMPTY list is a filter like any other — a non-nil empty bitmap seeds nothing and
 * the request returns no result — so callers whose empty container has a NULL data pointer use
 * this entry point (n_filters >= 1) instead of sdb_search_batch's `filter_ids != NULL` rule.
 * n_filters == 0 = nobody is filtered. Unfiltered requests of a mixed batch run through the
 * same kernels as an unfiltered batch. */
int sdb_search_batch_filters(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, uint32_t search_size,
                             uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                             const int32_t* query_filter, uint64_t* out_ids, float* out_dists, uint32_t* out_counts);
/* Same with device-resident queries/outputs; enqueues on `stream` (cudaStream_t). */
int sdb_search_batch_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint32_t search_size,
                            uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, void* stream);
/* Per-query counters of the most recent search on this handle (nodes expanded, distances
 * evaluated): the terms of the algorithmic-bytes formula, SURVEY.md §8d. Synchronises. */
int sdb_last_search_stats(sdb_index* ix, uint32_t B, uint32_t* hops_out, uint32_t* ndist_out);
/* Kernel timing for the roofline figure: while enabled, every search on the handle brackets its
 * first-pass beam-search kernel with CUDA events on the launching stream (up to 256 searches per
 * enabling; no synchronisation is added). _read waits for the recorded events and returns the
 * per-search kernel durations in ms: *n_out = searches recorded, min(*n_out, cap) values copied. */
int sdb_search_profile(sdb_index* ix, int32_t enable);
int sdb_search_profile_read(sdb_index* ix, uint32_t cap, float* ms_out, uint32_t* n_out);
/* Total kernel launches issued by this handle so far (bench.py's gpu_launches). */
uint64_t sdb_launch_count(const sdb_index* ix);
/* Diagnostic twin of greedySearch's second return value (search.go:100): the visited
 * list (expanded nodes, stably sorted by distance) for each query. vis_cap slots/query. */
int sdb_search_visited(sdb_index* ix, uint32_t B, const float* queries, uint32_t search_size, uint32_t vis_cap,
                       uint64_t* out_vis_ids, float* out_vis_dists, uint32_t* out_vis_len);

/* ---- flat: replaces IndexFlat.Search (flat.go:76-132) for a batch. Scans ids >= 2 in
 * ascending id order (the reference's Go-map order is unspecified; ties: lower id wins). */
int sdb_flat_search_batch(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, const uint64_t* filter_ids,
                          uint64_t n_filter, uint64_t* out_ids, float* out_dists, uint32_t* out_counts);
/* Flat search with one filter per request (shard/index/search.go:59-85 -> flat.go:94-96). The
 * filters follow sdb_search_batch_filters: filter f is filter_ids[filter_offsets[f] ..
 * filter_offsets[f+1]), strictly ascending; request b uses filter query_filter[b], or none if
 * query_filter[b] < 0 (query_filter == NULL: every request uses filter 0); an EMPTY list is a
 * filter and its request returns no result; n_filters == 0 = nobody is filtered. Flat rules:
 *   - an id that is not stored (deleted or never inserted), is >= the allocated rows, or is < 2
 *     is simply never matched — not an error (flat search has no GetMany of seeds);
 *   - unsorted or duplicate ids, or a query_filter index >= n_filters, return SDB_ERR_INVALID;
 *   - k must be 1..75.
 * Row b of the output equals, bit for bit, sdb_flat_search_batch run on query b alone with b's
 * filter (or with none). Each filter takes one of two routes, chosen from its size and its number
 * of requests: its rows gathered by id and scored for each of its requests, or the range scan
 * over the store with its bitmap (sdb_flat_last_filter_stats reports the split). Unfiltered
 * requests of a mixed batch go through the unfiltered pass. sdb_flat_search_batch(filter_ids,
 * n_filter) is the one-filter case: it sorts and de-duplicates the ids, so any order is accepted. */
int sdb_flat_search_batch_filters(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, uint32_t n_filters,
                                  const uint64_t* filter_ids, const uint64_t* filter_offsets, const int32_t* query_filter,
                                  uint64_t* out_ids, float* out_dists, uint32_t* out_counts);
/* Diagnostics of the most recent flat search on this handle: filters (with at least one request)
 * that took the gather route and the range-scan route, and the (request, id) pairs the gather
 * route scored (ids of deleted points included). All 0 after an unfiltered call. */
int sdb_flat_last_filter_stats(sdb_index* ix, uint32_t* gathered_filters, uint32_t* scanned_filters,
                               uint64_t* gathered_pairs);
/* Memory the handle keeps for staging filtered calls: page-locked host bytes (both staging slots and
 * their gather work items) and device bytes (the device copy of a slot). Grow-only; a filter that
 * takes the range scan stages only its ids, offsets and request rows. */
int sdb_filter_staging_bytes(sdb_index* ix, uint64_t* pinned_bytes, uint64_t* device_bytes);

/* Unfiltered flat search with device-resident queries and outputs (the flat twin of
 * sdb_search_batch_device): enqueues everything on `stream` (cudaStream_t) and returns without
 * synchronising; row b equals sdb_flat_search_batch's row b on the same queries, byte for byte.
 * Serves every store the flat search serves (f32 on the tensor-core or exact path, haversine, binary,
 * PQ); a rebuild of the bf16 shadow after a store change runs on `stream` too. d_queries may be
 * page-locked host memory (mapped). k must be 1..75. The first call of a larger shape allocates
 * scratch, which synchronises the device. */
int sdb_flat_search_batch_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint64_t* d_out_ids,
                                 float* d_out_dists, uint32_t* d_out_counts, void* stream);
/* Diagnostics of the most recent flat search on this handle: path = 0 exact CUDA-core
 * scan, 1 tensor-core candidate pass (mma.sync), 2 tensor-core candidate pass (tcgen05 + TMA);
 * candidates = (query, point) pairs the last candidate level kept for exact re-scoring, summed
 * over the batch; overflowed = queries that fell back to the exact scan. With filters, these
 * describe the pass that served the unfiltered requests (all 0 when there were none). After a
 * device-entry call (sdb_flat_search_batch_device, sdb_flat_search_batch_gather_device) this waits
 * for that call to complete on its stream before it reads the counters. */
int sdb_flat_last_stats(sdb_index* ix, int32_t* path, uint64_t* candidates, uint32_t* overflowed);

/* ---- insert: replaces IndexVamana.InsertUpdateDelete's insert branch (vamana.go:136-201,
 * insert.go:16-68): greedySearch + robustPrune + back-edges for n new points, batched. */
int sdb_insert_batch(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors);
/* Same with the n x dim vectors already resident on the index's GPU (bulk loads whose vectors are
 * produced on the device); ids stay on the host. Orders itself after all prior device work. */
int sdb_insert_batch_device(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* d_vectors);
/* Inserts (since creation) whose visited list exceeded the robustPrune candidate capacity (512) and
 * was cut to its first 512 expansions; the reference's list is unbounded. Not an error: the graph
 * stays valid and the call's state is committed. */
uint64_t sdb_insert_truncated(const sdb_index* ix);
/* Running totals of the batched insert since creation (or the last reset), the terms of the build's
 * algorithmic-bytes figure (DESIGN.md K8): out8 = {points inserted, nodes expanded by their
 * searches, distances evaluated by their searches, out-edges written by robustPrune(new), back-edge
 * targets updated, robustPrune(B) runs on saturated targets, candidates of those runs, 0}. */
int sdb_insert_stats(sdb_index* ix, uint64_t* out8, int32_t reset);
/* The whole of IndexVamana.InsertUpdateDelete (vamana.go:136-263) except the trailing Fit and
 * flush: has_vector[i] == 0 stands for a nil vector (IndexVectorChange.Vector == nil,
 * vamana.go:122-125; NULL = all have vectors). Each change is classified against the store
 * (vamana.go:158-185): absent+vector = insert, present+vector = update, present+nil = delete,
 * absent+nil = skipped. Inserts run first (batched); then removeInboundEdges over the
 * updated and deleted ids (EdgeScan node.go:142-199, pruneDeleteNeighbour prune.go:12-84,
 * orphans re-attached to the start node prune.go:137-151); then the deleted rows are dropped
 * and the updated points re-inserted one by one in input order (vamana.go:249-253; batched if
 * the index is `relaxed`). Ids 0 and 1 are errors (vamana.go:150-157). */
int sdb_insert_update_delete(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors,
                             const uint8_t* has_vector);
/* EdgeScan alone (node.go:142-199; vamana_test.go:142-175): ids flagged toPrune / toSave for a
 * delete set, ascending. Buffers need room for sdb_index_max_node_id()+1 ids. */
int sdb_edge_scan(sdb_index* ix, uint64_t n_delete, const uint64_t* delete_ids, uint64_t* to_prune,
                  uint64_t* n_prune, uint64_t* to_save, uint64_t* n_save);
/* Edges of the start node beyond degreeBound (AddNeighbourIfNotExists is unbounded,
 * node.go:73-80): hydrate / flush the tail of n1e. get: *n = count, copies min(*n, cap). */
int sdb_index_get_start_overflow(sdb_index* ix, uint64_t cap, uint64_t* out, uint64_t* n);
int sdb_index_set_start_overflow(sdb_index* ix, uint64_t n, const uint64_t* ids);
/* Ascending ids of the nodes whose edge list changed since the last clearing call (the
 * graphNode.isDirty / CheckAndClearDirty protocol of ItemCache.Flush, node.go:17,104-110,
 * itemcache.go:236): what nodeStore.Flush must rewrite under n<id>e. *n = how many are dirty;
 * copies min(*n, cap); flags are cleared only if clear != 0 and everything fitted. */
int sdb_index_dirty_edges(sdb_index* ix, uint64_t cap, uint64_t* ids_out, uint64_t* n_out, int32_t clear);
/* Mini-batch schedule of the batched insert: batch b has min(max_batch, max(min_batch,
 * inserted_so_far / growth_div)) points. 0 keeps a field's default (min 1; max / growth_div
 * 32768 / 8 while the rows the searches read are at most 512 bytes wide, else 16384 / 16).
 * 1, 1, x is the reference's sequential schedule (the oracle's graph edge for edge). */
int sdb_insert_config(sdb_index* ix, uint32_t min_batch, uint32_t max_batch, uint32_t growth_div);

/* ---- quantizers: replaces VectorStore.Fit (vamana.go:258): binaryQuantizer.Fit
 * (binary.go:145-185) / productQuantizer.Fit (product.go:175-236). pq_first_row = index
 * (in ascending id order) of the first k-means centre (kmeans.go:61 draws it at random).
 * Returns via *fitted whether a fit happened (0 = skipped: already fitted / below trigger). */
int sdb_index_fit(sdb_index* ix, uint64_t pq_first_row, int32_t* fitted);
/* PQ state (product.go:36-37): flatCentroids M*K*sub, centroidDists M*K*K. */
int sdb_index_get_pq(sdb_index* ix, float* flat_centroids, float* centroid_dists);
int sdb_index_set_pq(sdb_index* ix, const float* flat_centroids, const float* centroid_dists);
/* BQ threshold vector (binary.go:28), dim floats. */
int sdb_index_get_bq_threshold(sdb_index* ix, float* threshold);
int sdb_index_set_bq_threshold(sdb_index* ix, const float* threshold);
/* Stored codes of n points: PQ -> M bytes each; BQ -> ceil(dim/64) u64 each (LE bytes). */
int sdb_index_get_codes(sdb_index* ix, uint64_t n, const uint64_t* ids, uint8_t* out);
/* Hydrate quantized points from their n<id>q payload alone (binary.go:275-296, product.go:
 * 349-371: once a point has codes its raw vector is no longer loaded). Same layout as
 * sdb_index_get_codes; the quantizer must be fitted (sdb_index_set_pq / set_bq_threshold). */
int sdb_index_set_codes(sdb_index* ix, uint64_t n, const uint64_t* ids, const uint8_t* codes);

/* ---- distance family (distance/distance.go:11-12 FloatDistFunc / BitDistFunc), batched:
 * out[i] = dist(x[i], y[i]) for n pairs of dim floats / `words` u64 words. */
int sdb_distance_float(int32_t metric, int32_t device, uint64_t n, uint32_t dim, const float* x, const float* y,
                       float* out);
int sdb_distance_bits(int32_t metric, int32_t device, uint64_t n, uint32_t words, const uint64_t* x,
                      const uint64_t* y, float* out);
/* Store-level closures, batched: DistanceFromFloat(query)(ids[i]) (plain.go:76, binary.go:187,
 * product.go:238) and DistanceFromPoint(x)(ids[i]) (plain.go:87, binary.go:213, product.go:279). */
int sdb_index_query_dists(sdb_index* ix, const float* query, uint64_t n, const uint64_t* ids, float* out);
int sdb_index_point_dists(sdb_index* ix, uint64_t x, uint64_t n, const uint64_t* ids, float* out);
/* binaryQuantizer.encode (binary.go:103-129) for n vectors; out n x ceil(dim/64) u64. */
int sdb_bq_encode(int32_t device, uint64_t n, uint32_t dim, const float* vectors, const float* threshold,
                  uint64_t* out);
/* ADC table of DistanceFromFloat (product.go:255-263) for B queries: B x M x K floats. */
int sdb_pq_adc_tables(sdb_index* ix, uint32_t B, const float* queries, float* out);

/* ---- cross-shard merge: replaces the sort+truncate of ClusterNode.SearchPoints
 * (cluster/actions.go:357-376). in_*: S x B x k (shard-major), counts S x B. Sorted by
 * distance ascending (= HybridScore descending); ties: lower shard, then lower rank. */
int sdb_merge_topk(int32_t device, uint32_t S, uint32_t B, uint32_t k, const uint64_t* in_ids,
                   const float* in_dists, const uint32_t* in_counts, uint64_t* out_ids, float* out_dists,
                   uint32_t* out_counts);
int sdb_merge_topk_device(int32_t device, uint32_t S, uint32_t B, uint32_t k, const uint64_t* d_in_ids,
                          const float* d_in_dists, const uint32_t* d_in_counts, uint64_t* d_out_ids,
                          float* d_out_dists, uint32_t* d_out_counts, void* stream);
/* ---- hybrid-score merge: replaces the dedupe-and-add + sort of indexManager.searchParallel
 * (shard/index/search.go:211-298) for B requests of S sub-searches each (an "_and" / "_or" query
 * whose members are vector searches). in_*: S x B x k (sub-search-major), counts S x B;
 * in_hybrid = HybridScore (-distance * weight, vamana.go:303), in_dists NaN = no distance.
 * disjunction != 0: "_or" (union of the result-id sets), else "_and" (ids present in every
 * sub-search). A node found again adds its HybridScore to its first occurrence. out_*: B x (S*k),
 * sorted by HybridScore descending (ties: first-appearance order), padded with id 0 / -inf / +inf. */
int sdb_hybrid_merge(int32_t device, uint32_t S, uint32_t B, uint32_t k, int32_t disjunction, const uint64_t* in_ids,
                     const float* in_hybrid, const float* in_dists, const uint32_t* in_counts, uint64_t* out_ids,
                     float* out_hybrid, float* out_dists, uint32_t* out_counts);

/* ---- cross-shard exchange fused into the search kernel (replaces the fan-in of
 * ClusterNode.SearchPoints, cluster/actions.go:316-376, without a separate collective).
 * Every GPU owns a gather buffer ids[S][B][k] / dists[S][B][k] / counts[S][B] that its peers
 * can write: peer-mapped device pointers (cudaDeviceEnablePeerAccess inside one process, CUDA
 * IPC / symmetric memory between processes). sdb_search_batch_gather_device runs the beam
 * search on this GPU's shard and its epilogue stores each query's top-k, node ids tagged as
 * (shard << 40 | id), into slot [shard][query] of EVERY peer's buffer over NVLink.
 * sdb_peer_barrier_device then publishes `epoch` to every peer's flag word [me] and waits for
 * every peer's epoch in its own words (flags: >= 2*SDB_MAX_PEERS u32 per GPU, zeroed once;
 * epochs must grow by 1 per step), after which sdb_merge_topk_device reads the local gather
 * buffer. Callers alternate two gather buffers (epoch parity) so a fast peer's next step
 * cannot overwrite a buffer still being merged. */
#define SDB_MAX_PEERS 16
typedef struct sdb_peer_gather {
  uint32_t n_peers;          /* destination GPUs, this one included (= S with one shard per GPU) */
  uint32_t shard;            /* shard index of this search: slot [shard] of every buffer, tag of its ids */
  uint32_t per_shard_limit;  /* sdb_shard_limit(k, S, ...); 0 = k */
  uint32_t reserved;
  uint64_t* ids[SDB_MAX_PEERS];     /* peer p's ids    [S][B][k] */
  float* dists[SDB_MAX_PEERS];      /* peer p's dists  [S][B][k] */
  uint32_t* counts[SDB_MAX_PEERS];  /* peer p's counts [S][B] */
} sdb_peer_gather;
int sdb_search_batch_gather_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint32_t search_size,
                                   uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                                   const sdb_peer_gather* peers, void* stream);
/* Flat shards: sdb_flat_search_batch_device on this GPU's shard, then one kernel stores every
 * query's final list (the exact fallback of overflowed queries included) into slot [shard][query]
 * of EVERY peer's buffer, byte for byte what the beam-search epilogue stores: ids (shard << 40 | id)
 * and distances of the first count ranks, id 0 and +inf in the other slots, count
 * min(count, per_shard_limit or k). Same argument checks and SDB_ERR_STATE refusal as
 * sdb_search_batch_gather_device; k must be 1..75. Unfiltered; no synchronisation. */
int sdb_flat_search_batch_gather_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k,
                                        uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                                        const sdb_peer_gather* peers, void* stream);
/* Filtered shard search with device-resident queries and outputs, enqueued on `stream`.
 * The filter arguments are those of sdb_search_batch_filters / sdb_flat_search_batch_filters, in
 * host memory; they are copied before the call returns, so the caller may free or reuse them at
 * once (cgo: Go memory is not retained). Filters are shard-local ids: each shard gets its own lists.
 * A request filtered on one shard must be filtered on every shard (its list there may be empty);
 * the library cannot check this across shards.
 *   - Row b of the outputs equals row b of the matching host filter entry, byte for byte, on every
 *     store each serves (beam search: f32 L2 / dot / cosine, haversine, binary, PQ; flat search:
 *     the same stores, on both routes). n_filters == 0 gives the bytes of sdb_search_batch_device /
 *     sdb_flat_search_batch_device (with peers: of the _gather_device entry).
 *   - peers == NULL: no exchange. Otherwise every query's final list also goes into slot
 *     [shard][query] of every peer's buffer, with the bytes the _gather_device entries store
 *     (tagged ids, id 0 / +inf past the count, count clamped to per_shard_limit).
 *   - Checks, in order: those of the host filter entry and their error codes (unsorted ids, a
 *     query_filter index >= n_filters, missing seeds = SDB_ERR_NOTFOUND for the beam search,
 *     searchSize < k, k outside 1..75 for flat search); then those of the _gather_device entry on
 *     `peers`; then its SDB_ERR_STATE refusal after a timed-out barrier. A failed call enqueues
 *     nothing.
 *   - No host synchronisation: the filters go to the device through one of two page-locked
 *     staging slots of the handle; the host waits only before refilling a slot whose copy (two
 *     filtered calls ago) has not run yet. A filtered call on any stream waits, on the device, for
 *     the previous filtered call on the handle to finish reading the lists it overwrites. The
 *     first call of a larger shape allocates scratch, which synchronises the device. */
int sdb_search_batch_filters_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint32_t search_size,
                                    uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                                    const int32_t* query_filter, uint64_t* d_out_ids, float* d_out_dists,
                                    uint32_t* d_out_counts, const sdb_peer_gather* peers, void* stream);
int sdb_flat_search_batch_filters_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k,
                                         uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                                         const int32_t* query_filter, uint64_t* d_out_ids, float* d_out_dists,
                                         uint32_t* d_out_counts, const sdb_peer_gather* peers, void* stream);
/* ---- per-request parameters: the reference gives every request its own Limit and SearchSize
 * (models/search.go:268-314) as it gives every request its own filter. One batch serves any mix.
 *   - Outputs are B x k_stride: row b holds out_counts[b] <= req[b].limit results, every other slot
 *     is id 0 / +inf. Row b equals, byte for byte, the row the matching filter entry returns for
 *     request b alone with k = req[b].limit, search_size = req[b].search_size and b's filter
 *     (slots past the limit padded). A req array whose entries share one (limit, search_size), with
 *     k_stride = limit, gives the bytes of the filter entry on the same batch.
 *   - filter = index into the filters (sdb_search_batch_filters' filter_ids / filter_offsets), -1 =
 *     unfiltered; n_filters may be 0 when no request is filtered.
 *   - Checks, before anything is enqueued: every limit is 1..75, every search_size 25..75 (1..75 on a
 *     `relaxed` index; ignored by flat search), limit > search_size = SDB_ERR_SEARCHSIZE, limit >
 *     k_stride or k_stride > 75 = SDB_ERR_INVALID, then the checks of the filter entries. The seeds
 *     of a filtered request are the first min(n_f, its search_size) ids of its filter, so requests
 *     sharing a filter may have different seeds; the existence check of a filter's seeds covers the
 *     largest search_size of the requests that use it (the batch's largest for a filter none uses).
 *     A failed call enqueues nothing and leaves the outputs untouched.
 *   - With peers, slot [shard][b] of every peer buffer (stride k_stride) gets request b's tagged ids,
 *     count clamped to shard_limit (0 = limit); peers->per_shard_limit is ignored.
 *   - Flat search runs the batch at k = k_stride and cuts every row to its limit: the exact top-k by
 *     (distance, id) at a smaller k is a prefix of it.
 *   - Staging: req travels with the filters through the handle's page-locked slots (an unfiltered
 *     batch uses a slot too); the _device entries do no host synchronisation and copy req and the
 *     filters before returning. */
typedef struct sdb_request {
  uint32_t limit;        /* k of this request, 1..75 */
  uint32_t search_size;  /* L of this request (beam search; ignored by flat search) */
  uint32_t shard_limit;  /* with peers: ranks published into the gather buffers, 0 = limit */
  int32_t filter;        /* index into the filters, -1 = unfiltered (below -1: SDB_ERR_INVALID) */
} sdb_request;
int sdb_search_batch_requests(sdb_index* ix, uint32_t B, const float* queries, const sdb_request* req, uint32_t n_filters,
                              const uint64_t* filter_ids, const uint64_t* filter_offsets, uint32_t k_stride,
                              uint64_t* out_ids, float* out_dists, uint32_t* out_counts);
int sdb_search_batch_requests_device(sdb_index* ix, uint32_t B, const float* d_queries, const sdb_request* req,
                                     uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                                     uint32_t k_stride, uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                                     const sdb_peer_gather* peers, void* stream);
int sdb_flat_search_batch_requests(sdb_index* ix, uint32_t B, const float* queries, const sdb_request* req,
                                   uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                                   uint32_t k_stride, uint64_t* out_ids, float* out_dists, uint32_t* out_counts);
int sdb_flat_search_batch_requests_device(sdb_index* ix, uint32_t B, const float* d_queries, const sdb_request* req,
                                          uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                                          uint32_t k_stride, uint64_t* d_out_ids, float* d_out_dists,
                                          uint32_t* d_out_counts, const sdb_peer_gather* peers, void* stream);
/* sdb_merge_topk_device with one output limit per request: d_limits[b] (device, 1..k_stride) bounds
 * row b's merged list; inputs S x B x k_stride, outputs B x k_stride padded with id 0 / +inf. */
int sdb_merge_topk_requests_device(int32_t device, uint32_t S, uint32_t B, uint32_t k_stride, const uint32_t* d_limits,
                                   const uint64_t* d_in_ids, const float* d_in_dists, const uint32_t* d_in_counts,
                                   uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, void* stream);
int sdb_peer_barrier_device(int32_t device, uint32_t n_peers, uint32_t me, uint32_t* const* peer_flags, uint32_t epoch,
                            void* stream);
/* A peer that never arrives is given ~20 s; the barrier kernel then records the timeout in a
 * page-locked status word of its device. From then on sdb_peer_barrier_device,
 * sdb_search_batch_gather_device, sdb_flat_search_batch_gather_device and sdb_merge_topk_device on
 * that device fail with SDB_ERR_STATE
 * (the step whose barrier timed out merged stale slots). sdb_peer_barrier_check reads the word
 * (no synchronisation: call it after synchronising the step's stream to validate that step) and
 * returns SDB_OK or SDB_ERR_STATE; clear != 0 resets it once the caller has recovered. */
int sdb_peer_barrier_check(int32_t device, int32_t clear);
/* Per-shard request limit (cluster/actions.go:291-299). Pure host arithmetic. */
uint32_t sdb_shard_limit(uint32_t limit, uint32_t n_shards, uint32_t max_search_limit);

#ifdef __cplusplus
}
#endif
#endif /* SEMADB_B200_H */
