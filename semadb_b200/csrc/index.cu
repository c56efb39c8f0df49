// index.cu — handle management and the C-ABI entry points (include/semadb_b200.h).
#include "index.cuh"

#include <algorithm>
#include <cstring>
#include <limits>

#include "common.cuh"

namespace sdb {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + what;
  cudaGetLastError();  // clear sticky-less errors
  return e == cudaErrorMemoryAllocation ? SDB_ERR_OOM : SDB_ERR_CUDA;
}

// ---- small device kernels for hydrate / flush --------------------------------------
__global__ void scatter_vectors_kernel(float* vec, uint32_t pitch, uint8_t* exists, const uint32_t* ids,
                                       const float* src, uint32_t dim, uint32_t n) {
  uint32_t r = blockIdx.x;
  if (r >= n) return;
  uint32_t id = ids[r];
  float* dst = vec + size_t(id) * pitch;
  for (uint32_t i = threadIdx.x; i < pitch; i += blockDim.x) dst[i] = i < dim ? src[size_t(r) * dim + i] : 0.0f;
  if (threadIdx.x == 0) exists[id] = 1;
}
__global__ void gather_vectors_kernel(const float* vec, uint32_t pitch, const uint32_t* ids, float* dst, uint32_t dim,
                                      uint32_t n) {
  uint32_t r = blockIdx.x;
  if (r >= n) return;
  const float* src = vec + size_t(ids[r]) * pitch;
  for (uint32_t i = threadIdx.x; i < dim; i += blockDim.x) dst[size_t(r) * dim + i] = src[i];
}
__global__ void scatter_edges_kernel(uint32_t* adj, uint32_t* deg, uint32_t R, const uint32_t* ids,
                                     const uint32_t* rows /*n x R padded*/, const uint32_t* degs, uint32_t n) {
  uint32_t r = blockIdx.x;
  if (r >= n) return;
  uint32_t id = ids[r];
  for (uint32_t i = threadIdx.x; i < R; i += blockDim.x) adj[size_t(id) * R + i] = rows[size_t(r) * R + i];
  if (threadIdx.x == 0) deg[id] = degs[r];
}
__global__ void gather_edges_kernel(const uint32_t* adj, const uint32_t* deg, uint32_t R, const uint32_t* ids,
                                    uint32_t* rows, uint32_t* degs, uint32_t n) {
  uint32_t r = blockIdx.x;
  if (r >= n) return;
  uint32_t id = ids[r];
  for (uint32_t i = threadIdx.x; i < R; i += blockDim.x) rows[size_t(r) * R + i] = adj[size_t(id) * R + i];
  if (threadIdx.x == 0) degs[r] = deg[id];
}
// code rows (PQ bytes / bit words) <-> a dense staging buffer: one thread per byte
__global__ void scatter_codes_kernel(uint8_t* base, uint32_t pitch, uint32_t width, uint8_t* exists, const uint32_t* ids,
                                     const uint8_t* src, uint64_t n) {
  const uint64_t t = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= n * width) return;
  const uint64_t r = t / width;
  const uint32_t c = uint32_t(t % width);
  const uint32_t id = ids[r];
  base[size_t(id) * pitch + c] = src[t];
  if (c == 0) exists[id] = 1;
}
__global__ void gather_codes_kernel(const uint8_t* base, uint32_t pitch, uint32_t width, const uint32_t* ids, uint8_t* dst,
                                    uint64_t n) {
  const uint64_t t = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= n * width) return;
  dst[t] = base[size_t(ids[t / width]) * pitch + uint32_t(t % width)];
}
__global__ void fill_u32_kernel(uint32_t* p, uint32_t v, size_t n) {
  size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t stride = size_t(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

template <class T>
static int grow(T** p, size_t old_elems, size_t new_elems, cudaStream_t s, bool fill_ff = false) {
  T* np_ = nullptr;
  SDB_CUDA(cudaMalloc(reinterpret_cast<void**>(&np_), new_elems * sizeof(T)));
  if (fill_ff) SDB_CUDA(cudaMemsetAsync(np_, 0xFF, new_elems * sizeof(T), s));
  else SDB_CUDA(cudaMemsetAsync(np_, 0, new_elems * sizeof(T), s));
  if (*p && old_elems) SDB_CUDA(cudaMemcpyAsync(np_, *p, old_elems * sizeof(T), cudaMemcpyDeviceToDevice, s));
  SDB_CUDA(cudaStreamSynchronize(s));
  if (*p) cudaFree(*p);
  *p = np_;
  return SDB_OK;
}

int index_reserve_locked(sdb_index* ix, uint64_t max_node_id) {
  if (max_node_id >= (uint64_t(1) << 31) - 1) return fail(SDB_ERR_INVALID, "node id too large for a device index (>= 2^31-1)");
  uint64_t need = max_node_id + 1;
  if (need <= ix->rows) return SDB_OK;
  uint64_t nr = std::max<uint64_t>(need, std::max<uint64_t>(uint64_t(ix->rows) * 3 / 2, 1024));
  nr = std::min<uint64_t>(nr, (uint64_t(1) << 31) - 1);
  size_t o = ix->rows, n = size_t(nr);
  int rc;
  if ((rc = grow(&ix->d_vec, o * ix->vec_pitch, n * ix->vec_pitch, ix->stream))) return rc;
  if (ix->p.quantizer == SDB_QUANT_BINARY && (rc = grow(&ix->d_bits, o * ix->bits_pitch, n * ix->bits_pitch, ix->stream))) return rc;
  if (ix->p.quantizer == SDB_QUANT_PRODUCT && (rc = grow(&ix->d_codes, o * ix->codes_pitch, n * ix->codes_pitch, ix->stream))) return rc;
  if ((rc = grow(&ix->d_adj, o * ix->p.degree_bound, n * ix->p.degree_bound, ix->stream, true))) return rc;
  if ((rc = grow(&ix->d_deg, o, n, ix->stream))) return rc;
  if ((rc = grow(&ix->d_exists, o, n, ix->stream))) return rc;
  if ((rc = grow(&ix->d_dirty, o, n, ix->stream))) return rc;
  ix->h_exists.resize(n, 0);
  ix->rows = uint32_t(n);
  ix->vec_epoch++;
  return SDB_OK;
}

int set_rows_device(sdb_index* ix, uint32_t n, const uint32_t* d_ids, const float* d_vecs, cudaStream_t stream) {
  if (n == 0) return SDB_OK;
  ix->vec_epoch++;
  scatter_vectors_kernel<<<n, 128, 0, stream>>>(ix->d_vec, ix->vec_pitch, ix->d_exists, d_ids, d_vecs, ix->p.dim, n);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  if (ix->quant_active()) return launch_encode_rows(ix, n, d_ids, stream);
  return SDB_OK;
}

static int validate(const sdb_params& p) {
  if (p.dim < 1 || p.dim > MAX_DIM) return fail(SDB_ERR_INVALID, "vector size must be between 1 and 4096");  // models/index.go:285
  if (p.metric < SDB_METRIC_EUCLIDEAN || p.metric > SDB_METRIC_HAVERSINE) return fail(SDB_ERR_INVALID, "unknown distance metric");
  if (p.metric == SDB_METRIC_HAVERSINE && p.dim != 2) return fail(SDB_ERR_INVALID, "haversine distance metric requires vector size 2");
  if (p.search_size > 75 || p.degree_bound > 64) return fail(SDB_ERR_INVALID, "searchSize must be <= 75 and degreeBound <= 64");
  if (p.search_size < 1 || p.degree_bound < 1) return fail(SDB_ERR_INVALID, "searchSize and degreeBound must be positive");
  if (!p.relaxed) {
    if (p.search_size < 25) return fail(SDB_ERR_INVALID, "search size must be between 25 and 75");  // models/index.go:299
    if (p.degree_bound < 32) return fail(SDB_ERR_INVALID, "degree bound must be between 32 and 64");
    if (!(p.alpha >= 1.1f && p.alpha <= 1.5f)) return fail(SDB_ERR_INVALID, "alpha must be between 1.1 and 1.5");
  }
  if (p.quantizer < SDB_QUANT_NONE || p.quantizer > SDB_QUANT_PRODUCT) return fail(SDB_ERR_INVALID, "unknown quantizer type");
  bool bitmetric = p.metric == SDB_METRIC_HAMMING || p.metric == SDB_METRIC_JACCARD;
  if (p.quantizer == SDB_QUANT_BINARY && !bitmetric) {
    if (p.bq_metric != SDB_METRIC_HAMMING && p.bq_metric != SDB_METRIC_JACCARD)
      return fail(SDB_ERR_INVALID, "invalid distance metric for binary quantization");  // models/quantizer.go:45
    if (std::isnan(p.bq_threshold) && !p.relaxed && p.bq_trigger > 50000)
      return fail(SDB_ERR_INVALID, "triggerThreshold must be between 0 and 50000");
  }
  if (p.quantizer == SDB_QUANT_PRODUCT && !bitmetric) {
    if (p.pq_centroids < 2 || p.pq_centroids > 256) return fail(SDB_ERR_INVALID, "numCentroids must be between 2 and 256");
    if (p.pq_subvectors < (p.relaxed ? 1u : 2u)) return fail(SDB_ERR_INVALID, "numSubVectors must be at least 2");
    if (p.dim % p.pq_subvectors != 0) return fail(SDB_ERR_INVALID, "vector length must be divisible by num subvectors");  // product.go:44
    if (p.metric != SDB_METRIC_EUCLIDEAN && p.metric != SDB_METRIC_COSINE && p.metric != SDB_METRIC_DOT)
      return fail(SDB_ERR_INVALID, "distance function not supported for product quantisation");  // product.go:48
    if (!p.relaxed && (p.pq_trigger < 1000 || p.pq_trigger > 10000))
      return fail(SDB_ERR_INVALID, "triggerThreshold must be between 1000 and 10000");
  }
  return SDB_OK;
}

// ids (u64, host) -> validated u32 on device scratch d_tmp32[0..n)
static int stage_ids(sdb_index* ix, uint64_t n, const uint64_t* ids, bool must_exist, bool grow_rows,
                     std::vector<uint32_t>& h32) {
  h32.resize(n);
  uint64_t mx = 0;
  for (uint64_t i = 0; i < n; ++i) {
    if (ids[i] == 0) return fail(SDB_ERR_INVALID, "invalid point id: 0");
    if (ids[i] >= (uint64_t(1) << 31) - 1) return fail(SDB_ERR_INVALID, "node id too large for a device index");
    mx = std::max(mx, ids[i]);
    h32[i] = uint32_t(ids[i]);
  }
  if (grow_rows) {
    int rc = index_reserve_locked(ix, mx);
    if (rc) return rc;
  }
  if (must_exist)
    for (uint64_t i = 0; i < n; ++i)
      if (h32[i] >= ix->rows || !ix->h_exists[h32[i]]) return fail(SDB_ERR_NOTFOUND, "node id does not exist: " + std::to_string(ids[i]));
  int rc = ix->d_tmp32.ensure(n + 1);
  if (rc) return rc;
  SDB_CUDA(cudaMemcpyAsync(ix->d_tmp32.p, h32.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, ix->stream));
  return SDB_OK;
}

}  // namespace sdb

using namespace sdb;

extern "C" {

const char* sdb_last_error(void) { return g_err.c_str(); }
int sdb_abi_version(void) { return SDB_ABI_VERSION; }
int sdb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int sdb_index_create(const sdb_params* params, sdb_index** out) {
  if (!params || !out) return fail(SDB_ERR_INVALID, "null argument");
  *out = nullptr;
  sdb_params p = *params;
  // vectorstore.go:56-66: hamming/jaccard force the binary quantizer with threshold 0.5
  if (p.metric == SDB_METRIC_HAMMING || p.metric == SDB_METRIC_JACCARD) {
    p.quantizer = SDB_QUANT_BINARY;
    p.bq_metric = p.metric;
    p.bq_threshold = 0.5f;
  }
  int rc = validate(p);
  if (rc) return rc;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(SDB_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
  }
  if (p.device < 0 || p.device >= ndev) return fail(SDB_ERR_INVALID, "device ordinal out of range");
  SDB_CUDA(cudaSetDevice(p.device));
  sdb_index* ix = new (std::nothrow) sdb_index;
  if (!ix) return fail(SDB_ERR_OOM, "host allocation failed");
  ix->p = p;
  ix->device = p.device;
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, p.device)) != cudaSuccess) {
    delete ix;
    return cuda_fail(e, "cudaGetDeviceProperties");
  }
  if (prop.major < 10) {
    delete ix;
    return fail(SDB_ERR_CUDA, "device is not sm_100 (this library is built for sm_100a only)");
  }
  ix->sm_count = prop.multiProcessorCount;
  ix->smem_optin = prop.sharedMemPerBlockOptin;
  ix->smem_per_sm = prop.sharedMemPerMultiprocessor;
  if ((e = cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    delete ix;
    return cuda_fail(e, "cudaStreamCreate");
  }
  for (cudaEvent_t* ev : {&ix->fstage_ev[0], &ix->fstage_ev[1], &ix->filter_done_ev})
    if ((e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming)) != cudaSuccess) {
      sdb_index_destroy(ix);
      return cuda_fail(e, "cudaEventCreate");
    }
  ix->vec_pitch = (p.dim + 3) / 4 * 4;
  ix->words = (p.dim + 63) / 64;
  ix->bits_pitch = (ix->words + 1) / 2 * 2;
  ix->store_metric = p.metric;
  if (p.quantizer == SDB_QUANT_BINARY) {
    ix->bq_metric = p.bq_metric;
    if ((e = cudaMalloc(reinterpret_cast<void**>(&ix->d_bq_thr), p.dim * sizeof(float))) != cudaSuccess) {
      sdb_index_destroy(ix);
      return cuda_fail(e, "cudaMalloc(bq threshold)");
    }
    if (!std::isnan(p.bq_threshold)) {
      std::vector<float> thr(p.dim, p.bq_threshold);
      cudaMemcpy(ix->d_bq_thr, thr.data(), p.dim * sizeof(float), cudaMemcpyHostToDevice);
      ix->bq_fitted = true;
    }
  }
  if (p.quantizer == SDB_QUANT_PRODUCT) {
    ix->pqM = p.pq_subvectors;
    ix->pqK = p.pq_centroids;
    ix->pqSub = p.dim / p.pq_subvectors;
    ix->codes_pitch = (ix->pqM + 15) / 16 * 16;
    if (p.metric == SDB_METRIC_COSINE) ix->store_metric = SDB_METRIC_EUCLIDEAN;  // product.go:52-61
  }
  rc = index_reserve_locked(ix, 1023);
  if (rc) {
    sdb_index_destroy(ix);
    return rc;
  }
  *out = ix;
  return SDB_OK;
}

void sdb_index_destroy(sdb_index* ix) {
  if (!ix) return;
  cudaSetDevice(ix->device);
  if (ix->stream) cudaStreamSynchronize(ix->stream);
  cudaFree(ix->d_vec);
  cudaFree(ix->d_bits);
  cudaFree(ix->d_codes);
  cudaFree(ix->d_adj);
  cudaFree(ix->d_deg);
  cudaFree(ix->d_exists);
  cudaFree(ix->d_dirty);
  ix->d_start_extra.release();
  ix->d_x16.release(); ix->d_q16.release(); ix->d_xn.release(); ix->d_bias.release(); ix->d_mu.release(); ix->d_gmin.release(); ix->d_xmax.release(); ix->d_qn.release(); ix->d_thr.release();
  ix->d_sample_d.release(); ix->d_cand.release(); ix->d_candcnt.release(); ix->d_sample_cnt.release(); ix->d_sample_ids.release();
  cudaFree(ix->d_bq_thr);
  cudaFree(ix->d_pq_centroids);
  cudaFree(ix->d_pq_cdist);
  cudaFree(ix->d_ins_stats);
  ix->d_q.release(); ix->d_oid.release(); ix->d_od.release(); ix->d_oc.release(); ix->d_hops.release();
  ix->d_ndist.release(); ix->d_work.release(); ix->d_adc.release(); ix->d_fstage.release();
  ix->d_filter_bits.release(); ix->d_retry_bitmap.release(); ix->d_vis_ids.release(); ix->d_vis_len.release(); ix->d_vis_d.release();
  ix->d_ids64.release(); ix->d_tmp32.release(); ix->d_tmpf.release(); ix->d_tmp8.release();
  ix->d_fg_part32.release(); ix->d_fsub_cnt.release(); ix->d_fg_partf.release(); ix->d_fsub_q.release(); ix->d_fsub_d.release();
  ix->d_fsub_ids.release();
  for (auto& h : ix->h_stage) h.release();
  for (auto& h : ix->h_stage_items) h.release();
  ix->h_flat_misc.release();
  if (ix->flat_stats_ev) cudaEventDestroy(ix->flat_stats_ev);
  for (cudaEvent_t e : {ix->fstage_ev[0], ix->fstage_ev[1], ix->filter_done_ev})
    if (e) cudaEventDestroy(e);
  for (auto& e : ix->prof_ev)
    if (e) cudaEventDestroy(e);
  if (ix->stream) cudaStreamDestroy(ix->stream);
  cudaGetLastError();
  delete ix;
}

int64_t sdb_index_size_bytes(const sdb_index* ix) {
  if (!ix) return 0;
  std::lock_guard<std::mutex> g(ix->mu);
  int64_t r = ix->rows;
  int64_t b = r * ix->vec_pitch * 4 + r * ix->p.degree_bound * 4 + r * 4 + r;
  if (ix->d_bits) b += r * ix->bits_pitch * 8;
  if (ix->d_codes) b += r * ix->codes_pitch;
  if (ix->d_pq_centroids) b += int64_t(ix->pqM) * ix->pqK * ix->pqSub * 4 + int64_t(ix->pqM) * ix->pqK * ix->pqK * 4;
  return b;
}

int sdb_index_reserve(sdb_index* ix, uint64_t max_node_id) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  return index_reserve_locked(ix, max_node_id);
}
uint64_t sdb_index_max_node_id(const sdb_index* ix) { return ix ? ix->max_node_id : 0; }
uint64_t sdb_index_count(const sdb_index* ix) { return ix ? ix->count : 0; }
uint64_t sdb_launch_count(const sdb_index* ix) { return ix ? ix->launches : 0; }

static int set_vectors_locked(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors, bool allow_start) {
  if (n == 0) return SDB_OK;
  if (!ids || !vectors) return fail(SDB_ERR_INVALID, "null argument");
  std::vector<uint32_t> h32;
  if (!allow_start)
    for (uint64_t i = 0; i < n; ++i)
      if (ids[i] == START_ID) return fail(SDB_ERR_RESERVED_ID, "cannot modify point with start id: 1");
  int rc = stage_ids(ix, n, ids, false, true, h32);
  if (rc) return rc;
  size_t bytes = size_t(n) * ix->p.dim * sizeof(float);
  if ((rc = ix->d_tmpf.ensure(size_t(n) * ix->p.dim))) return rc;
  SDB_CUDA(cudaMemcpyAsync(ix->d_tmpf.p, vectors, bytes, cudaMemcpyHostToDevice, ix->stream));
  ix->vec_epoch++;
  scatter_vectors_kernel<<<uint32_t(n), 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, ix->d_exists, ix->d_tmp32.p,
                                                              ix->d_tmpf.p, ix->p.dim, uint32_t(n));
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  if (ix->quant_active()) {
    if ((rc = launch_encode_rows(ix, uint32_t(n), ix->d_tmp32.p, ix->stream))) return rc;
  }
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  for (uint64_t i = 0; i < n; ++i) {
    if (!ix->h_exists[h32[i]]) {
      ix->h_exists[h32[i]] = 1;
      ix->count++;
    }
    if (h32[i] != START_ID && h32[i] > ix->max_node_id) ix->max_node_id = h32[i];
  }
  return SDB_OK;
}

int sdb_index_set_start(sdb_index* ix, const float* vec) {
  if (!ix || !vec) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  uint64_t id = START_ID;
  return set_vectors_locked(ix, 1, &id, vec, true);
}

int sdb_index_set_vectors(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  // chunk to bound staging memory
  const uint64_t chunk = std::max<uint64_t>(1, (uint64_t(256) << 20) / (ix->p.dim * sizeof(float)));
  for (uint64_t s = 0; s < n; s += chunk) {
    uint64_t m = std::min(chunk, n - s);
    int rc = set_vectors_locked(ix, m, ids + s, vectors + s * ix->p.dim, true);
    if (rc) return rc;
  }
  return SDB_OK;
}

int sdb_index_get_vectors(sdb_index* ix, uint64_t n, const uint64_t* ids, float* out) {
  if (!ix || (n && (!ids || !out))) return fail(SDB_ERR_INVALID, "null argument");
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  std::vector<uint32_t> h32;
  int rc = stage_ids(ix, n, ids, true, false, h32);
  if (rc) return rc;
  if ((rc = ix->d_tmpf.ensure(size_t(n) * ix->p.dim))) return rc;
  gather_vectors_kernel<<<uint32_t(n), 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, ix->d_tmp32.p, ix->d_tmpf.p,
                                                             ix->p.dim, uint32_t(n));
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaMemcpyAsync(out, ix->d_tmpf.p, size_t(n) * ix->p.dim * sizeof(float), cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  return SDB_OK;
}

int sdb_index_set_edges(sdb_index* ix, uint64_t n, const uint64_t* ids, const uint32_t* degrees,
                        const uint64_t* edges) {
  if (!ix || (n && (!ids || !degrees))) return fail(SDB_ERR_INVALID, "null argument");
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  const uint32_t R = ix->p.degree_bound;
  const uint64_t chunk = 1 << 20;
  size_t off = 0;
  std::vector<uint32_t> h32, rows, degs;
  for (uint64_t s = 0; s < n; s += chunk) {
    uint64_t m = std::min(chunk, n - s);
    int rc = stage_ids(ix, m, ids + s, false, true, h32);
    if (rc) return rc;
    rows.assign(size_t(m) * R, INVALID_ID);
    degs.resize(m);
    for (uint64_t i = 0; i < m; ++i) {
      uint32_t d = degrees[s + i];
      if (d > R) return fail(SDB_ERR_INVALID, "edge list longer than degreeBound");
      for (uint32_t j = 0; j < d; ++j) {
        uint64_t e = edges[off + j];
        if (e == 0 || e >= (uint64_t(1) << 31) - 1) return fail(SDB_ERR_INVALID, "edge target out of range");
        // a dangling edge (target never stored, or deleted) would send the search kernel to a row
        // that does not exist; the reference fails with "failed to get node for neighbours"
        // (search.go:77-80). Points are hydrated before edges (sdb_index_set_vectors / set_codes).
        if (e >= ix->rows || !ix->h_exists[e])
          return fail(SDB_ERR_NOTFOUND, "edge of node " + std::to_string(ids[s + i]) + " points at a node that does not exist: " + std::to_string(e));
        rows[size_t(i) * R + j] = uint32_t(e);
      }
      off += d;
      degs[i] = d;
    }
    if ((rc = ix->d_ids64.ensure((size_t(m) * R + m + 1) / 2 + 1))) return rc;
    uint32_t* d_rows = reinterpret_cast<uint32_t*>(ix->d_ids64.p);
    uint32_t* d_degs = d_rows + size_t(m) * R;
    SDB_CUDA(cudaMemcpyAsync(d_rows, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice, ix->stream));
    SDB_CUDA(cudaMemcpyAsync(d_degs, degs.data(), degs.size() * 4, cudaMemcpyHostToDevice, ix->stream));
    scatter_edges_kernel<<<uint32_t(m), 64, 0, ix->stream>>>(ix->d_adj, ix->d_deg, R, ix->d_tmp32.p, d_rows, d_degs, uint32_t(m));
    ix->launches++;
    SDB_CUDA(cudaGetLastError());
    SDB_CUDA(cudaStreamSynchronize(ix->stream));
  }
  return SDB_OK;
}

int sdb_index_get_edges(sdb_index* ix, uint64_t n, const uint64_t* ids, uint32_t* degrees_out, uint64_t* edges_out) {
  if (!ix || (n && (!ids || !degrees_out || !edges_out))) return fail(SDB_ERR_INVALID, "null argument");
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  const uint32_t R = ix->p.degree_bound;
  const uint64_t chunk = 1 << 20;
  std::vector<uint32_t> h32, rows, degs;
  for (uint64_t s = 0; s < n; s += chunk) {
    uint64_t m = std::min(chunk, n - s);
    int rc = stage_ids(ix, m, ids + s, false, false, h32);
    if (rc) return rc;
    for (uint64_t i = 0; i < m; ++i)
      if (h32[i] >= ix->rows) return fail(SDB_ERR_NOTFOUND, "node id does not exist: " + std::to_string(ids[s + i]));
    if ((rc = ix->d_ids64.ensure((size_t(m) * R + m + 1) / 2 + 1))) return rc;
    uint32_t* d_rows = reinterpret_cast<uint32_t*>(ix->d_ids64.p);
    uint32_t* d_degs = d_rows + size_t(m) * R;
    gather_edges_kernel<<<uint32_t(m), 64, 0, ix->stream>>>(ix->d_adj, ix->d_deg, R, ix->d_tmp32.p, d_rows, d_degs, uint32_t(m));
    ix->launches++;
    SDB_CUDA(cudaGetLastError());
    rows.resize(size_t(m) * R);
    degs.resize(m);
    SDB_CUDA(cudaMemcpyAsync(rows.data(), d_rows, rows.size() * 4, cudaMemcpyDeviceToHost, ix->stream));
    SDB_CUDA(cudaMemcpyAsync(degs.data(), d_degs, degs.size() * 4, cudaMemcpyDeviceToHost, ix->stream));
    SDB_CUDA(cudaStreamSynchronize(ix->stream));
    for (uint64_t i = 0; i < m; ++i) {
      degrees_out[s + i] = degs[i];
      for (uint32_t j = 0; j < R; ++j)
        edges_out[(s + i) * R + j] = j < degs[i] ? uint64_t(rows[size_t(i) * R + j]) : 0;
    }
  }
  return SDB_OK;
}

int sdb_index_delete(sdb_index* ix, uint64_t n, const uint64_t* ids) {
  if (!ix || (n && !ids)) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  for (uint64_t i = 0; i < n; ++i) {
    if (ids[i] == START_ID) return fail(SDB_ERR_RESERVED_ID, "cannot modify point with start id: 1");
    if (ids[i] == 0 || ids[i] >= ix->rows || !ix->h_exists[ids[i]]) continue;
    uint32_t id = uint32_t(ids[i]);
    ix->h_exists[id] = 0;
    ix->count--;
    ix->vec_epoch++;
    SDB_CUDA(cudaMemsetAsync(ix->d_exists + id, 0, 1, ix->stream));
    SDB_CUDA(cudaMemsetAsync(ix->d_adj + size_t(id) * ix->p.degree_bound, 0xFF, ix->p.degree_bound * 4, ix->stream));
    SDB_CUDA(cudaMemsetAsync(ix->d_deg + id, 0, 4, ix->stream));
  }
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  return SDB_OK;
}

// ---- search -------------------------------------------------------------------------

}  // extern "C"

namespace sdb {

int check_search_args(sdb_index* ix, uint32_t k, uint32_t L) {
  if (k < 1 || k > 75) return fail(SDB_ERR_INVALID, "invalid limit for vector query, expected 1-75");  // models/search.go:291
  if (L > 75 || L < 1 || (!ix->p.relaxed && L < 25)) return fail(SDB_ERR_INVALID, "invalid searchSize for vector query, expected 25-75");
  if (L < k) return fail(SDB_ERR_SEARCHSIZE, "searchSize (" + std::to_string(L) + ") must be greater than k (" + std::to_string(k) + ")");
  if (ix->rows <= START_ID || !ix->h_exists[START_ID]) return fail(SDB_ERR_STATE, "failed to get start point");  // search.go:57-60
  return SDB_OK;
}

int check_requests(sdb_index* ix, uint32_t B, const sdb_request* req, uint32_t n_filters, uint32_t k_stride, bool flat) {
  if (!req) return fail(SDB_ERR_INVALID, "null argument");
  for (uint32_t b = 0; b < B; ++b) {
    const sdb_request& r = req[b];
    if (r.limit < 1 || r.limit > 75) return fail(SDB_ERR_INVALID, "invalid limit for vector query, expected 1-75");  // models/search.go:291
    if (!flat) {
      const uint32_t L = r.search_size;
      if (L > 75 || L < 1 || (!ix->p.relaxed && L < 25)) return fail(SDB_ERR_INVALID, "invalid searchSize for vector query, expected 25-75");
      if (L < r.limit)
        return fail(SDB_ERR_SEARCHSIZE, "searchSize (" + std::to_string(L) + ") must be greater than k (" + std::to_string(r.limit) + ")");
    }
    if (r.limit > k_stride || k_stride > 75) return fail(SDB_ERR_INVALID, "requests: k_stride must be 1..75 and at least every limit");
    if (r.filter < -1 || (r.filter >= 0 && uint32_t(r.filter) >= n_filters))
      return fail(SDB_ERR_INVALID, "requests: filter must be -1 or a filter index");
  }
  if (!flat && (ix->rows <= START_ID || !ix->h_exists[START_ID])) return fail(SDB_ERR_STATE, "failed to get start point");
  return SDB_OK;
}

static int ensure_out_scratch(sdb_index* ix, uint32_t B, uint32_t k) {
  int rc;
  if ((rc = ix->d_oid.ensure(size_t(B) * k))) return rc;
  if ((rc = ix->d_od.ensure(size_t(B) * k))) return rc;
  if ((rc = ix->d_oc.ensure(B))) return rc;
  return SDB_OK;
}

// Staging of a batch's filters (search.go:33-51,93-95; one roaring bitmap per request,
// shard/index/search.go:59-85) into the device form of SearchFilters: concatenated ascending u32
// id lists + offsets, the per-query filter index, the batch positions of the filtered and of the
// unfiltered requests, and — for a single shared filter — a dense bitmask over rows, built on the
// device. filter f = filter_ids[filter_offsets[f] .. filter_offsets[f+1]); query_filter[b] < 0 =
// request b is not filtered (nullptr: every request uses filter 0). An EMPTY list is still a
// filter: the reference then seeds nothing and returns no result (search.go:33-51 with an empty
// bitmap). Flat search drops ids below 2 (the scan's first id) like ids beyond the store.
// Everything goes into one page-locked slot (and, for the gather route's work items, its item
// buffer), moved to the device by one copy each (commit_filters), so a filtered call enqueues its
// staging without a host synchronisation. A request batch (req) also stages every request's
// parameters, and takes a slot even when nobody is filtered.
int stage_filters(sdb_index* ix, uint32_t B, uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                  const int32_t* query_filter, uint32_t L, bool flat, FilterStage* out, const sdb_request* req) {
  if ((!req && n_filters == 0) || (n_filters && !filter_offsets))
    return fail(SDB_ERR_INVALID, "filters: need at least one filter and its offsets");
  for (uint32_t f = 0; f < n_filters; ++f)
    if (filter_offsets[f + 1] < filter_offsets[f]) return fail(SDB_ERR_INVALID, "filters: offsets must ascend");
  const uint64_t n_raw = n_filters ? filter_offsets[n_filters] - filter_offsets[0] : 0;
  // request batch: per-request filter index, and per filter the seeds its requests read (the largest
  // search_size among them; the batch's largest for a filter no request uses)
  std::vector<int32_t> req_qf;
  std::vector<uint32_t> seed_L;
  if (req) {
    req_qf.resize(B);
    seed_L.assign(n_filters, 0);
    uint32_t L_max = 0;
    for (uint32_t b = 0; b < B; ++b) {
      req_qf[b] = req[b].filter < 0 ? -1 : req[b].filter;
      L_max = std::max(L_max, req[b].search_size);
      if (req[b].filter >= 0) seed_L[req[b].filter] = std::max(seed_L[req[b].filter], req[b].search_size);
    }
    for (uint32_t& x : seed_L) x = flat ? 0 : (x ? x : L_max);
    query_filter = req_qf.data();
  }
  if (n_raw >= (uint64_t(1) << 32)) return fail(SDB_ERR_INVALID, "filters: too many ids in one batch");
  // slot layout: ids | offsets | query filter | qmap | flat: request rows and gather requests (all
  // bounded by the id count and B; the gather work items are sized by flat_plan once routed)
  FilterStage& fs = *out;
  fs.ids_at = 0;
  fs.off_at = align16(size_t(n_raw) * 4 + 4);
  fs.qf_at = fs.off_at + align16((size_t(n_filters) + 1) * 4);
  fs.qmap_at = fs.qf_at + (query_filter ? align16(size_t(B) * 4) : 0);
  fs.req_at = fs.qmap_at + (query_filter ? align16(size_t(B) * 4 + 4) : 0);
  const size_t flat_at = fs.req_at + (req ? align16(size_t(B) * sizeof(uint4)) : 0);
  const size_t bytes = flat_at + (flat && n_filters ? flat_plan_bytes(B) : 0);
  // the slot is refilled once the copy out of it two filtered calls ago has run
  const uint32_t s = ix->fstage_next;
  SDB_CUDA(cudaEventSynchronize(ix->fstage_ev[s]));
  int rc;
  if ((rc = ix->h_stage[s].ensure(bytes))) return rc;
  uint8_t* h = ix->h_stage[s].p;
  uint32_t* ids = reinterpret_cast<uint32_t*>(h + fs.ids_at);
  uint32_t* off = reinterpret_cast<uint32_t*>(h + fs.off_at);
  const uint64_t min_id = flat ? 2 : 0;
  uint32_t n = 0;
  for (uint32_t f = 0; f < n_filters; ++f) {
    const uint64_t b0 = filter_offsets[f], b1 = filter_offsets[f + 1];
    if (b1 > b0 && !filter_ids) return fail(SDB_ERR_INVALID, "filters: offsets must ascend");
    off[f] = n;
    const uint64_t seeds = req ? seed_L[f] : L;
    uint64_t prev = 0;
    for (uint64_t i = b0; i < b1; ++i) {
      const uint64_t id = filter_ids[i];
      if (i > b0 && id <= prev) return fail(SDB_ERR_INVALID, "filter ids must be strictly ascending");
      prev = id;
      if (i - b0 < seeds && (id == 0 || id >= ix->rows || !ix->h_exists[id]))
        return fail(SDB_ERR_NOTFOUND, "failed to get filter points");  // GetMany of the seeds, search.go:45-48
      if (id < ix->rows && id >= min_id) ids[n++] = uint32_t(id);  // ids beyond the store can never be expanded
    }
  }
  off[n_filters] = n;
  fs.n_ids = n;
  fs.h_off = off;
  // one filter shared by every request: the dense bitmap (a request batch: every request uses filter 0)
  const bool all_first = req && std::all_of(req, req + B, [](const sdb_request& r) { return r.filter == 0; });
  fs.shared_bits = !flat && n_filters == 1 && (!query_filter || all_first);
  fs.per_request = query_filter != nullptr;
  fs.has_req = req != nullptr;
  fs.is_flat = flat;
  fs.sf = SearchFilters{};
  fs.sf.n_filtered = B;
  if (query_filter) {
    uint32_t n_filtered = 0;
    for (uint32_t b = 0; b < B; ++b) {
      if (query_filter[b] >= int32_t(n_filters)) return fail(SDB_ERR_INVALID, "filters: query_filter index out of range");
      n_filtered += query_filter[b] >= 0;
    }
    int32_t* qf = reinterpret_cast<int32_t*>(h + fs.qf_at);
    uint32_t* qmap = reinterpret_cast<uint32_t*>(h + fs.qmap_at);  // filtered positions, then unfiltered ones
    uint32_t nf = 0, np = n_filtered;
    for (uint32_t b = 0; b < B; ++b) {
      qf[b] = query_filter[b] < 0 ? 0 : query_filter[b];
      qmap[query_filter[b] < 0 ? np++ : nf++] = b;
    }
    fs.sf.n_filtered = n_filtered;
    fs.sf.n_plain = B - n_filtered;
  }
  if (req) {
    uint4* rq = reinterpret_cast<uint4*>(h + fs.req_at);
    for (uint32_t b = 0; b < B; ++b) {
      const sdb_request& r = req[b];
      const uint32_t plim = r.shard_limit == 0 || r.shard_limit > r.limit ? r.limit : r.shard_limit;
      rq[b] = make_uint4(r.search_size, r.limit, plim, 0);
    }
  }
  fs.flat = FlatFilterPlan{};
  if (flat && n_filters) {
    const uint32_t npts = std::max<uint32_t>(2, ix->max_node_id + 1) - 2;
    if ((rc = flat_plan(ix, s, B, n_filters, off, query_filter, npts, h, flat_at, &fs.flat))) return rc;
    fs.bytes = fs.flat.items_at;
  } else {
    fs.bytes = flat_at;
  }
  fs.slot = s;
  return SDB_OK;
}

int commit_filters(sdb_index* ix, FilterStage* fs, cudaStream_t stream) {
  int rc;
  // before the copy occupies the stream: the beam search's visited-table step-up reads an idle stream
  if (!fs->is_flat && (rc = retry_check(ix))) return rc;
  const size_t item_bytes = fs->is_flat ? size_t(fs->flat.n_items) * sizeof(uint4) : 0;
  if ((rc = ix->d_fstage.ensure(fs->bytes + item_bytes))) return rc;
  if (fs->shared_bits && (rc = ix->d_filter_bits.ensure((size_t(ix->rows) + 31) / 32 + 1))) return rc;
  // the previous filtered call, on whichever stream, has read its lists, bitmap and scratch
  SDB_CUDA(cudaStreamWaitEvent(stream, ix->filter_done_ev, 0));
  SDB_CUDA(cudaMemcpyAsync(ix->d_fstage.p, ix->h_stage[fs->slot].p, fs->bytes, cudaMemcpyHostToDevice, stream));
  if (item_bytes)
    SDB_CUDA(cudaMemcpyAsync(ix->d_fstage.p + fs->flat.items_at, ix->h_stage_items[fs->slot].p, item_bytes, cudaMemcpyHostToDevice,
                             stream));
  SDB_CUDA(cudaEventRecord(ix->fstage_ev[fs->slot], stream));
  ix->fstage_next = fs->slot ^ 1;
  uint8_t* d = ix->d_fstage.p;
  SearchFilters& sf = fs->sf;
  sf.ids = reinterpret_cast<const uint32_t*>(d + fs->ids_at);
  sf.off = reinterpret_cast<const uint32_t*>(d + fs->off_at);
  if (fs->per_request) {
    sf.query_filter = reinterpret_cast<const int32_t*>(d + fs->qf_at);
    sf.qmap_filtered = reinterpret_cast<const uint32_t*>(d + fs->qmap_at);
    sf.qmap_plain = sf.qmap_filtered + sf.n_filtered;
  }
  if (fs->has_req) sf.req = reinterpret_cast<const uint4*>(d + fs->req_at);
  if (fs->shared_bits) {
    if ((rc = launch_filter_bits(ix, sf.ids, fs->n_ids, ix->d_filter_bits.p, stream))) return rc;
    sf.bits = ix->d_filter_bits.p;
  }
  return SDB_OK;
}

void filters_done(sdb_index* ix, cudaStream_t stream) { cudaEventRecord(ix->filter_done_ev, stream); }

}  // namespace sdb

extern "C" {

static int search_batch_locked(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, uint32_t search_size,
                               const SearchFilters* filters, uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  int rc;
  // Page-locked caller buffers (cudaHostAlloc / cudaHostRegister: what a cgo wrapper keeps for its
  // request batches) are mapped into the device address space: the kernel then reads each query
  // once straight from host memory (512 B per query, when a warp picks the query up) and stores
  // the top-k straight back, so the copies disappear from the critical path instead of preceding
  // and following the kernel. Pageable buffers go through the staging copies.
  auto mapped = [&](const void* p) -> void* {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
  };
  const float* q_dev = static_cast<const float*>(mapped(queries));
  uint64_t* oid_dev = static_cast<uint64_t*>(mapped(out_ids));
  float* od_dev = static_cast<float*>(mapped(out_dists));
  uint32_t* oc_dev = static_cast<uint32_t*>(mapped(out_counts));
  if (!q_dev) {
    if ((rc = ix->d_q.ensure(size_t(B) * ix->p.dim))) return rc;
    SDB_CUDA(cudaMemcpyAsync(ix->d_q.p, queries, size_t(B) * ix->p.dim * sizeof(float), cudaMemcpyHostToDevice, ix->stream));
    q_dev = ix->d_q.p;
  }
  if ((rc = ensure_out_scratch(ix, B, k))) return rc;
  rc = launch_search(ix, B, q_dev, k, search_size, oid_dev ? oid_dev : ix->d_oid.p, od_dev ? od_dev : ix->d_od.p,
                     oc_dev ? oc_dev : ix->d_oc.p, nullptr, nullptr, nullptr, 0, filters, ix->stream);
  if (filters) filters_done(ix, ix->stream);
  if (rc) return rc;
  if (!oid_dev) SDB_CUDA(cudaMemcpyAsync(out_ids, ix->d_oid.p, size_t(B) * k * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->stream));
  if (!od_dev) SDB_CUDA(cudaMemcpyAsync(out_dists, ix->d_od.p, size_t(B) * k * sizeof(float), cudaMemcpyDeviceToHost, ix->stream));
  if (!oc_dev) SDB_CUDA(cudaMemcpyAsync(out_counts, ix->d_oc.p, size_t(B) * sizeof(uint32_t), cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  return SDB_OK;
}

int sdb_search_batch(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, uint32_t search_size,
                     const uint64_t* filter_ids, uint64_t n_filter, uint64_t* out_ids, float* out_dists,
                     uint32_t* out_counts) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!queries || !out_ids || !out_dists || !out_counts) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  int rc = check_search_args(ix, k, search_size);
  if (rc) return rc;
  // filter_ids != NULL = filtered, even with n_filter == 0 (an empty bitmap filters everything out);
  // callers whose empty container has a NULL data pointer use sdb_search_batch_filters
  FilterStage fs;
  const bool filtered = filter_ids != nullptr;
  if (filtered) {
    const uint64_t offs[2] = {0, n_filter};
    if ((rc = stage_filters(ix, B, 1, filter_ids, offs, nullptr, search_size, false, &fs)) ||
        (rc = commit_filters(ix, &fs, ix->stream)))
      return rc;
  }
  return search_batch_locked(ix, B, queries, k, search_size, filtered ? &fs.sf : nullptr, out_ids, out_dists, out_counts);
}

int sdb_search_batch_filters(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, uint32_t search_size,
                             uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                             const int32_t* query_filter, uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!queries || !out_ids || !out_dists || !out_counts) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  int rc = check_search_args(ix, k, search_size);
  if (rc) return rc;
  if (n_filters == 0) return search_batch_locked(ix, B, queries, k, search_size, nullptr, out_ids, out_dists, out_counts);
  FilterStage fs;
  if ((rc = stage_filters(ix, B, n_filters, filter_ids, filter_offsets, query_filter, search_size, false, &fs)) ||
      (rc = commit_filters(ix, &fs, ix->stream)))
    return rc;
  return search_batch_locked(ix, B, queries, k, search_size, &fs.sf, out_ids, out_dists, out_counts);
}

int sdb_search_batch_requests(sdb_index* ix, uint32_t B, const float* queries, const sdb_request* req, uint32_t n_filters,
                              const uint64_t* filter_ids, const uint64_t* filter_offsets, uint32_t k_stride,
                              uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!queries || !out_ids || !out_dists || !out_counts) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  int rc = check_requests(ix, B, req, n_filters, k_stride, false);
  if (rc) return rc;
  FilterStage fs;
  if ((rc = stage_filters(ix, B, n_filters, filter_ids, filter_offsets, nullptr, 0, false, &fs, req)) ||
      (rc = commit_filters(ix, &fs, ix->stream)))
    return rc;
  return search_batch_locked(ix, B, queries, k_stride, 75, &fs.sf, out_ids, out_dists, out_counts);
}

int sdb_search_batch_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint32_t search_size,
                            uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, void* stream) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!d_queries || !d_out_ids || !d_out_dists || !d_out_counts) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  int rc = check_search_args(ix, k, search_size);
  if (rc) return rc;
  return launch_search(ix, B, d_queries, k, search_size, d_out_ids, d_out_dists, d_out_counts, nullptr, nullptr, nullptr, 0,
                       nullptr, static_cast<cudaStream_t>(stream));
}

int sdb_last_search_stats(sdb_index* ix, uint32_t B, uint32_t* hops_out, uint32_t* ndist_out) {
  if (!ix || !hops_out || !ndist_out) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (B > ix->last_B) return fail(SDB_ERR_STATE, "no search of that size has run on this handle");
  SDB_CUDA(cudaDeviceSynchronize());
  SDB_CUDA(cudaMemcpy(hops_out, ix->d_hops.p, size_t(B) * 4, cudaMemcpyDeviceToHost));
  SDB_CUDA(cudaMemcpy(ndist_out, ix->d_ndist.p, size_t(B) * 4, cudaMemcpyDeviceToHost));
  return SDB_OK;
}

int sdb_search_profile(sdb_index* ix, int32_t enable) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (enable && ix->prof_ev.empty()) {
    ix->prof_ev.resize(2 * sdb_index::PROF_RING, nullptr);
    for (auto& e : ix->prof_ev) SDB_CUDA(cudaEventCreate(&e));
  }
  ix->prof_on = enable != 0;
  ix->prof_n = 0;
  return SDB_OK;
}

int sdb_search_profile_read(sdb_index* ix, uint32_t cap, float* ms_out, uint32_t* n_out) {
  if (!ix || !n_out || (cap && !ms_out)) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  *n_out = ix->prof_n;
  for (uint32_t i = 0; i < ix->prof_n && i < cap; ++i) {
    SDB_CUDA(cudaEventSynchronize(ix->prof_ev[2 * i + 1]));
    SDB_CUDA(cudaEventElapsedTime(ms_out + i, ix->prof_ev[2 * i], ix->prof_ev[2 * i + 1]));
  }
  return SDB_OK;
}

int sdb_search_visited(sdb_index* ix, uint32_t B, const float* queries, uint32_t search_size, uint32_t vis_cap,
                       uint64_t* out_vis_ids, float* out_vis_dists, uint32_t* out_vis_len) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!queries || !out_vis_ids || !out_vis_dists || !out_vis_len || vis_cap == 0) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  int rc = check_search_args(ix, 1, search_size);
  if (rc) return rc;
  if ((rc = ix->d_q.ensure(size_t(B) * ix->p.dim))) return rc;
  if ((rc = ensure_out_scratch(ix, B, 1))) return rc;
  if ((rc = ix->d_vis_ids.ensure(size_t(B) * vis_cap))) return rc;
  if ((rc = ix->d_vis_d.ensure(size_t(B) * vis_cap))) return rc;
  if ((rc = ix->d_vis_len.ensure(B))) return rc;
  SDB_CUDA(cudaMemcpyAsync(ix->d_q.p, queries, size_t(B) * ix->p.dim * sizeof(float), cudaMemcpyHostToDevice, ix->stream));
  rc = launch_search(ix, B, ix->d_q.p, 1, search_size, ix->d_oid.p, ix->d_od.p, ix->d_oc.p, ix->d_vis_ids.p, ix->d_vis_d.p,
                     ix->d_vis_len.p, vis_cap, nullptr, ix->stream);
  if (rc) return rc;
  std::vector<uint32_t> ids(size_t(B) * vis_cap);
  std::vector<float> d(size_t(B) * vis_cap);
  SDB_CUDA(cudaMemcpyAsync(ids.data(), ix->d_vis_ids.p, ids.size() * 4, cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaMemcpyAsync(d.data(), ix->d_vis_d.p, d.size() * 4, cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaMemcpyAsync(out_vis_len, ix->d_vis_len.p, size_t(B) * 4, cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  // visitedSet.Sort() (search.go:100; distset.go:223-238 with sortedUntil == 0): stable
  // insertion sort by distance of the expansion-ordered list.
  for (uint32_t b = 0; b < B; ++b) {
    uint32_t n = std::min(out_vis_len[b], vis_cap);
    uint32_t* bi = &ids[size_t(b) * vis_cap];
    float* bd = &d[size_t(b) * vis_cap];
    for (uint32_t i = 0; i < n; ++i)
      for (uint32_t j = i; j > 0 && bd[j] < bd[j - 1]; --j) {
        std::swap(bd[j], bd[j - 1]);
        std::swap(bi[j], bi[j - 1]);
      }
    for (uint32_t i = 0; i < vis_cap; ++i) {
      out_vis_ids[size_t(b) * vis_cap + i] = i < n ? bi[i] : 0;
      out_vis_dists[size_t(b) * vis_cap + i] = i < n ? bd[i] : std::numeric_limits<float>::infinity();
    }
  }
  return SDB_OK;
}

// Flat search of a batch (sdb_flat_search_batch, sdb_flat_search_batch_filters): n_filters == 0 =
// nobody is filtered, otherwise the filters of sdb_search_batch_filters, routed by launch_flat_filtered.
static int flat_batch_locked(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, uint32_t n_filters,
                             const uint64_t* filter_ids, const uint64_t* filter_offsets, const int32_t* query_filter,
                             uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  int rc;
  FilterStage fs;
  // flat search has no GetMany of seeds (L = 0): ids that are not stored are simply never matched
  if (n_filters && (rc = stage_filters(ix, B, n_filters, filter_ids, filter_offsets, query_filter, 0, true, &fs))) return rc;
  if ((rc = ix->d_q.ensure(size_t(B) * ix->p.dim))) return rc;
  if ((rc = ensure_out_scratch(ix, B, k))) return rc;
  SDB_CUDA(cudaMemcpyAsync(ix->d_q.p, queries, size_t(B) * ix->p.dim * sizeof(float), cudaMemcpyHostToDevice, ix->stream));
  if (n_filters) {
    if ((rc = commit_filters(ix, &fs, ix->stream))) return rc;
    rc = launch_flat_filtered(ix, B, ix->d_q.p, k, fs, ix->d_oid.p, ix->d_od.p, ix->d_oc.p, ix->stream);
    filters_done(ix, ix->stream);
    if (rc) return rc;
  } else {
    rc = flat_device_locked(ix, B, ix->d_q.p, k, ix->d_oid.p, ix->d_od.p, ix->d_oc.p, ix->stream);
    if (rc) return rc;
  }
  // the result copies go in front of the call's one synchronisation
  SDB_CUDA(cudaMemcpyAsync(out_ids, ix->d_oid.p, size_t(B) * k * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaMemcpyAsync(out_dists, ix->d_od.p, size_t(B) * k * sizeof(float), cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaMemcpyAsync(out_counts, ix->d_oc.p, size_t(B) * sizeof(uint32_t), cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  return flat_stats_settle(ix);
}

int sdb_flat_search_batch(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, const uint64_t* filter_ids,
                          uint64_t n_filter, uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!queries || !out_ids || !out_dists || !out_counts) return fail(SDB_ERR_INVALID, "null argument");
  if (k < 1 || k > 75) return fail(SDB_ERR_INVALID, "invalid limit for vector query, expected 1-75");  // models/search.go:329
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (!filter_ids) return flat_batch_locked(ix, B, queries, k, 0, nullptr, nullptr, nullptr, out_ids, out_dists, out_counts);
  // this entry takes the ids in any order, duplicates included: the one-filter case of the per-request form
  std::vector<uint64_t> ids(filter_ids, filter_ids + n_filter);
  std::sort(ids.begin(), ids.end());
  ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
  const uint64_t offs[2] = {0, ids.size()};
  return flat_batch_locked(ix, B, queries, k, 1, ids.data(), offs, nullptr, out_ids, out_dists, out_counts);
}

int sdb_flat_search_batch_filters(sdb_index* ix, uint32_t B, const float* queries, uint32_t k, uint32_t n_filters,
                                  const uint64_t* filter_ids, const uint64_t* filter_offsets, const int32_t* query_filter,
                                  uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!queries || !out_ids || !out_dists || !out_counts) return fail(SDB_ERR_INVALID, "null argument");
  if (k < 1 || k > 75) return fail(SDB_ERR_INVALID, "invalid limit for vector query, expected 1-75");  // models/search.go:329
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  return flat_batch_locked(ix, B, queries, k, n_filters, filter_ids, filter_offsets, query_filter, out_ids, out_dists,
                           out_counts);
}

int sdb_flat_search_batch_requests(sdb_index* ix, uint32_t B, const float* queries, const sdb_request* req,
                                   uint32_t n_filters, const uint64_t* filter_ids, const uint64_t* filter_offsets,
                                   uint32_t k_stride, uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!queries || !out_ids || !out_dists || !out_counts) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  int rc = check_requests(ix, B, req, n_filters, k_stride, true);
  if (rc) return rc;
  FilterStage fs;
  if ((rc = stage_filters(ix, B, n_filters, filter_ids, filter_offsets, nullptr, 0, true, &fs, req))) return rc;
  if ((rc = ix->d_q.ensure(size_t(B) * ix->p.dim))) return rc;
  if ((rc = ensure_out_scratch(ix, B, k_stride))) return rc;
  SDB_CUDA(cudaMemcpyAsync(ix->d_q.p, queries, size_t(B) * ix->p.dim * sizeof(float), cudaMemcpyHostToDevice, ix->stream));
  if ((rc = commit_filters(ix, &fs, ix->stream))) return rc;
  if ((rc = flat_requests_locked(ix, B, ix->d_q.p, n_filters, fs, k_stride, ix->d_oid.p, ix->d_od.p, ix->d_oc.p, nullptr,
                                 ix->stream)))
    return rc;
  const size_t n = size_t(B) * k_stride;
  SDB_CUDA(cudaMemcpyAsync(out_ids, ix->d_oid.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaMemcpyAsync(out_dists, ix->d_od.p, n * sizeof(float), cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaMemcpyAsync(out_counts, ix->d_oc.p, size_t(B) * sizeof(uint32_t), cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  return flat_stats_settle(ix);
}

int sdb_flat_search_batch_device(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint64_t* d_out_ids,
                                 float* d_out_dists, uint32_t* d_out_counts, void* stream) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (B == 0) return SDB_OK;
  if (!d_queries || !d_out_ids || !d_out_dists || !d_out_counts) return fail(SDB_ERR_INVALID, "null argument");
  if (k < 1 || k > 75) return fail(SDB_ERR_INVALID, "invalid limit for vector query, expected 1-75");  // models/search.go:329
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  return flat_device_locked(ix, B, d_queries, k, d_out_ids, d_out_dists, d_out_counts, static_cast<cudaStream_t>(stream));
}

int sdb_flat_last_filter_stats(sdb_index* ix, uint32_t* gathered_filters, uint32_t* scanned_filters, uint64_t* gathered_pairs) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  std::lock_guard<std::mutex> g(ix->mu);
  if (gathered_filters) *gathered_filters = ix->flat_last_gathered;
  if (scanned_filters) *scanned_filters = ix->flat_last_scanned;
  if (gathered_pairs) *gathered_pairs = ix->flat_last_pairs;
  return SDB_OK;
}

int sdb_filter_staging_bytes(sdb_index* ix, uint64_t* pinned_bytes, uint64_t* device_bytes) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  std::lock_guard<std::mutex> g(ix->mu);
  uint64_t pinned = 0;
  for (int s = 0; s < 2; ++s) pinned += ix->h_stage[s].n + ix->h_stage_items[s].n * sizeof(uint4);
  if (pinned_bytes) *pinned_bytes = pinned;
  if (device_bytes) *device_bytes = ix->d_fstage.n;
  return SDB_OK;
}

int sdb_insert_batch(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (n == 0) return SDB_OK;
  if (!ids || !vectors) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  return insert_batch_locked(ix, n, ids, vectors);
}

int sdb_insert_batch_device(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* d_vectors) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (n == 0) return SDB_OK;
  if (!ids || !d_vectors) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, d_vectors) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != ix->device) {
    cudaGetLastError();
    return fail(SDB_ERR_INVALID, "sdb_insert_batch_device: vectors must be device memory of the index's GPU");
  }
  SDB_CUDA(cudaDeviceSynchronize());  // the caller's producer stream is unknown: order after everything
  return insert_batch_locked(ix, n, ids, d_vectors, false, true);
}

uint64_t sdb_insert_truncated(const sdb_index* ix) { return ix ? ix->insert_truncated : 0; }

int sdb_insert_stats(sdb_index* ix, uint64_t* out8, int32_t reset) {
  if (!ix || !out8) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  for (int i = 0; i < 8; ++i) out8[i] = 0;
  if (!ix->d_ins_stats) return SDB_OK;
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  SDB_CUDA(cudaMemcpy(out8, ix->d_ins_stats, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  if (reset) SDB_CUDA(cudaMemset(ix->d_ins_stats, 0, 8 * sizeof(uint64_t)));
  return SDB_OK;
}

int sdb_insert_update_delete(sdb_index* ix, uint64_t n, const uint64_t* ids, const float* vectors,
                             const uint8_t* has_vector) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  if (n == 0) return SDB_OK;
  if (!ids || !vectors) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  return insert_update_delete_locked(ix, n, ids, vectors, has_vector);
}

int sdb_edge_scan(sdb_index* ix, uint64_t n_delete, const uint64_t* delete_ids, uint64_t* to_prune, uint64_t* n_prune,
                  uint64_t* to_save, uint64_t* n_save) {
  if (!ix || (n_delete && !delete_ids) || !to_prune || !n_prune || !to_save || !n_save)
    return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  return edge_scan_locked(ix, n_delete, delete_ids, to_prune, n_prune, to_save, n_save);
}

int sdb_index_get_start_overflow(sdb_index* ix, uint64_t cap, uint64_t* out, uint64_t* n) {
  if (!ix || !n || (cap && !out)) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  *n = ix->h_start_extra.size();
  for (uint64_t i = 0; i < *n && i < cap; ++i) out[i] = ix->h_start_extra[i];
  return SDB_OK;
}

int sdb_index_set_start_overflow(sdb_index* ix, uint64_t n, const uint64_t* ids) {
  if (!ix || (n && !ids)) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  for (uint64_t i = 0; i < n; ++i)
    if (ids[i] >= ix->rows || !ix->h_exists[ids[i]]) return fail(SDB_ERR_NOTFOUND, "node id does not exist: " + std::to_string(ids[i]));
  ix->h_start_extra.assign(ids, ids + n);
  return upload_start_extra(ix);
}

int sdb_insert_config(sdb_index* ix, uint32_t min_batch, uint32_t max_batch, uint32_t growth_div) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  std::lock_guard<std::mutex> g(ix->mu);
  if (min_batch) ix->ins_min_batch = min_batch;
  if (max_batch) ix->ins_max_batch = max_batch;
  if (growth_div) ix->ins_growth_div = growth_div;
  if (ix->ins_max_batch && ix->ins_max_batch < ix->ins_min_batch) ix->ins_max_batch = ix->ins_min_batch;
  return SDB_OK;
}

int sdb_index_fit(sdb_index* ix, uint64_t pq_first_row, int32_t* fitted) {
  if (!ix) return fail(SDB_ERR_INVALID, "null index");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  int32_t f = 0;
  int rc = fit_locked(ix, pq_first_row, &f);
  if (fitted) *fitted = f;
  return rc;
}

int sdb_index_get_pq(sdb_index* ix, float* flat_centroids, float* centroid_dists) {
  if (!ix || !flat_centroids || !centroid_dists) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (!ix->pq_fitted) return fail(SDB_ERR_STATE, "product quantizer is not fitted");
  SDB_CUDA(cudaMemcpy(flat_centroids, ix->d_pq_centroids, size_t(ix->pqM) * ix->pqK * ix->pqSub * 4, cudaMemcpyDeviceToHost));
  SDB_CUDA(cudaMemcpy(centroid_dists, ix->d_pq_cdist, size_t(ix->pqM) * ix->pqK * ix->pqK * 4, cudaMemcpyDeviceToHost));
  return SDB_OK;
}

int sdb_index_set_pq(sdb_index* ix, const float* flat_centroids, const float* centroid_dists) {
  if (!ix || !flat_centroids || !centroid_dists) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (ix->p.quantizer != SDB_QUANT_PRODUCT) return fail(SDB_ERR_STATE, "index has no product quantizer");
  size_t nc = size_t(ix->pqM) * ix->pqK * ix->pqSub, nd = size_t(ix->pqM) * ix->pqK * ix->pqK;
  if (!ix->d_pq_centroids) SDB_CUDA(cudaMalloc(reinterpret_cast<void**>(&ix->d_pq_centroids), nc * 4));
  if (!ix->d_pq_cdist) SDB_CUDA(cudaMalloc(reinterpret_cast<void**>(&ix->d_pq_cdist), nd * 4));
  SDB_CUDA(cudaMemcpy(ix->d_pq_centroids, flat_centroids, nc * 4, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(ix->d_pq_cdist, centroid_dists, nd * 4, cudaMemcpyHostToDevice));
  ix->pq_fitted = true;
  // re-encode every stored point with the index metric (productQuantizer.encode)
  std::vector<uint32_t> ids;
  for (uint32_t id = 0; id < ix->rows; ++id)
    if (ix->h_exists[id]) ids.push_back(id);
  if (!ids.empty()) {
    int rc = ix->d_tmp32.ensure(ids.size());
    if (rc) return rc;
    SDB_CUDA(cudaMemcpy(ix->d_tmp32.p, ids.data(), ids.size() * 4, cudaMemcpyHostToDevice));
    if ((rc = launch_encode_rows(ix, uint32_t(ids.size()), ix->d_tmp32.p, ix->stream))) return rc;
    SDB_CUDA(cudaStreamSynchronize(ix->stream));
  }
  return SDB_OK;
}

int sdb_index_get_bq_threshold(sdb_index* ix, float* threshold) {
  if (!ix || !threshold) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (ix->p.quantizer != SDB_QUANT_BINARY || !ix->bq_fitted) return fail(SDB_ERR_STATE, "binary quantizer threshold is not set");
  SDB_CUDA(cudaMemcpy(threshold, ix->d_bq_thr, ix->p.dim * 4, cudaMemcpyDeviceToHost));
  return SDB_OK;
}

int sdb_index_set_bq_threshold(sdb_index* ix, const float* threshold) {
  if (!ix || !threshold) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (ix->p.quantizer != SDB_QUANT_BINARY) return fail(SDB_ERR_STATE, "index has no binary quantizer");
  SDB_CUDA(cudaMemcpy(ix->d_bq_thr, threshold, ix->p.dim * 4, cudaMemcpyHostToDevice));
  ix->bq_fitted = true;
  std::vector<uint32_t> ids;
  for (uint32_t id = 0; id < ix->rows; ++id)
    if (ix->h_exists[id]) ids.push_back(id);
  if (!ids.empty()) {
    int rc = ix->d_tmp32.ensure(ids.size());
    if (rc) return rc;
    SDB_CUDA(cudaMemcpy(ix->d_tmp32.p, ids.data(), ids.size() * 4, cudaMemcpyHostToDevice));
    if ((rc = launch_encode_rows(ix, uint32_t(ids.size()), ix->d_tmp32.p, ix->stream))) return rc;
    SDB_CUDA(cudaStreamSynchronize(ix->stream));
  }
  return SDB_OK;
}

int sdb_index_get_codes(sdb_index* ix, uint64_t n, const uint64_t* ids, uint8_t* out) {
  if (!ix || (n && (!ids || !out))) return fail(SDB_ERR_INVALID, "null argument");
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (!ix->quant_active()) return fail(SDB_ERR_STATE, "quantizer is not fitted");
  const uint32_t width = ix->p.quantizer == SDB_QUANT_PRODUCT ? ix->pqM : ix->words * 8;
  const uint32_t pitch = ix->p.quantizer == SDB_QUANT_PRODUCT ? ix->codes_pitch : ix->bits_pitch * 8;
  const uint8_t* base = ix->p.quantizer == SDB_QUANT_PRODUCT ? ix->d_codes : reinterpret_cast<const uint8_t*>(ix->d_bits);
  // one gather kernel + one copy per chunk (a 1M-point flush used to issue 1M small copies)
  const uint64_t chunk = std::max<uint64_t>(1, (uint64_t(256) << 20) / width);
  std::vector<uint32_t> h32;
  for (uint64_t s0 = 0; s0 < n; s0 += chunk) {
    const uint64_t m = std::min(chunk, n - s0);
    int rc = stage_ids(ix, m, ids + s0, true, false, h32);
    if (rc) return rc;
    if ((rc = ix->d_tmp8.ensure(size_t(m) * width))) return rc;
    gather_codes_kernel<<<uint32_t((m * width + 255) / 256), 256, 0, ix->stream>>>(base, pitch, width, ix->d_tmp32.p, ix->d_tmp8.p, m);
    ix->launches++;
    SDB_CUDA(cudaGetLastError());
    SDB_CUDA(cudaMemcpyAsync(out + s0 * width, ix->d_tmp8.p, size_t(m) * width, cudaMemcpyDeviceToHost, ix->stream));
    SDB_CUDA(cudaStreamSynchronize(ix->stream));
  }
  return SDB_OK;
}

int sdb_index_set_codes(sdb_index* ix, uint64_t n, const uint64_t* ids, const uint8_t* codes) {
  if (!ix || (n && (!ids || !codes))) return fail(SDB_ERR_INVALID, "null argument");
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (!ix->quant_active()) return fail(SDB_ERR_STATE, "quantizer is not fitted");
  for (uint64_t i = 0; i < n; ++i)
    if (ids[i] == 0) return fail(SDB_ERR_RESERVED_ID, "invalid point id: 0");
  const uint32_t width = ix->p.quantizer == SDB_QUANT_PRODUCT ? ix->pqM : ix->words * 8;
  const uint32_t pitch = ix->p.quantizer == SDB_QUANT_PRODUCT ? ix->codes_pitch : ix->bits_pitch * 8;
  const uint64_t chunk = std::max<uint64_t>(1, (uint64_t(256) << 20) / width);
  std::vector<uint32_t> h32;
  for (uint64_t s0 = 0; s0 < n; s0 += chunk) {
    const uint64_t m = std::min(chunk, n - s0);
    int rc = stage_ids(ix, m, ids + s0, false, true, h32);  // grows the row arrays
    if (rc) return rc;
    uint8_t* base = ix->p.quantizer == SDB_QUANT_PRODUCT ? ix->d_codes : reinterpret_cast<uint8_t*>(ix->d_bits);
    if ((rc = ix->d_tmp8.ensure(size_t(m) * width))) return rc;
    SDB_CUDA(cudaMemcpyAsync(ix->d_tmp8.p, codes + s0 * width, size_t(m) * width, cudaMemcpyHostToDevice, ix->stream));
    scatter_codes_kernel<<<uint32_t((m * width + 255) / 256), 256, 0, ix->stream>>>(base, pitch, width, ix->d_exists, ix->d_tmp32.p, ix->d_tmp8.p, m);
    ix->launches++;
    SDB_CUDA(cudaGetLastError());
    SDB_CUDA(cudaStreamSynchronize(ix->stream));
    for (uint64_t i = 0; i < m; ++i) {
      if (!ix->h_exists[h32[i]]) {
        ix->h_exists[h32[i]] = 1;
        ix->count++;
      }
      if (h32[i] != START_ID && h32[i] > ix->max_node_id) ix->max_node_id = h32[i];
    }
  }
  ix->vec_epoch++;
  return SDB_OK;
}

int sdb_index_dirty_edges(sdb_index* ix, uint64_t cap, uint64_t* ids_out, uint64_t* n_out, int32_t clear) {
  if (!ix || !n_out || (cap && !ids_out)) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  return dirty_edges_locked(ix, cap, ids_out, n_out, clear);
}

int sdb_pq_adc_tables(sdb_index* ix, uint32_t B, const float* queries, float* out) {
  if (!ix || !queries || !out) return fail(SDB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (!ix->pq_fitted) return fail(SDB_ERR_STATE, "product quantizer is not fitted");
  int rc;
  size_t tsz = size_t(ix->pqM) * ix->pqK;
  if ((rc = ix->d_q.ensure(size_t(B) * ix->p.dim))) return rc;
  if ((rc = ix->d_adc.ensure(size_t(B) * tsz))) return rc;
  SDB_CUDA(cudaMemcpyAsync(ix->d_q.p, queries, size_t(B) * ix->p.dim * 4, cudaMemcpyHostToDevice, ix->stream));
  if ((rc = launch_adc_tables(ix, B, ix->d_q.p, ix->d_adc.p, ix->stream))) return rc;
  SDB_CUDA(cudaMemcpyAsync(out, ix->d_adc.p, size_t(B) * tsz * 4, cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  return SDB_OK;
}

uint32_t sdb_shard_limit(uint32_t limit, uint32_t n_shards, uint32_t max_search_limit) {
  // cluster/actions.go:291-299 (poissonApproxA = 1.42, poissonApproxB = 10.0, f32 math)
  if (n_shards == 0) return limit;
  int target = int(float(limit) * (1 / float(n_shards)) * 1.42f + 10.0f);
  if (target > int(max_search_limit)) target = int(max_search_limit);
  if (target > int(limit)) target = int(limit);
  return uint32_t(target);
}

}  // extern "C"
