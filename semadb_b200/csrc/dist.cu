// dist.cu — the distance family as batched C-ABI calls (distance/distance.go:11-97), the
// store-level closures DistanceFromFloat / DistanceFromPoint evaluated for id lists
// (shard/vectorstore/plain.go:76-97, binary.go:187-234, product.go:238-305), the binary
// encoder (binary.go:103-129), the PQ encoder (product.go:136-159), the ADC table builder
// (product.go:255-263, K4) and the cross-shard top-k merge (cluster/actions.go:357-376, K6).
#include <mutex>
#include <string>

#include "common.cuh"
#include "index.cuh"

namespace sdb {

namespace {

template <int METRIC>
__global__ void pair_dist_kernel(const float* x, const float* y, uint32_t dim, uint64_t n, float* out) {
  uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* a = x + i * dim;
  const float* b = y + i * dim;
  out[i] = (METRIC == METRIC_HAVERSINE) ? haversine_thread(a, b) : float_dist_thread<METRIC>(a, b, int(dim));
}

__global__ void pair_bits_kernel(int metric, const uint64_t* x, const uint64_t* y, uint32_t words, uint64_t n,
                                 float* out) {
  uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int a = 0, u = 0;
  for (uint32_t w = 0; w < words; ++w) {
    uint64_t xv = x[i * words + w], yv = y[i * words + w];
    if (metric == METRIC_JACCARD) { a += __popcll(xv & yv); u += __popcll(xv | yv); }
    else a += __popcll(xv ^ yv);
  }
  out[i] = bits_finish(metric, a, u);
}

// One warp per row: bit i%64 of word i/64 = v[i] > thr[i] (binary.go:123-127).
__global__ void bq_encode_kernel(const float* src, size_t src_pitch, const uint32_t* row_ids /*or null*/,
                                 const float* thr, uint32_t dim, uint32_t words, uint64_t* dst, size_t dst_pitch,
                                 uint64_t n, bool dst_by_id) {
  uint64_t r = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (r >= n) return;
  uint64_t srow = row_ids ? row_ids[r] : r;
  uint64_t drow = dst_by_id ? srow : r;
  const float* v = src + srow * src_pitch;
  for (uint32_t w = 0; w < dst_pitch; ++w) {
    uint64_t word = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t i = w * 64 + h * 32 + lane;
      bool on = (i < dim) && (v[i] > thr[i]);
      word |= uint64_t(__ballot_sync(SDB_FULL, on)) << (32 * h);
    }
    if (lane == 0 && (w < words || dst_by_id)) dst[drow * dst_pitch + w] = word;
  }
}

// productQuantizer.encode (product.go:136-159): one thread per (row, sub-vector); argmin
// over K centroids with the index metric, strict '<' from MaxFloat32 (lowest index wins).
template <int METRIC>
__global__ void pq_encode_kernel(const float* vec, uint32_t pitch, const uint32_t* row_ids, uint32_t n,
                                 const float* cent, uint32_t M, uint32_t K, uint32_t sub, uint8_t* codes,
                                 uint32_t codes_pitch) {
  uint64_t t = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= uint64_t(n) * M) return;
  uint32_t r = uint32_t(t / M), m = uint32_t(t % M);
  uint32_t id = row_ids[r];
  const float* sv = vec + size_t(id) * pitch + m * sub;
  float best = 3.402823466e+38f;
  uint32_t bid = 0;
  for (uint32_t j = 0; j < K; ++j) {
    float d = float_dist_thread<METRIC>(sv, cent + (size_t(m) * K + j) * sub, int(sub));
    if (d < best) { best = d; bid = j; }
  }
  codes[size_t(id) * codes_pitch + m] = uint8_t(bid);
}

// K4: ADC tables, dists[i*K+j] = distFn(x[i*sub:(i+1)*sub], centroid_ij) (product.go:255-263).
template <int METRIC>
__global__ void adc_table_kernel(const float* queries, uint32_t dim, uint32_t B, const float* cent, uint32_t M,
                                 uint32_t K, uint32_t sub, float* out) {
  uint64_t t = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  uint64_t per = uint64_t(M) * K;
  if (t >= uint64_t(B) * per) return;
  uint32_t b = uint32_t(t / per);
  uint32_t mk = uint32_t(t % per);
  uint32_t m = mk / K;
  out[t] = float_dist_thread<METRIC>(queries + size_t(b) * dim + m * sub, cent + size_t(mk) * sub, int(sub));
}

// DistanceFromFloat(query)(id) for a list of ids; mode 0 float, 1 bits, 2 adc.
template <int METRIC>
__global__ void query_dists_float_kernel(const float* vec, uint32_t pitch, const float* q, uint32_t dim,
                                         const uint32_t* ids, uint64_t n, float* out) {
  uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* y = vec + size_t(ids[i]) * pitch;
  out[i] = (METRIC == METRIC_HAVERSINE) ? haversine_thread(q, y) : float_dist_thread<METRIC>(q, y, int(dim));
}
__global__ void query_dists_bits_kernel(int metric, const uint64_t* bits, uint32_t pitch, uint32_t words,
                                        const uint64_t* qb, const uint32_t* ids, uint64_t n, float* out) {
  uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t* y = bits + size_t(ids[i]) * pitch;
  int a = 0, u = 0;
  for (uint32_t w = 0; w < words; ++w) {
    if (metric == METRIC_JACCARD) { a += __popcll(qb[w] & y[w]); u += __popcll(qb[w] | y[w]); }
    else a += __popcll(qb[w] ^ y[w]);
  }
  out[i] = bits_finish(metric, a, u);
}
__global__ void query_dists_adc_kernel(const uint8_t* codes, uint32_t pitch, const float* table, uint32_t M,
                                       uint32_t K, const uint32_t* ids, uint64_t n, float* out) {
  uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t* c = codes + size_t(ids[i]) * pitch;
  float d = 0.0f;
  for (uint32_t m = 0; m < M; ++m) d = __fadd_rn(d, table[m * K + c[m]]);
  out[i] = d;
}
// DistanceFromPoint(x)(id): SDC for fitted PQ (product.go:299-303)
__global__ void point_dists_sdc_kernel(const uint8_t* codes, uint32_t pitch, const float* cdist, uint32_t M,
                                       uint32_t K, uint32_t x, const uint32_t* ids, uint64_t n, float* out) {
  uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t* cx = codes + size_t(x) * pitch;
  const uint8_t* cy = codes + size_t(ids[i]) * pitch;
  float d = 0.0f;
  for (uint32_t m = 0; m < M; ++m) d = __fadd_rn(d, cdist[(size_t(m) * K + cx[m]) * K + cy[m]]);
  out[i] = d;
}

// K6: one thread per query merges S sorted lists; stable by (dist asc, shard asc, rank asc).
// k is the row stride of inputs and outputs; row b keeps limits[b] results (nullptr: k).
__global__ void merge_topk_kernel(uint32_t S, uint32_t B, uint32_t k, const uint64_t* in_ids, const float* in_d,
                                  const uint32_t* in_c, uint64_t* out_ids, float* out_d, uint32_t* out_c,
                                  const uint32_t* limits) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  uint32_t heads[64];  // S <= 64 (checked by launch_merge)
  for (uint32_t s = 0; s < S; ++s) heads[s] = 0;
  const uint32_t lim = limits ? min(limits[b], k) : k;
  uint32_t n = 0;
  for (; n < lim; ++n) {
    int best = -1;
    float bd = 0.0f;
    for (uint32_t s = 0; s < S; ++s) {
      uint32_t c = min(in_c[size_t(s) * B + b], k);
      if (heads[s] >= c) continue;
      float d = in_d[(size_t(s) * B + b) * k + heads[s]];
      // HybridScore = -d descending == d ascending; strict '<' keeps the lower shard on ties
      if (best < 0 || d < bd) { best = int(s); bd = d; }
    }
    if (best < 0) break;
    out_ids[size_t(b) * k + n] = in_ids[(size_t(best) * B + b) * k + heads[best]];
    out_d[size_t(b) * k + n] = bd;
    heads[best]++;
  }
  out_c[b] = n;
  for (uint32_t j = n; j < k; ++j) {
    out_ids[size_t(b) * k + j] = 0;
    out_d[size_t(b) * k + j] = __int_as_float(0x7f800000);
  }
}

// Hybrid-score merge of S sub-searches per request (indexManager.searchParallel,
// shard/index/search.go:211-298): final set = OR / AND of the sub-searches' result-id sets; results
// are walked in sub-search order, rank order; a node seen again adds its HybridScore to the first
// occurrence (f32, in that order) and donates its distance if the first had none (NaN = nil);
// then sort by HybridScore descending. The reference's sort is unstable: ties keep first-appearance
// order here (and in the oracle). One thread per request; lists are S*k <= 1200 entries.
__global__ void hybrid_merge_kernel(uint32_t S, uint32_t B, uint32_t k, int disjunction, const uint64_t* in_ids,
                                    const float* in_h, const float* in_d, const uint32_t* in_c, uint64_t* out_ids,
                                    float* out_h, float* out_d, uint32_t* out_c) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const uint32_t M = S * k;
  uint64_t* oi = out_ids + size_t(b) * M;
  float* oh = out_h + size_t(b) * M;
  float* od = out_d + size_t(b) * M;
  uint32_t n = 0;
  for (uint32_t s = 0; s < S; ++s) {
    const uint32_t cs = min(in_c[size_t(s) * B + b], k);
    for (uint32_t r = 0; r < cs; ++r) {
      const size_t o = (size_t(s) * B + b) * k + r;
      const uint64_t id = in_ids[o];
      if (!disjunction) {  // finalSet.Contains(r.NodeId): present in every sub-search's set
        bool everywhere = true;
        for (uint32_t t = 0; t < S && everywhere; ++t) {
          if (t == s) continue;
          const uint32_t ct = min(in_c[size_t(t) * B + b], k);
          bool found = false;
          for (uint32_t j = 0; j < ct && !found; ++j) found = in_ids[(size_t(t) * B + b) * k + j] == id;
          everywhere = found;
        }
        if (!everywhere) continue;
      }
      uint32_t idx = n;
      for (uint32_t j = 0; j < n; ++j)
        if (oi[j] == id) { idx = j; break; }
      if (idx == n) {
        oi[n] = id;
        oh[n] = in_h[o];
        od[n] = in_d[o];
        ++n;
      } else {
        oh[idx] = __fadd_rn(oh[idx], in_h[o]);
        if (isnan(od[idx]) && !isnan(in_d[o])) od[idx] = in_d[o];
      }
    }
  }
  // stable insertion sort, HybridScore descending
  for (uint32_t i = 1; i < n; ++i) {
    const uint64_t ci = oi[i];
    const float ch = oh[i], cd = od[i];
    uint32_t j = i;
    while (j > 0 && oh[j - 1] < ch) {
      oi[j] = oi[j - 1];
      oh[j] = oh[j - 1];
      od[j] = od[j - 1];
      --j;
    }
    oi[j] = ci;
    oh[j] = ch;
    od[j] = cd;
  }
  out_c[b] = n;
  for (uint32_t j = n; j < M; ++j) {
    oi[j] = 0;
    oh[j] = -__int_as_float(0x7f800000);
    od[j] = __int_as_float(0x7f800000);
  }
}

int set_device_checked(int device) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(SDB_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
  }
  if (device < 0 || device >= ndev) return fail(SDB_ERR_INVALID, "device ordinal out of range");
  SDB_CUDA(cudaSetDevice(device));
  return SDB_OK;
}

struct TmpDev {
  void* p = nullptr;
  ~TmpDev() { if (p) cudaFree(p); }
  int alloc(size_t bytes) {
    cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(tmp)");
    return SDB_OK;
  }
};

}  // namespace

int launch_encode_rows(sdb_index* ix, uint32_t n, const uint32_t* d_ids, cudaStream_t stream) {
  if (n == 0) return SDB_OK;
  if (ix->p.quantizer == SDB_QUANT_BINARY && ix->bq_fitted) {
    uint32_t threads = 128, rows_per_block = threads / 32;
    bq_encode_kernel<<<(n + rows_per_block - 1) / rows_per_block, threads, 0, stream>>>(
        ix->d_vec, ix->vec_pitch, d_ids, ix->d_bq_thr, ix->p.dim, ix->words, ix->d_bits, ix->bits_pitch, n, true);
    ix->launches++;
    SDB_CUDA(cudaGetLastError());
  } else if (ix->p.quantizer == SDB_QUANT_PRODUCT && ix->pq_fitted) {
    uint64_t total = uint64_t(n) * ix->pqM;
    uint32_t blocks = uint32_t((total + 127) / 128);
    switch (ix->store_metric) {
      case SDB_METRIC_EUCLIDEAN:
        pq_encode_kernel<METRIC_EUCLIDEAN><<<blocks, 128, 0, stream>>>(ix->d_vec, ix->vec_pitch, d_ids, n, ix->d_pq_centroids, ix->pqM, ix->pqK, ix->pqSub, ix->d_codes, ix->codes_pitch);
        break;
      case SDB_METRIC_DOT:
        pq_encode_kernel<METRIC_DOT><<<blocks, 128, 0, stream>>>(ix->d_vec, ix->vec_pitch, d_ids, n, ix->d_pq_centroids, ix->pqM, ix->pqK, ix->pqSub, ix->d_codes, ix->codes_pitch);
        break;
      default: return fail(SDB_ERR_INTERNAL, "unexpected PQ metric");
    }
    ix->launches++;
    SDB_CUDA(cudaGetLastError());
  }
  return SDB_OK;
}

int launch_adc_tables(sdb_index* ix, uint32_t B, const float* d_queries, float* d_out, cudaStream_t stream) {
  uint64_t total = uint64_t(B) * ix->pqM * ix->pqK;
  uint32_t blocks = uint32_t((total + 255) / 256);
  if (ix->store_metric == SDB_METRIC_EUCLIDEAN)
    adc_table_kernel<METRIC_EUCLIDEAN><<<blocks, 256, 0, stream>>>(d_queries, ix->p.dim, B, ix->d_pq_centroids, ix->pqM, ix->pqK, ix->pqSub, d_out);
  else if (ix->store_metric == SDB_METRIC_DOT)
    adc_table_kernel<METRIC_DOT><<<blocks, 256, 0, stream>>>(d_queries, ix->p.dim, B, ix->d_pq_centroids, ix->pqM, ix->pqK, ix->pqSub, d_out);
  else return fail(SDB_ERR_INTERNAL, "unexpected PQ metric");
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

int launch_merge(uint32_t S, uint32_t B, uint32_t k, const uint64_t* in_ids, const float* in_d, const uint32_t* in_c,
                 uint64_t* out_ids, float* out_d, uint32_t* out_c, cudaStream_t stream, const uint32_t* limits) {
  if (S == 0 || S > 64) return fail(SDB_ERR_INVALID, "merge supports 1..64 shards");
  merge_topk_kernel<<<(B + 127) / 128, 128, 0, stream>>>(S, B, k, in_ids, in_d, in_c, out_ids, out_d, out_c, limits);
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

// Cross-GPU barrier on peer-mapped flag words (NVLink): thread p publishes `epoch` into peer
// p's flags[me] with a system-scope release (the peer stores of the kernels before it on this
// stream are ordered first), then waits until peer p's epoch has arrived in flags_me[p].
// Epochs only grow, so the words are never reset. A peer that never arrives (a crashed rank)
// is given ~20 s; then the kernel records the failure in flags_me[SDB_MAX_PEERS + p] AND in the
// library's page-locked status word of this device, which every later exchange call on the
// device (and sdb_peer_barrier_check) reads on the host without a synchronisation and turns
// into SDB_ERR_STATE: the merge that follows a timed-out barrier read stale slots.
struct PeerFlags { uint32_t* f[SDB_MAX_PEERS]; };
__global__ void peer_barrier_kernel(PeerFlags pf, uint32_t n, uint32_t me, uint32_t epoch, uint32_t* host_status) {
  const uint32_t p = threadIdx.x;
  if (p >= n) return;
  __threadfence_system();
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(pf.f[p] + me), "r"(epoch) : "memory");
  const uint32_t* mine = pf.f[me] + p;
  const long long t0 = clock64();
  uint32_t v;
  for (;;) {
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
    if (int32_t(v - epoch) >= 0) break;
    if (clock64() - t0 > 40000000000LL) {
      pf.f[me][SDB_MAX_PEERS + p] = epoch;
      if (host_status) {
        host_status[1] = p;
        __threadfence_system();
        host_status[0] = epoch;  // non-zero = a barrier of this device timed out at that epoch
        __threadfence_system();
      }
      break;
    }
    __nanosleep(200);
  }
}

// one {epoch, peer} pair of page-locked, device-mapped words per device, allocated on first use
constexpr int kMaxDevices = 64;
static volatile uint32_t* g_barrier_status[kMaxDevices] = {};
static std::mutex g_barrier_mu;
static int barrier_status_word(int device, volatile uint32_t** out) {
  if (device < 0 || device >= kMaxDevices) return fail(SDB_ERR_INVALID, "device ordinal out of range");
  std::lock_guard<std::mutex> g(g_barrier_mu);
  if (!g_barrier_status[device]) {
    void* p = nullptr;
    SDB_CUDA(cudaHostAlloc(&p, 2 * sizeof(uint32_t), cudaHostAllocMapped | cudaHostAllocPortable));
    static_cast<uint32_t*>(p)[0] = 0;
    static_cast<uint32_t*>(p)[1] = 0;
    g_barrier_status[device] = static_cast<volatile uint32_t*>(p);
  }
  *out = g_barrier_status[device];
  return SDB_OK;
}
// SDB_ERR_STATE if a peer barrier on this device has timed out (sticky until cleared)
int peer_barrier_poisoned(int device) {
  if (device < 0 || device >= kMaxDevices) return SDB_OK;
  volatile uint32_t* w = g_barrier_status[device];
  if (!w || w[0] == 0) return SDB_OK;
  return fail(SDB_ERR_STATE, "cross-GPU barrier timed out at epoch " + std::to_string(w[0]) + " waiting for peer " +
                                 std::to_string(w[1]) + ": the merged lists of that step are invalid");
}

}  // namespace sdb

using namespace sdb;

extern "C" {

int sdb_distance_float(int32_t metric, int32_t device, uint64_t n, uint32_t dim, const float* x, const float* y,
                       float* out) {
  if (n == 0) return SDB_OK;
  if (!x || !y || !out || dim == 0) return fail(SDB_ERR_INVALID, "null argument");
  if (metric == SDB_METRIC_HAVERSINE && dim != 2) return fail(SDB_ERR_INVALID, "haversine needs dim 2");
  int rc = set_device_checked(device);
  if (rc) return rc;
  TmpDev dx, dy, dout;
  size_t bytes = size_t(n) * dim * sizeof(float);
  if ((rc = dx.alloc(bytes)) || (rc = dy.alloc(bytes)) || (rc = dout.alloc(n * sizeof(float)))) return rc;
  SDB_CUDA(cudaMemcpy(dx.p, x, bytes, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(dy.p, y, bytes, cudaMemcpyHostToDevice));
  uint32_t blocks = uint32_t((n + 127) / 128);
  const float* a = static_cast<const float*>(dx.p);
  const float* b = static_cast<const float*>(dy.p);
  float* o = static_cast<float*>(dout.p);
  switch (metric) {
    case SDB_METRIC_EUCLIDEAN: pair_dist_kernel<METRIC_EUCLIDEAN><<<blocks, 128>>>(a, b, dim, n, o); break;
    case SDB_METRIC_DOT: pair_dist_kernel<METRIC_DOT><<<blocks, 128>>>(a, b, dim, n, o); break;
    case SDB_METRIC_COSINE: pair_dist_kernel<METRIC_COSINE><<<blocks, 128>>>(a, b, dim, n, o); break;
    case SDB_METRIC_HAVERSINE: pair_dist_kernel<METRIC_HAVERSINE><<<blocks, 128>>>(a, b, dim, n, o); break;
    default: return fail(SDB_ERR_INVALID, "unknown float32 distance function");  // distance.go:82
  }
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaMemcpy(out, dout.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return SDB_OK;
}

int sdb_distance_bits(int32_t metric, int32_t device, uint64_t n, uint32_t words, const uint64_t* x,
                      const uint64_t* y, float* out) {
  if (n == 0) return SDB_OK;
  if (!x || !y || !out) return fail(SDB_ERR_INVALID, "null argument");
  if (metric != SDB_METRIC_HAMMING && metric != SDB_METRIC_JACCARD) return fail(SDB_ERR_INVALID, "unknown bit distance function");  // distance.go:95
  int rc = set_device_checked(device);
  if (rc) return rc;
  TmpDev dx, dy, dout;
  size_t bytes = size_t(n) * words * 8;
  if ((rc = dx.alloc(bytes)) || (rc = dy.alloc(bytes)) || (rc = dout.alloc(n * sizeof(float)))) return rc;
  SDB_CUDA(cudaMemcpy(dx.p, x, bytes, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(dy.p, y, bytes, cudaMemcpyHostToDevice));
  pair_bits_kernel<<<uint32_t((n + 127) / 128), 128>>>(metric, static_cast<const uint64_t*>(dx.p), static_cast<const uint64_t*>(dy.p), words, n, static_cast<float*>(dout.p));
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaMemcpy(out, dout.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return SDB_OK;
}

int sdb_bq_encode(int32_t device, uint64_t n, uint32_t dim, const float* vectors, const float* threshold,
                  uint64_t* out) {
  if (n == 0) return SDB_OK;
  if (!vectors || !threshold || !out || dim == 0) return fail(SDB_ERR_INVALID, "null argument");
  int rc = set_device_checked(device);
  if (rc) return rc;
  uint32_t words = (dim + 63) / 64;
  TmpDev dv, dt, dout;
  if ((rc = dv.alloc(size_t(n) * dim * 4)) || (rc = dt.alloc(size_t(dim) * 4)) || (rc = dout.alloc(size_t(n) * words * 8))) return rc;
  SDB_CUDA(cudaMemcpy(dv.p, vectors, size_t(n) * dim * 4, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(dt.p, threshold, size_t(dim) * 4, cudaMemcpyHostToDevice));
  bq_encode_kernel<<<uint32_t((n + 3) / 4), 128>>>(static_cast<const float*>(dv.p), dim, nullptr, static_cast<const float*>(dt.p), dim, words, static_cast<uint64_t*>(dout.p), words, n, false);
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaMemcpy(out, dout.p, size_t(n) * words * 8, cudaMemcpyDeviceToHost));
  return SDB_OK;
}

static int stage_id_list(sdb_index* ix, uint64_t n, const uint64_t* ids) {
  std::vector<uint32_t> h(n);
  for (uint64_t i = 0; i < n; ++i) {
    // a point of the wrong type yields MaxFloat32 in the reference (plain.go:78-82); an id
    // that is not stored is an error here
    if (ids[i] >= ix->rows || !ix->h_exists[ids[i]]) return fail(SDB_ERR_NOTFOUND, "node id does not exist: " + std::to_string(ids[i]));
    h[i] = uint32_t(ids[i]);
  }
  int rc = ix->d_tmp32.ensure(n + 1);
  if (rc) return rc;
  SDB_CUDA(cudaMemcpy(ix->d_tmp32.p, h.data(), n * 4, cudaMemcpyHostToDevice));
  return SDB_OK;
}

int sdb_index_query_dists(sdb_index* ix, const float* query, uint64_t n, const uint64_t* ids, float* out) {
  if (!ix || !query || (n && (!ids || !out))) return fail(SDB_ERR_INVALID, "null argument");
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  int rc = stage_id_list(ix, n, ids);
  if (rc) return rc;
  if ((rc = ix->d_q.ensure(ix->p.dim))) return rc;
  if ((rc = ix->d_tmpf.ensure(n))) return rc;
  SDB_CUDA(cudaMemcpyAsync(ix->d_q.p, query, ix->p.dim * 4, cudaMemcpyHostToDevice, ix->stream));
  uint32_t blocks = uint32_t((n + 127) / 128);
  if (ix->p.quantizer == SDB_QUANT_BINARY && ix->bq_fitted) {
    if ((rc = ix->d_ids64.ensure(ix->bits_pitch))) return rc;
    bq_encode_kernel<<<1, 32, 0, ix->stream>>>(ix->d_q.p, ix->p.dim, nullptr, ix->d_bq_thr, ix->p.dim, ix->words, ix->d_ids64.p, ix->bits_pitch, 1, true);
    query_dists_bits_kernel<<<blocks, 128, 0, ix->stream>>>(ix->bq_metric, ix->d_bits, ix->bits_pitch, ix->words, ix->d_ids64.p, ix->d_tmp32.p, n, ix->d_tmpf.p);
    ix->launches += 2;
  } else if (ix->p.quantizer == SDB_QUANT_PRODUCT && ix->pq_fitted) {
    if ((rc = ix->d_adc.ensure(size_t(ix->pqM) * ix->pqK))) return rc;
    if ((rc = launch_adc_tables(ix, 1, ix->d_q.p, ix->d_adc.p, ix->stream))) return rc;
    query_dists_adc_kernel<<<blocks, 128, 0, ix->stream>>>(ix->d_codes, ix->codes_pitch, ix->d_adc.p, ix->pqM, ix->pqK, ix->d_tmp32.p, n, ix->d_tmpf.p);
    ix->launches++;
  } else {
    switch (ix->store_metric) {
      case SDB_METRIC_EUCLIDEAN: query_dists_float_kernel<METRIC_EUCLIDEAN><<<blocks, 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, ix->d_q.p, ix->p.dim, ix->d_tmp32.p, n, ix->d_tmpf.p); break;
      case SDB_METRIC_DOT: query_dists_float_kernel<METRIC_DOT><<<blocks, 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, ix->d_q.p, ix->p.dim, ix->d_tmp32.p, n, ix->d_tmpf.p); break;
      case SDB_METRIC_COSINE: query_dists_float_kernel<METRIC_COSINE><<<blocks, 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, ix->d_q.p, ix->p.dim, ix->d_tmp32.p, n, ix->d_tmpf.p); break;
      case SDB_METRIC_HAVERSINE: query_dists_float_kernel<METRIC_HAVERSINE><<<blocks, 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, ix->d_q.p, ix->p.dim, ix->d_tmp32.p, n, ix->d_tmpf.p); break;
      default: return fail(SDB_ERR_INVALID, "metric has no float distance");
    }
    ix->launches++;
  }
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaMemcpyAsync(out, ix->d_tmpf.p, n * 4, cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  return SDB_OK;
}

int sdb_index_point_dists(sdb_index* ix, uint64_t x, uint64_t n, const uint64_t* ids, float* out) {
  if (!ix || (n && (!ids || !out))) return fail(SDB_ERR_INVALID, "null argument");
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (x >= ix->rows || !ix->h_exists[x]) return fail(SDB_ERR_NOTFOUND, "node id does not exist: " + std::to_string(x));
  int rc = stage_id_list(ix, n, ids);
  if (rc) return rc;
  if ((rc = ix->d_tmpf.ensure(n))) return rc;
  uint32_t blocks = uint32_t((n + 127) / 128);
  if (ix->p.quantizer == SDB_QUANT_BINARY && ix->bq_fitted) {
    query_dists_bits_kernel<<<blocks, 128, 0, ix->stream>>>(ix->bq_metric, ix->d_bits, ix->bits_pitch, ix->words, ix->d_bits + size_t(x) * ix->bits_pitch, ix->d_tmp32.p, n, ix->d_tmpf.p);
  } else if (ix->p.quantizer == SDB_QUANT_PRODUCT && ix->pq_fitted) {
    point_dists_sdc_kernel<<<blocks, 128, 0, ix->stream>>>(ix->d_codes, ix->codes_pitch, ix->d_pq_cdist, ix->pqM, ix->pqK, uint32_t(x), ix->d_tmp32.p, n, ix->d_tmpf.p);
  } else {
    const float* xv = ix->d_vec + size_t(x) * ix->vec_pitch;
    switch (ix->store_metric) {
      case SDB_METRIC_EUCLIDEAN: query_dists_float_kernel<METRIC_EUCLIDEAN><<<blocks, 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, xv, ix->p.dim, ix->d_tmp32.p, n, ix->d_tmpf.p); break;
      case SDB_METRIC_DOT: query_dists_float_kernel<METRIC_DOT><<<blocks, 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, xv, ix->p.dim, ix->d_tmp32.p, n, ix->d_tmpf.p); break;
      case SDB_METRIC_COSINE: query_dists_float_kernel<METRIC_COSINE><<<blocks, 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, xv, ix->p.dim, ix->d_tmp32.p, n, ix->d_tmpf.p); break;
      case SDB_METRIC_HAVERSINE: query_dists_float_kernel<METRIC_HAVERSINE><<<blocks, 128, 0, ix->stream>>>(ix->d_vec, ix->vec_pitch, xv, ix->p.dim, ix->d_tmp32.p, n, ix->d_tmpf.p); break;
      default: return fail(SDB_ERR_INVALID, "metric has no float distance");
    }
  }
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaMemcpyAsync(out, ix->d_tmpf.p, n * 4, cudaMemcpyDeviceToHost, ix->stream));
  SDB_CUDA(cudaStreamSynchronize(ix->stream));
  return SDB_OK;
}

int sdb_merge_topk_device(int32_t device, uint32_t S, uint32_t B, uint32_t k, const uint64_t* d_in_ids,
                          const float* d_in_dists, const uint32_t* d_in_counts, uint64_t* d_out_ids,
                          float* d_out_dists, uint32_t* d_out_counts, void* stream) {
  if (B == 0) return SDB_OK;
  if (!d_in_ids || !d_in_dists || !d_in_counts || !d_out_ids || !d_out_dists || !d_out_counts) return fail(SDB_ERR_INVALID, "null argument");
  if (k < 1 || k > 75) return fail(SDB_ERR_INVALID, "invalid limit");
  int rc = set_device_checked(device);
  if (rc) return rc;
  if ((rc = peer_barrier_poisoned(device))) return rc;  // an earlier cross-GPU barrier on this device timed out
  return launch_merge(S, B, k, d_in_ids, d_in_dists, d_in_counts, d_out_ids, d_out_dists, d_out_counts, static_cast<cudaStream_t>(stream));
}

int sdb_merge_topk_requests_device(int32_t device, uint32_t S, uint32_t B, uint32_t k_stride, const uint32_t* d_limits,
                                   const uint64_t* d_in_ids, const float* d_in_dists, const uint32_t* d_in_counts,
                                   uint64_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, void* stream) {
  if (B == 0) return SDB_OK;
  if (!d_limits || !d_in_ids || !d_in_dists || !d_in_counts || !d_out_ids || !d_out_dists || !d_out_counts)
    return fail(SDB_ERR_INVALID, "null argument");
  if (k_stride < 1 || k_stride > 75) return fail(SDB_ERR_INVALID, "invalid limit");
  int rc = set_device_checked(device);
  if (rc) return rc;
  if ((rc = peer_barrier_poisoned(device))) return rc;
  return launch_merge(S, B, k_stride, d_in_ids, d_in_dists, d_in_counts, d_out_ids, d_out_dists, d_out_counts,
                      static_cast<cudaStream_t>(stream), d_limits);
}

int sdb_merge_topk(int32_t device, uint32_t S, uint32_t B, uint32_t k, const uint64_t* in_ids, const float* in_dists,
                   const uint32_t* in_counts, uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  if (B == 0) return SDB_OK;
  if (!in_ids || !in_dists || !in_counts || !out_ids || !out_dists || !out_counts) return fail(SDB_ERR_INVALID, "null argument");
  if (k < 1 || k > 75) return fail(SDB_ERR_INVALID, "invalid limit");
  int rc = set_device_checked(device);
  if (rc) return rc;
  size_t n = size_t(S) * B * k;
  TmpDev di, dd, dc, oi, od, oc;
  if ((rc = di.alloc(n * 8)) || (rc = dd.alloc(n * 4)) || (rc = dc.alloc(size_t(S) * B * 4)) ||
      (rc = oi.alloc(size_t(B) * k * 8)) || (rc = od.alloc(size_t(B) * k * 4)) || (rc = oc.alloc(size_t(B) * 4))) return rc;
  SDB_CUDA(cudaMemcpy(di.p, in_ids, n * 8, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(dd.p, in_dists, n * 4, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(dc.p, in_counts, size_t(S) * B * 4, cudaMemcpyHostToDevice));
  rc = launch_merge(S, B, k, static_cast<uint64_t*>(di.p), static_cast<float*>(dd.p), static_cast<uint32_t*>(dc.p),
                    static_cast<uint64_t*>(oi.p), static_cast<float*>(od.p), static_cast<uint32_t*>(oc.p), nullptr);
  if (rc) return rc;
  SDB_CUDA(cudaMemcpy(out_ids, oi.p, size_t(B) * k * 8, cudaMemcpyDeviceToHost));
  SDB_CUDA(cudaMemcpy(out_dists, od.p, size_t(B) * k * 4, cudaMemcpyDeviceToHost));
  SDB_CUDA(cudaMemcpy(out_counts, oc.p, size_t(B) * 4, cudaMemcpyDeviceToHost));
  return SDB_OK;
}

int sdb_hybrid_merge(int32_t device, uint32_t S, uint32_t B, uint32_t k, int32_t disjunction, const uint64_t* in_ids,
                     const float* in_hybrid, const float* in_dists, const uint32_t* in_counts, uint64_t* out_ids,
                     float* out_hybrid, float* out_dists, uint32_t* out_counts) {
  if (B == 0) return SDB_OK;
  if (!in_ids || !in_hybrid || !in_dists || !in_counts || !out_ids || !out_hybrid || !out_dists || !out_counts)
    return fail(SDB_ERR_INVALID, "null argument");
  if (S < 1 || S > 16 || k < 1 || k > 75) return fail(SDB_ERR_INVALID, "hybrid merge supports 1..16 sub-searches of limit 1..75");
  int rc = set_device_checked(device);
  if (rc) return rc;
  const size_t n = size_t(S) * B * k;
  TmpDev di, dh, dd, dc, oi, oh, od, oc;
  if ((rc = di.alloc(n * 8)) || (rc = dh.alloc(n * 4)) || (rc = dd.alloc(n * 4)) || (rc = dc.alloc(size_t(S) * B * 4)) ||
      (rc = oi.alloc(n * 8)) || (rc = oh.alloc(n * 4)) || (rc = od.alloc(n * 4)) || (rc = oc.alloc(size_t(B) * 4)))
    return rc;
  SDB_CUDA(cudaMemcpy(di.p, in_ids, n * 8, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(dh.p, in_hybrid, n * 4, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(dd.p, in_dists, n * 4, cudaMemcpyHostToDevice));
  SDB_CUDA(cudaMemcpy(dc.p, in_counts, size_t(S) * B * 4, cudaMemcpyHostToDevice));
  hybrid_merge_kernel<<<(B + 63) / 64, 64>>>(S, B, k, disjunction, static_cast<uint64_t*>(di.p), static_cast<float*>(dh.p),
                                             static_cast<float*>(dd.p), static_cast<uint32_t*>(dc.p), static_cast<uint64_t*>(oi.p),
                                             static_cast<float*>(oh.p), static_cast<float*>(od.p), static_cast<uint32_t*>(oc.p));
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaMemcpy(out_ids, oi.p, n * 8, cudaMemcpyDeviceToHost));
  SDB_CUDA(cudaMemcpy(out_hybrid, oh.p, n * 4, cudaMemcpyDeviceToHost));
  SDB_CUDA(cudaMemcpy(out_dists, od.p, n * 4, cudaMemcpyDeviceToHost));
  SDB_CUDA(cudaMemcpy(out_counts, oc.p, size_t(B) * 4, cudaMemcpyDeviceToHost));
  return SDB_OK;
}

int sdb_peer_barrier_device(int32_t device, uint32_t n_peers, uint32_t me, uint32_t* const* peer_flags, uint32_t epoch,
                            void* stream) {
  if (!peer_flags || n_peers == 0 || n_peers > SDB_MAX_PEERS || me >= n_peers)
    return fail(SDB_ERR_INVALID, "peer barrier: n_peers must be 1..16 and me < n_peers");
  int rc = set_device_checked(device);
  if (rc) return rc;
  PeerFlags pf{};
  for (uint32_t p = 0; p < n_peers; ++p) {
    if (!peer_flags[p]) return fail(SDB_ERR_INVALID, "peer barrier: null flag pointer");
    pf.f[p] = peer_flags[p];
  }
  if ((rc = peer_barrier_poisoned(device))) return rc;
  volatile uint32_t* status = nullptr;
  if ((rc = barrier_status_word(device, &status))) return rc;
  uint32_t* d_status = nullptr;
  SDB_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d_status), const_cast<uint32_t*>(status), 0));
  peer_barrier_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(pf, n_peers, me, epoch, d_status);
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

int sdb_peer_barrier_check(int32_t device, int32_t clear) {
  int rc = peer_barrier_poisoned(device);
  if (rc && clear && device >= 0 && device < kMaxDevices && g_barrier_status[device]) {
    g_barrier_status[device][0] = 0;
    g_barrier_status[device][1] = 0;
  }
  return rc;
}

}  // extern "C"
