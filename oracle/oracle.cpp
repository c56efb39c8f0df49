// oracle.cpp — CPU restatement of SemaDB's vector-search hot path.
//
// TEST INFRASTRUCTURE ONLY. Nothing in the product path (semadb_b200/, the C-ABI
// library, bench.py's GPU arm) may link, import or execute this file. It exists so
// that tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
// reference legs have something to check the CUDA path against and to time on the
// host cores.
//
// The Go reference (github.com/semafind/semadb) cannot be built in this image (no Go
// toolchain), so this is a behavioural restatement in C++17, NOT a copy: flat
// arrays, dense u32 node ids, epoch-stamped visited set. Each function cites the
// reference file:line it follows (paths relative to /root/reference).
//
// Parity pinning: tests/test_oracle_kat.py replays every exact known-answer test
// the reference holds for this path (distance/distance_test.go:9-57,
// shard/vectorstore/binary_test.go:11-39, shard/index/vamana/distset_test.go:41-74)
// and the property tests (vamana_test.go:29-46,230-252; flat_test.go:134-191;
// kmeans_test.go:15-91; vectorestore_test.go:112-154) against this file.
//
// Build: see oracle/Makefile (g++ -O2 -mavx2 -mfma, never -ffast-math).

#include <immintrin.h>
#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

namespace {

// ---------------------------------------------------------------------------
// Distances
// ---------------------------------------------------------------------------

enum Metric : int {
  M_EUCLIDEAN = 0,  // squared L2 (distance/distance.go:14-16)
  M_DOT = 1,        // -dot      (distance/distance.go:19-21)
  M_COSINE = 2,     // 1-dot     (distance/distance.go:23-25), no normalisation
  M_HAMMING = 3,    // distance/distance.go:45-54
  M_JACCARD = 4,    // distance/distance.go:56-67
  M_HAVERSINE = 5,  // distance/distance.go:33-43
};

// distance/asm/euclidean.s:7-65 — 4 YMM accumulators x 8 lanes, 32 floats per trip,
// VSUBPS then VFMADD231PS, scalar FMA tail, reduction ((a0+a1)+a2)+a3, lo128+hi128,
// +tail in lane 0, two VHADDPS.
float sq_l2_avx(const float* x, const float* y, size_t n) {
  __m256 a0 = _mm256_setzero_ps(), a1 = a0, a2 = a0, a3 = a0;
  while (n >= 32) {
    __m256 d0 = _mm256_sub_ps(_mm256_loadu_ps(x), _mm256_loadu_ps(y));
    a0 = _mm256_fmadd_ps(d0, d0, a0);
    __m256 d1 = _mm256_sub_ps(_mm256_loadu_ps(x + 8), _mm256_loadu_ps(y + 8));
    a1 = _mm256_fmadd_ps(d1, d1, a1);
    __m256 d2 = _mm256_sub_ps(_mm256_loadu_ps(x + 16), _mm256_loadu_ps(y + 16));
    a2 = _mm256_fmadd_ps(d2, d2, a2);
    __m256 d3 = _mm256_sub_ps(_mm256_loadu_ps(x + 24), _mm256_loadu_ps(y + 24));
    a3 = _mm256_fmadd_ps(d3, d3, a3);
    x += 32; y += 32; n -= 32;
  }
  __m128 tail = _mm_setzero_ps();
  while (n > 0) {
    __m128 d = _mm_sub_ss(_mm_load_ss(x), _mm_load_ss(y));
    tail = _mm_fmadd_ss(d, d, tail);
    ++x; ++y; --n;
  }
  a0 = _mm256_add_ps(a0, a1);
  a0 = _mm256_add_ps(a0, a2);
  a0 = _mm256_add_ps(a0, a3);
  __m128 lo = _mm256_castps256_ps128(a0);
  __m128 hi = _mm256_extractf128_ps(a0, 1);
  lo = _mm_add_ps(lo, hi);
  lo = _mm_add_ps(lo, tail);
  lo = _mm_hadd_ps(lo, lo);
  lo = _mm_hadd_ps(lo, lo);
  return _mm_cvtss_f32(lo);
}

// distance/asm/dot.s:7-55 — same skeleton, VFMADD231PS straight from memory.
float dot_avx(const float* x, const float* y, size_t n) {
  __m256 a0 = _mm256_setzero_ps(), a1 = a0, a2 = a0, a3 = a0;
  while (n >= 32) {
    a0 = _mm256_fmadd_ps(_mm256_loadu_ps(x), _mm256_loadu_ps(y), a0);
    a1 = _mm256_fmadd_ps(_mm256_loadu_ps(x + 8), _mm256_loadu_ps(y + 8), a1);
    a2 = _mm256_fmadd_ps(_mm256_loadu_ps(x + 16), _mm256_loadu_ps(y + 16), a2);
    a3 = _mm256_fmadd_ps(_mm256_loadu_ps(x + 24), _mm256_loadu_ps(y + 24), a3);
    x += 32; y += 32; n -= 32;
  }
  __m128 tail = _mm_setzero_ps();
  while (n > 0) {
    tail = _mm_fmadd_ss(_mm_load_ss(x), _mm_load_ss(y), tail);
    ++x; ++y; --n;
  }
  a0 = _mm256_add_ps(a0, a1);
  a0 = _mm256_add_ps(a0, a2);
  a0 = _mm256_add_ps(a0, a3);
  __m128 lo = _mm256_castps256_ps128(a0);
  __m128 hi = _mm256_extractf128_ps(a0, 1);
  lo = _mm_add_ps(lo, hi);
  lo = _mm_add_ps(lo, tail);
  lo = _mm_hadd_ps(lo, lo);
  lo = _mm_hadd_ps(lo, lo);
  return _mm_cvtss_f32(lo);
}

// Scalar model of the two asm kernels' summation order (SURVEY.md §7.3-①). This is
// the order the CUDA kernels implement; tests assert model == avx bit-for-bit.
float ordered_model(const float* x, const float* y, size_t n, bool l2) {
  float acc[32];
  for (int i = 0; i < 32; ++i) acc[i] = 0.0f;
  size_t blocks = n / 32;
  for (size_t t = 0; t < blocks; ++t)
    for (int i = 0; i < 32; ++i) {
      float a = x[t * 32 + i], b = y[t * 32 + i];
      if (l2) { float d = a - b; acc[i] = std::fmaf(d, d, acc[i]); }
      else acc[i] = std::fmaf(a, b, acc[i]);
    }
  float tail = 0.0f;
  for (size_t i = blocks * 32; i < n; ++i) {
    float a = x[i], b = y[i];
    if (l2) { float d = a - b; tail = std::fmaf(d, d, tail); }
    else tail = std::fmaf(a, b, tail);
  }
  float v[8];
  for (int l = 0; l < 8; ++l) v[l] = ((acc[l] + acc[8 + l]) + acc[16 + l]) + acc[24 + l];
  float w[4];
  for (int l = 0; l < 4; ++l) w[l] = v[l] + v[4 + l];
  w[0] = w[0] + tail;
  w[1] = w[1] + 0.0f; w[2] = w[2] + 0.0f; w[3] = w[3] + 0.0f;
  return (w[0] + w[1]) + (w[2] + w[3]);
}

// distance/puredist.go:3-18 (no FMA on amd64: separate multiply and add).
float sq_l2_pure(const float* x, const float* y, size_t n) {
  volatile float sum = 0;
  for (size_t i = 0; i < n; ++i) {
    volatile float diff = x[i] - y[i];
    volatile float p = diff * diff;
    sum = sum + p;
  }
  return sum;
}
float dot_pure(const float* x, const float* y, size_t n) {
  volatile float sum = 0;
  for (size_t i = 0; i < n; ++i) {
    volatile float p = x[i] * y[i];
    sum = sum + p;
  }
  return sum;
}

// distance/distance.go:33-43
float haversine(const float* x, const float* y) {
  const double degToRad = M_PI / 180.0, earthRadius = 6371000.0;
  double latx = double(x[0]) * degToRad, lonx = double(x[1]) * degToRad;
  double laty = double(y[0]) * degToRad, lony = double(y[1]) * degToRad;
  double dlat = latx - laty, dlon = lonx - lony;
  double sdlat = std::sin(dlat / 2), sdlon = std::sin(dlon / 2);
  double a = sdlat * sdlat + std::cos(latx) * std::cos(laty) * sdlon * sdlon;
  double c = 2 * std::asin(std::sqrt(a));
  return float(earthRadius * c);
}

// distance/distance.go:70-83 (GetFloatDistanceFn) with the asm kernels selected as
// distance_amd64.go:19-23 does on AVX2+FMA hosts.
float float_dist(int metric, const float* x, const float* y, size_t n) {
  switch (metric) {
    case M_EUCLIDEAN: return sq_l2_avx(x, y, n);
    case M_DOT: return -dot_avx(x, y, n);
    case M_COSINE: return 1.0f - dot_avx(x, y, n);
    case M_HAVERSINE: return haversine(x, y);
    default: return FLT_MAX;
  }
}

// distance/distance.go:45-54
float hamming(const uint64_t* x, const uint64_t* y, size_t words) {
  int dist = 0;
  for (size_t i = 0; i < words; ++i) dist += __builtin_popcountll(x[i] ^ y[i]);
  return float(dist);
}
// distance/distance.go:56-67
float jaccard(const uint64_t* x, const uint64_t* y, size_t words) {
  int inter = 0, uni = 0;
  for (size_t i = 0; i < words; ++i) {
    inter += __builtin_popcountll(x[i] & y[i]);
    uni += __builtin_popcountll(x[i] | y[i]);
  }
  if (uni == 0) return 0.0f;
  return 1.0f - float(inter) / float(uni);
}
float bit_dist(int metric, const uint64_t* x, const uint64_t* y, size_t words) {
  return metric == M_JACCARD ? jaccard(x, y, words) : hamming(x, y, words);
}

// shard/vectorstore/binary.go:103-129 — bit i%64 of word i/64 set iff v[i] > threshold[i].
void bq_encode(const float* v, const float* thr, int dim, uint64_t* out) {
  int words = (dim + 63) / 64;
  for (int w = 0; w < words; ++w) out[w] = 0;
  for (int i = 0; i < dim; ++i)
    if (v[i] > thr[i]) out[i / 64] |= (uint64_t(1) << (i % 64));
}

// ---------------------------------------------------------------------------
// k-means (utils/kmeans.go:34-150)
// ---------------------------------------------------------------------------
// X is n rows of `stride` floats; the sub-vector is X[r][offset:offset+len].
// alias=true reproduces the reference quirk: centroids are sub-slices of the input
// rows (kmeans.go:63,82) so the update step (kmeans.go:144) writes through into X.
// alias=false copies the initial centres out ("clean" mode, what the GPU matches).
// first = index of the first centre (the reference draws rand.IntN(n), kmeans.go:61).
// Returns the number of assign/update iterations executed.
int kmeans_fit(float* X, size_t n, size_t stride, int offset, int len, int K, int maxIter,
               size_t first, bool alias, float* centroids_out /*K*len*/, uint8_t* labels /*n*/,
               int64_t* init_rows_out /*K or null*/) {
  std::vector<float> cdist(n, FLT_MAX);
  std::vector<uint8_t> already(n, 0);
  std::vector<float*> cent(K);
  std::vector<float> owned;
  if (!alias) owned.resize(size_t(K) * len);
  std::vector<size_t> rows(K);
  rows[0] = first;
  already[first] = 1;
  cent[0] = X + first * stride + offset;
  for (int i = 1; i < K; ++i) {
    float furthest = 0.0f;
    size_t fid = 0;
    for (size_t j = 0; j < n; ++j) {
      if (already[j]) continue;
      const float* sv = X + j * stride + offset;
      float d = sq_l2_avx(sv, cent[i - 1], len);
      if (d < cdist[j]) cdist[j] = d;
      if (cdist[j] > furthest) { furthest = cdist[j]; fid = j; }
    }
    // NOTE: the reference never records furthestId in alreadyCentroid (kmeans.go:67-83
    // only inserts randId), so a row can be chosen again only if its min-dist stays the
    // max, which cannot happen once it is a centre (dist 0) unless all are 0.
    rows[i] = fid;
    cent[i] = X + fid * stride + offset;
  }
  if (init_rows_out) for (int i = 0; i < K; ++i) init_rows_out[i] = int64_t(rows[i]);
  if (!alias) {
    for (int i = 0; i < K; ++i) {
      std::memcpy(&owned[size_t(i) * len], cent[i], sizeof(float) * len);
      cent[i] = &owned[size_t(i) * len];
    }
  }
  std::memset(labels, 0, n);
  std::vector<float> sums(size_t(K) * len, 0.0f);
  std::vector<int> counts(K, 0);
  int iters = 0;
  for (int iter = 0; iter < maxIter; ++iter) {
    ++iters;
    size_t changes = 0;
    for (size_t i = 0; i < n; ++i) {
      const float* sv = X + i * stride + offset;
      float best = sq_l2_avx(sv, cent[0], len);
      uint8_t bid = 0;
      for (int j = 1; j < K; ++j) {
        float d = sq_l2_avx(sv, cent[j], len);
        if (d < best) { best = d; bid = uint8_t(j); }
      }
      if (labels[i] != bid) { ++changes; labels[i] = bid; }
    }
    if (changes == 0) break;
    for (int i = 0; i < K; ++i) counts[i] = 0;
    for (size_t i = 0; i < n; ++i) {
      int lb = labels[i];
      if (counts[lb] == 0) for (int j = 0; j < len; ++j) sums[size_t(lb) * len + j] = 0.0f;
      counts[lb]++;
      const float* sv = X + i * stride + offset;
      for (int j = 0; j < len; ++j) sums[size_t(lb) * len + j] += sv[j];
    }
    for (int i = 0; i < K; ++i) {
      if (counts[i] == 0) continue;
      for (int j = 0; j < len; ++j) cent[i][j] = sums[size_t(i) * len + j] / float(counts[i]);
    }
  }
  for (int i = 0; i < K; ++i) std::memcpy(centroids_out + size_t(i) * len, cent[i], sizeof(float) * len);
  return iters;
}

// ---------------------------------------------------------------------------
// Index state
// ---------------------------------------------------------------------------

enum Quant : int { Q_NONE = 0, Q_BINARY = 1, Q_PRODUCT = 2 };

struct Spin {
  std::atomic_flag f = ATOMIC_FLAG_INIT;
  void lock() { while (f.test_and_set(std::memory_order_acquire)) { _mm_pause(); } }
  void unlock() { f.clear(std::memory_order_release); }
};

struct Index {
  int dim = 0, metric = 0, L = 75, R = 64;
  float alpha = 1.2f;
  int quant = Q_NONE;
  // binary quantiser (shard/vectorstore/binary.go:25-64)
  bool bq_fitted = false;
  std::vector<float> bq_thr;
  int bq_metric = M_HAMMING, bq_trigger = 0, words = 0;
  // product quantiser (shard/vectorstore/product.go:28-98)
  int pqM = 0, pqK = 0, pqSub = 0, pq_trigger = 0, pq_metric = M_EUCLIDEAN;
  std::vector<float> flatCentroids, centroidDists;
  bool pq_fitted() const { return !flatCentroids.empty(); }
  // storage, dense by node id (0 invalid, 1 = start node, users from 2:
  // vamana.go:28,150-157; idcounter.go:52-54)
  size_t cap = 0;
  bool codes_only = false;  // hydrated from n<id>q payloads alone: raw vectors are not loaded (binary.go:275-296, product.go:349-371)
  std::vector<float> vec;
  std::vector<uint64_t> bits;
  std::vector<uint8_t> codes;
  std::vector<uint8_t> exists;
  std::vector<uint32_t> adj;
  std::vector<uint16_t> deg;
  // edges of the start node beyond R: removeInboundEdges re-attaches orphans with
  // AddNeighbourIfNotExists, which has no degree bound (prune.go:137-151, node.go:73-80)
  std::vector<uint32_t> start_extra;
  uint32_t maxNodeId = 0;
  size_t count = 0;
  std::unique_ptr<Spin[]> locks;

  const float* V(uint32_t id) const { return &vec[size_t(id) * dim]; }
  float* V(uint32_t id) { return &vec[size_t(id) * dim]; }
  const uint64_t* B(uint32_t id) const { return &bits[size_t(id) * words]; }
  const uint8_t* C(uint32_t id) const { return &codes[size_t(id) * pqM]; }
  uint32_t* A(uint32_t id) { return &adj[size_t(id) * R]; }
  const uint32_t* A(uint32_t id) const { return &adj[size_t(id) * R]; }

  void reserve(size_t n) {
    if (n <= cap) return;
    size_t nc = std::max(n, cap * 2);
    if (!codes_only) vec.resize(nc * dim);
    if (quant == Q_BINARY) bits.resize(nc * words);
    if (quant == Q_PRODUCT) codes.resize(nc * pqM);
    exists.resize(nc, 0);
    adj.resize(nc * R);
    deg.resize(nc, 0);
    std::unique_ptr<Spin[]> nl(new Spin[nc]);
    locks.swap(nl);
    cap = nc;
  }

  // productQuantizer.encode (product.go:136-159): argmin with the index metric,
  // strict '<' from MaxFloat32 => lowest index wins ties.
  void pq_encode(const float* v, uint8_t* out) const {
    for (int i = 0; i < pqM; ++i) {
      const float* sv = v + i * pqSub;
      float best = FLT_MAX;
      int bid = 0;
      for (int j = 0; j < pqK; ++j) {
        const float* c = &flatCentroids[(size_t(i) * pqK + j) * pqSub];
        float d = float_dist(pq_metric, sv, c, pqSub);
        if (d < best) { best = d; bid = j; }
      }
      out[i] = uint8_t(bid);
    }
  }

  // VectorStore.Set for all three stores (plain.go:58-66, binary.go:131-139,
  // product.go:161-169): keep the raw vector, encode if the quantiser is fitted.
  void set(uint32_t id, const float* v) {
    reserve(size_t(id) + 1);
    std::memcpy(V(id), v, sizeof(float) * dim);
    if (!exists[id]) { exists[id] = 1; ++count; }
    if (quant == Q_BINARY && bq_fitted) bq_encode(v, bq_thr.data(), dim, &bits[size_t(id) * words]);
    if (quant == Q_PRODUCT && pq_fitted()) pq_encode(v, &codes[size_t(id) * pqM]);
  }
};

// DistanceFromFloat closures (plain.go:76-85, binary.go:187-211, product.go:238-277).
struct QueryDist {
  const Index* ix;
  const float* q;
  int mode;  // 0 float, 1 bits, 2 adc
  std::vector<uint64_t> qbits;
  std::vector<float> table;
  QueryDist(const Index* ix_, const float* q_) : ix(ix_), q(q_), mode(0) {
    if (ix->quant == Q_BINARY && ix->bq_fitted) {
      mode = 1;
      qbits.resize(ix->words);
      bq_encode(q, ix->bq_thr.data(), ix->dim, qbits.data());
    } else if (ix->quant == Q_PRODUCT && ix->pq_fitted()) {
      mode = 2;
      table.resize(size_t(ix->pqM) * ix->pqK);
      for (int i = 0; i < ix->pqM; ++i)
        for (int j = 0; j < ix->pqK; ++j)
          table[size_t(i) * ix->pqK + j] = float_dist(
              ix->pq_metric, q + i * ix->pqSub, &ix->flatCentroids[(size_t(i) * ix->pqK + j) * ix->pqSub], ix->pqSub);
    }
  }
  float operator()(uint32_t id) const {
    switch (mode) {
      case 1: return bit_dist(ix->bq_metric, qbits.data(), ix->B(id), ix->words);
      case 2: {
        float d = 0.0f;  // sequential f32 sum over sub-vectors (product.go:271-275)
        const uint8_t* c = ix->C(id);
        for (int i = 0; i < ix->pqM; ++i) d += table[size_t(i) * ix->pqK + c[i]];
        return d;
      }
      default: {
        int m = ix->quant == Q_PRODUCT ? ix->pq_metric : ix->metric;
        return float_dist(m, q, ix->V(id), ix->dim);
      }
    }
  }
};

// DistanceFromPoint closures (plain.go:87-97, binary.go:213-234, product.go:279-305).
struct PointDist {
  const Index* ix;
  uint32_t x;
  int mode;
  PointDist(const Index* ix_, uint32_t x_) : ix(ix_), x(x_), mode(0) {
    if (ix->quant == Q_BINARY && ix->bq_fitted) mode = 1;
    else if (ix->quant == Q_PRODUCT && ix->pq_fitted()) mode = 2;
  }
  float operator()(uint32_t y) const {
    switch (mode) {
      case 1: return bit_dist(ix->bq_metric, ix->B(x), ix->B(y), ix->words);
      case 2: {
        float d = 0.0f;
        const uint8_t *cx = ix->C(x), *cy = ix->C(y);
        size_t KK = size_t(ix->pqK) * ix->pqK;
        for (int i = 0; i < ix->pqM; ++i) d += ix->centroidDists[i * KK + size_t(cx[i]) * ix->pqK + cy[i]];
        return d;
      }
      default: {
        int m = ix->quant == Q_PRODUCT ? ix->pq_metric : ix->metric;
        return float_dist(m, ix->V(x), ix->V(y), ix->dim);
      }
    }
  }
};

// ---------------------------------------------------------------------------
// DistSet (shard/index/vamana/distset.go:118-238)
// ---------------------------------------------------------------------------

struct Elem {
  uint32_t id;
  float dist;
  bool visited;
  bool pruneRemoved;
};

// Exact visited set; stands in for both VisitedBitSet and VisitedMap
// (distset.go:62-116) — same observable behaviour (CheckAndVisit).
struct Visited {
  std::vector<uint32_t> stamp;
  uint32_t epoch = 0;
  void begin(size_t n) {
    if (stamp.size() < n) stamp.assign(n, 0), epoch = 0;
    if (++epoch == 0) { std::fill(stamp.begin(), stamp.end(), 0); epoch = 1; }
  }
  bool check_and_visit(uint32_t id) {
    if (id >= stamp.size()) stamp.resize(size_t(id) * 2 + 1, 0);
    if (stamp[id] == epoch) return true;
    stamp[id] = epoch;
    return false;
  }
};

template <class DistFn>
struct DistSet {
  std::vector<Elem> items;
  size_t capacity;
  Visited* set;
  const DistFn* fn;
  size_t sortedUntil = 0;
  uint64_t* ndist;
  DistSet(size_t cap, Visited* v, const DistFn* f, uint64_t* nd) : capacity(cap), set(v), fn(f), ndist(nd) {
    items.reserve(cap);
  }
  // distset.go:166-200
  void add_with_limit(const uint32_t* ids, size_t n) {
    for (size_t t = 0; t < n; ++t) {
      uint32_t p = ids[t];
      if (set->check_and_visit(p)) continue;
      float d = (*fn)(p);
      if (ndist) ++*ndist;
      if (items.size() == capacity && d > items[capacity - 1].dist) continue;
      Elem e{p, d, false, false};
      if (items.size() < capacity) { items.push_back(e); ++sortedUntil; }
      else items[items.size() - 1] = e;
      for (size_t i = items.size() - 1; i > 0 && items[i].dist < items[i - 1].dist; --i)
        std::swap(items[i], items[i - 1]);
    }
  }
  // distset.go:203-212
  void add(const uint32_t* ids, size_t n) {
    for (size_t t = 0; t < n; ++t) {
      uint32_t p = ids[t];
      if (set->check_and_visit(p)) continue;
      float d = (*fn)(p);
      if (ndist) ++*ndist;
      items.push_back(Elem{p, d, false, false});
    }
  }
  // distset.go:219-221
  void add_already_unique(const Elem& e) { items.push_back(e); }
  // distset.go:223-238
  void sort() {
    for (size_t i = sortedUntil; i < items.size(); ++i)
      for (size_t j = i; j > 0 && items[j].dist < items[j - 1].dist; --j) std::swap(items[j], items[j - 1]);
    sortedUntil = items.size();
  }
};

struct TableDist {  // distset_test.go:18-23 helper: distance looked up by id
  const float* d;
  float operator()(uint32_t id) const { return d[id]; }
};

// ---------------------------------------------------------------------------
// greedySearch (shard/index/vamana/search.go:9-102)
// ---------------------------------------------------------------------------

struct SearchScratch {
  Visited vis, vis2;
  std::vector<uint32_t> nb;
};

struct SearchOut {
  std::vector<Elem> result;    // resultSet items (searchSet if no filter)
  std::vector<Elem> expanded;  // visitedSet in expansion order (before Sort)
  std::vector<Elem> visited;   // visitedSet after Sort (search.go:100)
  uint64_t hops = 0, ndist = 0;
};

// filter: sorted ascending ids (roaring iterator order, search.go:40-44) or null.
// locked: copy adjacency under the node's lock (search.go:89-91).
int greedy_search(Index* ix, const float* query, int k, int L, const uint32_t* filter, size_t nfilter,
                  SearchScratch& sc, SearchOut& out, bool locked) {
  out.result.clear(); out.expanded.clear(); out.visited.clear(); out.hops = 0; out.ndist = 0;
  QueryDist fn(ix, query);
  sc.vis.begin(ix->cap);
  DistSet<QueryDist> searchSet(L, &sc.vis, &fn, &out.ndist);
  if (L < k) return 1;  // search.go:23-25
  std::unique_ptr<DistSet<QueryDist>> filt;
  DistSet<QueryDist>* resultSet = &searchSet;
  if (filter) {
    sc.vis2.begin(ix->cap);
    filt.reset(new DistSet<QueryDist>(k, &sc.vis2, &fn, nullptr));
    resultSet = filt.get();
    size_t take = std::min(nfilter, size_t(L));
    for (size_t i = 0; i < take; ++i)
      if (filter[i] >= ix->cap || !ix->exists[filter[i]]) return 2;  // GetMany error (search.go:45-48)
    searchSet.add(filter, take);
    resultSet->add_with_limit(filter, take);
  }
  uint32_t start = 1;
  if (ix->cap <= 1 || !ix->exists[1]) return 3;
  searchSet.add_with_limit(&start, 1);
  sc.nb.resize(size_t(ix->R) + ix->start_extra.size());
  for (size_t i = 0; i < std::min(searchSet.items.size(), size_t(L));) {
    Elem e = searchSet.items[i];
    if (e.visited) { ++i; continue; }
    out.expanded.push_back(e);
    searchSet.items[i].visited = true;
    ++out.hops;
    uint32_t id = e.id;
    int dg;
    if (locked) {
      ix->locks[id].lock();
      dg = ix->deg[id];
      std::memcpy(sc.nb.data(), ix->A(id), sizeof(uint32_t) * dg);
      ix->locks[id].unlock();
    } else {
      dg = ix->deg[id];
      std::memcpy(sc.nb.data(), ix->A(id), sizeof(uint32_t) * dg);
    }
    if (id == 1 && !ix->start_extra.empty()) {
      std::memcpy(sc.nb.data() + dg, ix->start_extra.data(), sizeof(uint32_t) * ix->start_extra.size());
      dg += int(ix->start_extra.size());
    }
    searchSet.add_with_limit(sc.nb.data(), dg);
    if (filter && std::binary_search(filter, filter + nfilter, id)) resultSet->add_with_limit(&id, 1);
    i = 0;
  }
  out.result = resultSet->items;
  out.visited = out.expanded;
  // visitedSet.Sort() with sortedUntil == 0: full stable insertion sort
  for (size_t i = 0; i < out.visited.size(); ++i)
    for (size_t j = i; j > 0 && out.visited[j].dist < out.visited[j - 1].dist; --j)
      std::swap(out.visited[j], out.visited[j - 1]);
  return 0;
}

// robustPrune (shard/index/vamana/search.go:106-138). cand is modified (pruneRemoved).
// Writes the new edge list of `node` into edges_out; returns the degree.
int robust_prune(const Index* ix, uint32_t node, std::vector<Elem>& cand, uint32_t* edges_out, uint64_t* npair) {
  int cnt = 0;
  for (size_t i = 0; i < cand.size(); ++i) {
    Elem& c = cand[i];
    if (c.pruneRemoved || c.id == node) continue;
    edges_out[cnt++] = c.id;
    if (cnt >= ix->R) break;
    PointDist fn(ix, c.id);
    for (size_t j = i + 1; j < cand.size(); ++j) {
      Elem& nx = cand[j];
      if (nx.pruneRemoved) continue;
      if (npair) ++*npair;
      if (ix->alpha * fn(nx.id) < nx.dist) nx.pruneRemoved = true;
    }
  }
  return cnt;
}

// insertSinglePoint, first half (insert.go:16-36): greedySearch from the start node and
// robustPrune of the visited set become the new point's edges.
int insert_link(Index* ix, uint32_t id, const float* v, SearchScratch& sc, SearchOut& so, bool locked) {
  // vecStore.Set happened already (capacity must not move under concurrent workers)
  int rc = greedy_search(ix, v, 1, ix->L, nullptr, 0, sc, so, locked);
  if (rc) return rc;
  std::vector<uint32_t> edgesA(ix->R);
  int dA = robust_prune(ix, id, so.visited, edgesA.data(), nullptr);
  if (locked) ix->locks[id].lock();
  std::memcpy(ix->A(id), edgesA.data(), sizeof(uint32_t) * dA);
  ix->deg[id] = uint16_t(dA);
  if (locked) ix->locks[id].unlock();
  return 0;
}

// insertSinglePoint, second half (insert.go:37-66): the back-edge b -> id, pruning b when full.
void insert_back_edge(Index* ix, uint32_t b, uint32_t id, std::vector<Elem>& cand, std::vector<uint32_t>& eb) {
  int dB = ix->deg[b];
  if (dB + 1 > ix->R) {
    PointDist fn(ix, b);
    cand.clear();
    // candidateSet.Add(nodeB.neighbours...), Add(vecA) with a VisitedMap dedupe (insert.go:48-57)
    uint32_t* nb = ix->A(b);
    for (int j = 0; j <= dB; ++j) {
      uint32_t p = j < dB ? nb[j] : id;
      bool dup = false;
      for (const Elem& e : cand) if (e.id == p) { dup = true; break; }
      if (dup) continue;
      cand.push_back(Elem{p, fn(p), false, false});
    }
    for (size_t i = 0; i < cand.size(); ++i)  // candidateSet.Sort()
      for (size_t j = i; j > 0 && cand[j].dist < cand[j - 1].dist; --j) std::swap(cand[j], cand[j - 1]);
    int nd = robust_prune(ix, b, cand, eb.data(), nullptr);
    std::memcpy(nb, eb.data(), sizeof(uint32_t) * nd);
    ix->deg[b] = uint16_t(nd);
  } else {
    ix->A(b)[dB] = id;  // nodeB.AddNeighbour(vecA)
    ix->deg[b] = uint16_t(dB + 1);
  }
}

// insertSinglePoint (shard/index/vamana/insert.go:16-68)
int insert_single(Index* ix, uint32_t id, const float* v, SearchScratch& sc, SearchOut& so, bool locked) {
  int rc = insert_link(ix, id, v, sc, so, locked);
  if (rc) return rc;
  if (locked) ix->locks[id].lock();
  std::vector<uint32_t> edgesA(ix->A(id), ix->A(id) + ix->deg[id]);
  if (locked) ix->locks[id].unlock();
  std::vector<Elem> cand;
  std::vector<uint32_t> eb(ix->R);
  for (uint32_t b : edgesA) {
    if (locked) ix->locks[b].lock();
    insert_back_edge(ix, b, id, cand, eb);
    if (locked) ix->locks[b].unlock();
  }
  return 0;
}

// Edge list of a node including the start node's overflow edges.
void node_edges(const Index* ix, uint32_t id, std::vector<uint32_t>& out) {
  out.assign(ix->A(id), ix->A(id) + ix->deg[id]);
  if (id == 1) out.insert(out.end(), ix->start_extra.begin(), ix->start_extra.end());
}

void set_node_edges(Index* ix, uint32_t id, const uint32_t* e, int n) {
  std::memcpy(ix->A(id), e, sizeof(uint32_t) * n);
  ix->deg[id] = uint16_t(n);
  if (id == 1) ix->start_extra.clear();
}

// EdgeScan (shard/index/vamana/node.go:142-199). del: per-row flags. Iteration order of the
// reference is Go map order; here ascending node id (SURVEY.md §8c). toPrune = valid nodes
// with an edge into the delete set; toSave = valid nodes (except the start node) that no
// valid node points at — counted before any pruning, edges into the delete set included.
void edge_scan(const Index* ix, const std::vector<uint8_t>& del, std::vector<uint32_t>& toPrune,
               std::vector<uint32_t>& toSave) {
  toPrune.clear();
  toSave.clear();
  std::vector<uint8_t> hasInbound(ix->cap, 0);
  std::vector<uint32_t> e;
  for (uint32_t id = 0; id < ix->cap; ++id) {
    if (!ix->exists[id] || del[id]) continue;
    node_edges(ix, id, e);
    bool added = false;
    for (uint32_t t : e) {
      hasInbound[t] = 1;
      if (!added && del[t]) { toPrune.push_back(id); added = true; }
    }
  }
  for (uint32_t id = 0; id < ix->cap; ++id)
    if (ix->exists[id] && !del[id] && !hasInbound[id] && id != 1) toSave.push_back(id);
}

// pruneDeleteNeighbour (shard/index/vamana/prune.go:12-84)
int prune_delete_neighbour(Index* ix, uint32_t a, const std::vector<uint8_t>& del) {
  std::vector<uint32_t> ea, eb, validIds, toExpand;
  node_edges(ix, a, ea);
  for (uint32_t b : ea) (del[b] ? toExpand : validIds).push_back(b);
  if (toExpand.empty()) return 20;  // prune.go:37-40
  for (uint32_t b : toExpand) {
    node_edges(ix, b, eb);
    for (uint32_t c : eb)
      if (!del[c]) validIds.push_back(c);
  }
  // candidateSet.Add(vecs...) dedupes with a VisitedMap, then Sort() (prune.go:59-66)
  PointDist fn(ix, a);
  std::vector<Elem> cand;
  {
    std::vector<uint32_t> seen(validIds);
    std::sort(seen.begin(), seen.end());
    std::vector<uint8_t> used(seen.size(), 0);
    for (uint32_t p : validIds) {
      size_t k = std::lower_bound(seen.begin(), seen.end(), p) - seen.begin();
      if (used[k]) continue;
      used[k] = 1;
      cand.push_back(Elem{p, fn(p), false, false});
    }
  }
  for (size_t i = 0; i < cand.size(); ++i)
    for (size_t j = i; j > 0 && cand[j].dist < cand[j - 1].dist; --j) std::swap(cand[j], cand[j - 1]);
  std::vector<uint32_t> out(std::max<size_t>(cand.size(), size_t(ix->R)));
  int n = 0;
  if (int(cand.size()) > ix->R) {
    n = robust_prune(ix, a, cand, out.data(), nullptr);  // prune.go:68-70
  } else {
    for (const Elem& c : cand)
      if (c.id != a) out[n++] = c.id;  // prune.go:72-81
  }
  set_node_edges(ix, a, out.data(), n);
  return 0;
}

// removeInboundEdges (shard/index/vamana/prune.go:88-154)
int remove_inbound_edges(Index* ix, const std::vector<uint8_t>& del, std::vector<uint32_t>* toPruneOut,
                         std::vector<uint32_t>* toSaveOut) {
  std::vector<uint32_t> toPrune, toSave;
  edge_scan(ix, del, toPrune, toSave);
  for (uint32_t a : toPrune) {
    int rc = prune_delete_neighbour(ix, a, del);
    if (rc) return rc;
  }
  if (!toSave.empty()) {
    if (ix->cap <= 1 || !ix->exists[1]) return 3;
    for (uint32_t p : toSave) {
      if (p == 1) continue;
      // startNode.AddNeighbourIfNotExists(point) (node.go:73-80): no degree bound
      bool present = false;
      for (int t = 0; t < ix->deg[1] && !present; ++t) present = ix->A(1)[t] == p;
      for (uint32_t x : ix->start_extra) present = present || x == p;
      if (present) continue;
      if (ix->deg[1] < ix->R) { ix->A(1)[ix->deg[1]] = p; ix->deg[1]++; }
      else ix->start_extra.push_back(p);
    }
  }
  if (toPruneOut) *toPruneOut = toPrune;
  if (toSaveOut) *toSaveOut = toSave;
  return 0;
}

template <class F>
void parallel_for(size_t n, int threads, F f) {
  if (threads <= 1 || n <= 1) { for (size_t i = 0; i < n; ++i) f(i, 0); return; }
  std::atomic<size_t> next(0);
  std::vector<std::thread> th;
  for (int t = 0; t < threads; ++t)
    th.emplace_back([&, t] {
      for (;;) {
        size_t i = next.fetch_add(1);
        if (i >= n) break;
        f(i, t);
      }
    });
  for (auto& x : th) x.join();
}

// Reusable barrier of a fixed set of threads (generation counter).
struct Barrier {
  explicit Barrier(int n) : n(n) {}
  void wait() {
    int gen = generation.load(std::memory_order_acquire);
    if (arrived.fetch_add(1, std::memory_order_acq_rel) + 1 == n) {
      arrived.store(0, std::memory_order_relaxed);
      generation.fetch_add(1, std::memory_order_acq_rel);
    } else {
      while (generation.load(std::memory_order_acquire) == gen) std::this_thread::yield();
    }
  }
  const int n;
  std::atomic<int> arrived{0};
  std::atomic<int> generation{0};
};

// Parallel insert whose graph depends on the input alone, not on the thread count or timing.
// The points go in rounds of a fixed length (1 while the call has inserted fewer than 16
// points, growing as 1/16 of them, at most max_round). In a round every point searches the
// graph as it stood at the start of the round and takes its own edges (insert_link, no other
// writes happen then); then the back-edges are applied, one target per task, in input order.
// A target's row depends only on its own row and the points added to it, so this is the
// sequential schedule's result for that round. max_round 1 is the 1-worker schedule.
int insert_rounds(Index* ix, const uint32_t* ids, const float* vecs, size_t n, int T, size_t max_round) {
  std::vector<SearchScratch> sc(T);
  std::vector<SearchOut> so(T);
  std::vector<std::vector<Elem>> cand(T);
  std::vector<std::vector<uint32_t>> eb(T, std::vector<uint32_t>(ix->R));
  std::vector<std::pair<uint32_t, uint32_t>> pairs;  // (target, input index of the new point)
  std::vector<size_t> group;                         // start of each target's run in pairs
  std::atomic<size_t> next_link(0), next_target(0);
  std::atomic<int> err(0);
  Barrier bar(T);
  auto worker = [&](int t) {
    for (size_t s = 0; s < n;) {
      size_t m = std::min(n - s, std::min(std::max<size_t>(max_round, 1), std::max<size_t>(1, s / 16)));
      for (size_t i; (i = next_link.fetch_add(1)) < m;) {
        int rc = insert_link(ix, ids[s + i], vecs + (s + i) * ix->dim, sc[t], so[t], false);
        if (rc) err.store(rc);
      }
      bar.wait();
      if (t == 0) {
        pairs.clear();
        for (size_t i = s; i < s + m; ++i)
          for (int j = 0; j < ix->deg[ids[i]]; ++j) pairs.emplace_back(ix->A(ids[i])[j], uint32_t(i));
        std::stable_sort(pairs.begin(), pairs.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
        group.clear();
        for (size_t k = 0; k < pairs.size(); ++k)
          if (k == 0 || pairs[k].first != pairs[k - 1].first) group.push_back(k);
        group.push_back(pairs.size());
        next_link.store(0);
        next_target.store(0);
      }
      bar.wait();
      for (size_t g; (g = next_target.fetch_add(1)) + 1 < group.size();)
        for (size_t k = group[g]; k < group[g + 1]; ++k)
          insert_back_edge(ix, pairs[k].first, ids[pairs[k].second], cand[t], eb[t]);
      bar.wait();
      s += m;
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < T; ++t) th.emplace_back(worker, t);
  worker(0);
  for (auto& x : th) x.join();
  return err.load();
}

}  // namespace

// ---------------------------------------------------------------------------
// C surface for ctypes (tests) and bench.py's cpu_baseline leg
// ---------------------------------------------------------------------------
extern "C" {

float orc_sq_l2_avx(const float* x, const float* y, size_t n) { return sq_l2_avx(x, y, n); }
float orc_dot_avx(const float* x, const float* y, size_t n) { return dot_avx(x, y, n); }
float orc_sq_l2_pure(const float* x, const float* y, size_t n) { return sq_l2_pure(x, y, n); }
float orc_dot_pure(const float* x, const float* y, size_t n) { return dot_pure(x, y, n); }
float orc_sq_l2_model(const float* x, const float* y, size_t n) { return ordered_model(x, y, n, true); }
float orc_dot_model(const float* x, const float* y, size_t n) { return ordered_model(x, y, n, false); }
float orc_float_dist(int metric, const float* x, const float* y, size_t n) { return float_dist(metric, x, y, n); }
float orc_bit_dist(int metric, const uint64_t* x, const uint64_t* y, size_t words) { return bit_dist(metric, x, y, words); }
void orc_bq_encode(const float* v, const float* thr, int dim, uint64_t* out) { bq_encode(v, thr, dim, out); }

// binaryQuantizer.Fit threshold (binary.go:145-170): running f32 sums in iteration
// order (oracle: ascending row order), then / float32(count).
void orc_bq_fit_threshold(const float* X, size_t n, int dim, float* thr_out) {
  std::vector<float> sum(dim, 0.0f);
  for (size_t r = 0; r < n; ++r)
    for (int i = 0; i < dim; ++i) sum[i] += X[r * dim + i];
  for (int i = 0; i < dim; ++i) thr_out[i] = sum[i] / float(n);
}

// distset_test.go harness: capacity-bounded AddWithLimit / Add / Sort over ids whose
// distance is dists[id]. op: 0 = AddWithLimit, 1 = Add, 2 = Sort (ids ignored).
struct OrcDistSet {
  Visited v;
  TableDist fn;
  std::vector<float> d;
  std::unique_ptr<DistSet<TableDist>> ds;
};
void* orc_distset_new(int capacity, const float* dists, int ndists) {
  auto* h = new OrcDistSet;
  h->d.assign(dists, dists + ndists);
  h->fn.d = h->d.data();
  h->v.begin(ndists + 1);
  h->ds.reset(new DistSet<TableDist>(capacity, &h->v, &h->fn, nullptr));
  return h;
}
void orc_distset_op(void* hp, int op, const uint32_t* ids, int n) {
  auto* h = static_cast<OrcDistSet*>(hp);
  if (op == 0) h->ds->add_with_limit(ids, n);
  else if (op == 1) h->ds->add(ids, n);
  else h->ds->sort();
}
int orc_distset_items(void* hp, uint32_t* ids_out, float* dists_out, int maxn) {
  auto* h = static_cast<OrcDistSet*>(hp);
  int n = int(std::min(h->ds->items.size(), size_t(maxn)));
  for (int i = 0; i < n; ++i) { ids_out[i] = h->ds->items[i].id; dists_out[i] = h->ds->items[i].dist; }
  return int(h->ds->items.size());
}
void orc_distset_free(void* hp) { delete static_cast<OrcDistSet*>(hp); }

int orc_kmeans_fit(float* X, size_t n, size_t stride, int offset, int len, int K, int maxIter, size_t first,
                   int alias, float* centroids_out, uint8_t* labels, int64_t* init_rows_out) {
  return kmeans_fit(X, n, stride, offset, len, K, maxIter, first, alias != 0, centroids_out, labels, init_rows_out);
}

// --- index -----------------------------------------------------------------

// quant: 0 none, 1 binary, 2 product. For metric hamming/jaccard the binary quantiser
// is forced on with threshold 0.5 (vectorstore.go:56-66). bq_threshold: NaN = unset
// (fit later from the mean). PQ: cosine silently becomes euclidean (product.go:52-61).
void* orc_index_new(int dim, int metric, int L, int R, float alpha, int quant, float bq_threshold, int bq_metric,
                    int bq_trigger, int pqM, int pqK, int pq_trigger) {
  auto* ix = new Index;
  ix->dim = dim; ix->metric = metric; ix->L = L; ix->R = R; ix->alpha = alpha;
  ix->quant = quant;
  ix->words = (dim + 63) / 64;
  if (metric == M_HAMMING || metric == M_JACCARD) {
    ix->quant = Q_BINARY;
    ix->bq_metric = metric;
    ix->bq_fitted = true;
    ix->bq_thr.assign(dim, 0.5f);
  } else if (quant == Q_BINARY) {
    ix->bq_metric = bq_metric;
    ix->bq_trigger = bq_trigger;
    if (!std::isnan(bq_threshold)) { ix->bq_fitted = true; ix->bq_thr.assign(dim, bq_threshold); }
  } else if (quant == Q_PRODUCT) {
    if (pqM <= 0 || dim % pqM != 0 || pqK > 256 || pqK < 1) { delete ix; return nullptr; }  // product.go:44-46,63-65
    if (metric != M_EUCLIDEAN && metric != M_COSINE && metric != M_DOT) { delete ix; return nullptr; }
    ix->pqM = pqM; ix->pqK = pqK; ix->pqSub = dim / pqM; ix->pq_trigger = pq_trigger;
    ix->pq_metric = metric == M_COSINE ? M_EUCLIDEAN : metric;
  }
  ix->reserve(1024);
  return ix;
}
void orc_index_free(void* h) { delete static_cast<Index*>(h); }

// setupStartNode (vamana.go:93-120): the caller supplies the (random unit) vector.
void orc_index_set_start(void* h, const float* v) {
  auto* ix = static_cast<Index*>(h);
  ix->set(1, v);
  ix->deg[1] = 0;
}

// vecStore.Set only (no graph work) — used to stage vectors, e.g. for flat search.
void orc_index_set_vectors(void* h, const uint32_t* ids, const float* vecs, size_t n) {
  auto* ix = static_cast<Index*>(h);
  uint32_t mx = 0;
  for (size_t i = 0; i < n; ++i) mx = std::max(mx, ids[i]);
  ix->reserve(size_t(mx) + 1);
  for (size_t i = 0; i < n; ++i) ix->set(ids[i], vecs + i * ix->dim);
}

// insertUpdateDelete, insert branch only (vamana.go:136-201): ids 0 and 1 rejected
// (vamana.go:150-157); threads<=1 = sequential in the given order (the 1-worker
// schedule); threads>1 = reference-style concurrent workers with per-node locks.
int orc_index_insert(void* h, const uint32_t* ids, const float* vecs, size_t n, int threads) {
  auto* ix = static_cast<Index*>(h);
  uint32_t mx = 0;
  for (size_t i = 0; i < n; ++i) {
    if (ids[i] == 0 || ids[i] == 1) return 10;
    mx = std::max(mx, ids[i]);
  }
  ix->reserve(size_t(mx) + 1);
  if (mx > ix->maxNodeId) ix->maxNodeId = mx;
  int T = std::max(1, threads);
  std::vector<SearchScratch> sc(T);
  std::vector<SearchOut> so(T);
  std::atomic<int> err(0);
  // vecStore.Set (insert.go:17) for the whole batch up front: a point is unreachable
  // until an edge points at it, so staging its vector early is unobservable.
  for (size_t i = 0; i < n; ++i) {
    ix->set(ids[i], vecs + i * ix->dim);
    ix->deg[ids[i]] = 0;
  }
  if (T == 1) {
    for (size_t i = 0; i < n; ++i) {
      int rc = insert_single(ix, ids[i], vecs + i * ix->dim, sc[0], so[0], false);
      if (rc) return rc;
    }
    return 0;
  }
  parallel_for(n, T, [&](size_t i, int t) {
    int rc = insert_single(ix, ids[i], vecs + i * ix->dim, sc[t], so[t], true);
    if (rc) err.store(rc);
  });
  return err.load();
}

// The same insert on the deterministic round schedule (insert_rounds): the graph is a function
// of the input and max_round only, whatever the thread count.
int orc_index_insert_rounds(void* h, const uint32_t* ids, const float* vecs, size_t n, int threads, size_t max_round) {
  auto* ix = static_cast<Index*>(h);
  uint32_t mx = 0;
  for (size_t i = 0; i < n; ++i) {
    if (ids[i] == 0 || ids[i] == 1) return 10;
    mx = std::max(mx, ids[i]);
  }
  ix->reserve(size_t(mx) + 1);
  if (mx > ix->maxNodeId) ix->maxNodeId = mx;
  for (size_t i = 0; i < n; ++i) {
    ix->set(ids[i], vecs + i * ix->dim);
    ix->deg[ids[i]] = 0;
  }
  return insert_rounds(ix, ids, vecs, n, std::max(1, threads), max_round);
}

// insertUpdateDelete (vamana.go:136-263) without the trailing Fit/flush: classify each
// change against the store (has_vec[i] == 0 means a nil vector), run the inserts
// (threads as in orc_index_insert), removeInboundEdges over updated ∪ deleted ids, drop the
// deleted rows, re-insert the updated points one by one in input order (vamana.go:249-253).
int orc_index_update_delete(void* h, const uint32_t* ids, const float* vecs, const uint8_t* has_vec, size_t n,
                            int threads) {
  auto* ix = static_cast<Index*>(h);
  std::vector<uint32_t> ins_ids, upd, dele;
  std::vector<float> ins_vecs;
  std::vector<size_t> upd_src;
  for (size_t i = 0; i < n; ++i) {
    if (ids[i] == 1 || ids[i] == 0) return 10;  // vamana.go:150-157
    bool exists = ids[i] < ix->cap && ix->exists[ids[i]];
    if (!exists && !has_vec[i]) continue;
    if (!exists) {
      ins_ids.push_back(ids[i]);
      ins_vecs.insert(ins_vecs.end(), vecs + i * ix->dim, vecs + (i + 1) * ix->dim);
    } else if (has_vec[i]) {
      upd.push_back(ids[i]);
      upd_src.push_back(i);
    } else {
      dele.push_back(ids[i]);
    }
  }
  if (!ins_ids.empty()) {
    int rc = orc_index_insert(h, ins_ids.data(), ins_vecs.data(), ins_ids.size(), threads);
    if (rc) return rc;
  }
  if (!upd.empty() || !dele.empty()) {
    std::vector<uint8_t> del(ix->cap, 0);
    for (uint32_t id : upd) del[id] = 1;
    for (uint32_t id : dele) del[id] = 1;
    int rc = remove_inbound_edges(ix, del, nullptr, nullptr);
    if (rc) return rc;
  }
  for (uint32_t id : dele) {  // vecStore.Delete + nodeStore.Delete (vamana.go:231-236)
    if (!ix->exists[id]) continue;
    ix->exists[id] = 0;
    ix->count--;
    ix->deg[id] = 0;
  }
  SearchScratch sc;
  SearchOut so;
  for (size_t u = 0; u < upd.size(); ++u) {
    const float* v = vecs + upd_src[u] * ix->dim;
    ix->set(upd[u], v);
    int rc = insert_single(ix, upd[u], v, sc, so, false);
    if (rc) return rc;
  }
  return 0;
}

// EdgeScan alone (vamana_test.go:142-175). Returns counts through n_prune / n_save.
void orc_edge_scan(void* h, const uint32_t* del_ids, size_t ndel, uint32_t* prune_out, size_t* n_prune,
                   uint32_t* save_out, size_t* n_save) {
  auto* ix = static_cast<Index*>(h);
  std::vector<uint8_t> del(ix->cap, 0);
  for (size_t i = 0; i < ndel; ++i)
    if (del_ids[i] < ix->cap) del[del_ids[i]] = 1;
  std::vector<uint32_t> tp, ts;
  edge_scan(ix, del, tp, ts);
  std::copy(tp.begin(), tp.end(), prune_out);
  std::copy(ts.begin(), ts.end(), save_out);
  *n_prune = tp.size();
  *n_save = ts.size();
}

size_t orc_index_start_extra(void* h, uint32_t* out, size_t cap) {
  auto* ix = static_cast<Index*>(h);
  for (size_t i = 0; i < ix->start_extra.size() && i < cap; ++i) out[i] = ix->start_extra[i];
  return ix->start_extra.size();
}

// vecStore.Fit() (vamana.go:258): BQ mean threshold (binary.go:145-185) or PQ k-means
// (product.go:175-236). pq_first = first-centre row index among existing points in
// ascending id order; pq_alias reproduces the in-place centroid aliasing.
// Returns 1 if a fit happened, 0 if skipped, <0 on error.
int orc_index_fit(void* h, size_t pq_first, int pq_alias, int threads) {
  auto* ix = static_cast<Index*>(h);
  if (ix->quant == Q_BINARY) {
    if (ix->bq_fitted || int64_t(ix->count) < int64_t(ix->bq_trigger)) return 0;
    std::vector<float> sum(ix->dim, 0.0f);
    size_t cnt = 0;
    for (uint32_t id = 0; id < ix->cap; ++id) {
      if (!ix->exists[id]) continue;
      const float* v = ix->V(id);
      for (int i = 0; i < ix->dim; ++i) sum[i] += v[i];
      ++cnt;
    }
    for (int i = 0; i < ix->dim; ++i) sum[i] /= float(cnt);
    ix->bq_thr = sum;
    ix->bq_fitted = true;
    for (uint32_t id = 0; id < ix->cap; ++id)
      if (ix->exists[id]) bq_encode(ix->V(id), ix->bq_thr.data(), ix->dim, &ix->bits[size_t(id) * ix->words]);
    return 1;
  }
  if (ix->quant == Q_PRODUCT) {
    if (ix->pq_fitted() || int64_t(ix->count) < int64_t(ix->pq_trigger)) return 0;
    std::vector<uint32_t> rows;
    for (uint32_t id = 0; id < ix->cap; ++id) if (ix->exists[id]) rows.push_back(id);
    size_t n = rows.size();
    std::vector<float> X(n * ix->dim);
    for (size_t r = 0; r < n; ++r) std::memcpy(&X[r * ix->dim], ix->V(rows[r]), sizeof(float) * ix->dim);
    std::vector<float> fc(size_t(ix->pqM) * ix->pqK * ix->pqSub);
    std::vector<float> cd(size_t(ix->pqM) * ix->pqK * ix->pqK);
    std::vector<uint8_t> labels(size_t(ix->pqM) * n);
    parallel_for(size_t(ix->pqM), threads, [&](size_t i, int) {
      float* cent = &fc[i * ix->pqK * ix->pqSub];
      kmeans_fit(X.data(), n, ix->dim, int(i) * ix->pqSub, ix->pqSub, ix->pqK, 100, pq_first, pq_alias != 0, cent,
                 &labels[i * n], nullptr);
      for (int j = 0; j < ix->pqK; ++j)
        for (int k = 0; k < ix->pqK; ++k)
          cd[(i * ix->pqK + j) * ix->pqK + k] =
              float_dist(ix->pq_metric, cent + size_t(j) * ix->pqSub, cent + size_t(k) * ix->pqSub, ix->pqSub);
    });
    for (size_t r = 0; r < n; ++r) {
      for (int i = 0; i < ix->pqM; ++i) ix->codes[size_t(rows[r]) * ix->pqM + i] = labels[size_t(i) * n + r];
      if (pq_alias) std::memcpy(ix->V(rows[r]), &X[r * ix->dim], sizeof(float) * ix->dim);
    }
    ix->flatCentroids.swap(fc);
    ix->centroidDists.swap(cd);
    return 1;
  }
  return 0;
}

// Install externally trained PQ state / BQ threshold (e.g. from the GPU path) and re-encode.
int orc_index_set_pq(void* h, const float* flatCentroids, const float* centroidDists, int reencode) {
  auto* ix = static_cast<Index*>(h);
  if (ix->quant != Q_PRODUCT) return -1;
  ix->flatCentroids.assign(flatCentroids, flatCentroids + size_t(ix->pqM) * ix->pqK * ix->pqSub);
  ix->centroidDists.assign(centroidDists, centroidDists + size_t(ix->pqM) * ix->pqK * ix->pqK);
  if (reencode)
    for (uint32_t id = 0; id < ix->cap; ++id)
      if (ix->exists[id]) ix->pq_encode(ix->V(id), &ix->codes[size_t(id) * ix->pqM]);
  return 0;
}
int orc_index_get_pq(void* h, float* flatCentroids, float* centroidDists) {
  auto* ix = static_cast<Index*>(h);
  if (!ix->pq_fitted()) return -1;
  std::memcpy(flatCentroids, ix->flatCentroids.data(), sizeof(float) * ix->flatCentroids.size());
  std::memcpy(centroidDists, ix->centroidDists.data(), sizeof(float) * ix->centroidDists.size());
  return 0;
}
int orc_index_get_bq_threshold(void* h, float* thr) {
  auto* ix = static_cast<Index*>(h);
  if (!ix->bq_fitted) return -1;
  std::memcpy(thr, ix->bq_thr.data(), sizeof(float) * ix->dim);
  return 0;
}
int orc_index_get_codes(void* h, const uint32_t* ids, size_t n, uint8_t* out) {
  auto* ix = static_cast<Index*>(h);
  if (ix->quant == Q_PRODUCT) for (size_t i = 0; i < n; ++i) std::memcpy(out + i * ix->pqM, ix->C(ids[i]), ix->pqM);
  else if (ix->quant == Q_BINARY) for (size_t i = 0; i < n; ++i) std::memcpy(out + i * ix->words * 8, ix->B(ids[i]), ix->words * 8);
  else return -1;
  return 0;
}
// Hydrate quantised points from their codes alone, like loading the n<id>q keys of a fitted
// store (binary.go:275-296, product.go:349-371: a point with codes does not load its raw vector).
// Only valid on an empty index or one already in this mode; searches then use the codes only.
int orc_index_set_codes(void* h, const uint32_t* ids, const uint8_t* codes, size_t n) {
  auto* ix = static_cast<Index*>(h);
  const bool bq = ix->quant == Q_BINARY && ix->bq_fitted, pq = ix->quant == Q_PRODUCT && ix->pq_fitted();
  if (!bq && !pq) return -1;
  if (ix->count != 0 && !ix->codes_only) return -2;
  if (!ix->codes_only) {
    ix->codes_only = true;
    std::vector<float>().swap(ix->vec);
  }
  uint32_t mx = 0;
  for (size_t i = 0; i < n; ++i) mx = std::max(mx, ids[i]);
  ix->reserve(size_t(mx) + 1);
  for (size_t i = 0; i < n; ++i) {
    const uint32_t id = ids[i];
    if (bq) std::memcpy(&ix->bits[size_t(id) * ix->words], codes + i * size_t(ix->words) * 8, size_t(ix->words) * 8);
    else std::memcpy(&ix->codes[size_t(id) * ix->pqM], codes + i * size_t(ix->pqM), ix->pqM);
    if (!ix->exists[id]) { ix->exists[id] = 1; ix->count++; }
    if (id != 1 && id > ix->maxNodeId) ix->maxNodeId = id;
  }
  return 0;
}
int orc_index_get_vectors(void* h, const uint32_t* ids, size_t n, float* out) {
  auto* ix = static_cast<Index*>(h);
  for (size_t i = 0; i < n; ++i) std::memcpy(out + i * ix->dim, ix->V(ids[i]), sizeof(float) * ix->dim);
  return 0;
}

uint64_t orc_index_capacity(void* h) { return static_cast<Index*>(h)->cap; }
uint64_t orc_index_count(void* h) { return static_cast<Index*>(h)->count; }
uint32_t orc_index_max_node_id(void* h) { return static_cast<Index*>(h)->maxNodeId; }

// Graph export/import: rows [0, n) of adj (n x R, unused slots = 0xFFFFFFFF) and deg.
void orc_index_get_graph(void* h, size_t n, uint32_t* adj_out, uint16_t* deg_out) {
  auto* ix = static_cast<Index*>(h);
  for (size_t id = 0; id < n; ++id) {
    int d = id < ix->cap ? ix->deg[id] : 0;
    for (int j = 0; j < ix->R; ++j) adj_out[id * ix->R + j] = j < d ? ix->A(uint32_t(id))[j] : 0xFFFFFFFFu;
    deg_out[id] = uint16_t(d);
  }
}
void orc_index_set_graph(void* h, size_t n, const uint32_t* adj_in, const uint16_t* deg_in) {
  auto* ix = static_cast<Index*>(h);
  ix->reserve(n);
  for (size_t id = 0; id < n; ++id) {
    ix->deg[id] = deg_in[id];
    std::memcpy(ix->A(uint32_t(id)), adj_in + id * ix->R, sizeof(uint32_t) * deg_in[id]);
  }
  if (n && uint32_t(n - 1) > ix->maxNodeId) ix->maxNodeId = uint32_t(n - 1);
}

// IndexVamana.Search batched over queries (vamana.go:278-310 per query): greedySearch,
// drop STARTID, first k items. filter (optional, shared by all queries): ascending ids.
// out_ids/out_dists: B x k (unused = 0 / +inf); out_counts: B. Optional diagnostics:
// out_hops/out_ndist (B each), out_list_ids/out_list_dists (B x L, full searchSet incl.
// start node, unused = 0xFFFFFFFF), out_list_len (B), out_vis_ids/out_vis_dists
// (B x vis_cap, sorted visited list), out_vis_len (B).
int orc_index_search(void* h, const float* queries, size_t B, int k, int L, const uint32_t* filter, size_t nfilter,
                     uint32_t* out_ids, float* out_dists, uint32_t* out_counts, uint32_t* out_hops,
                     uint32_t* out_ndist, uint32_t* out_list_ids, float* out_list_dists, uint32_t* out_list_len,
                     uint32_t* out_vis_ids, float* out_vis_dists, uint32_t* out_vis_len, int vis_cap, int threads) {
  auto* ix = static_cast<Index*>(h);
  int T = std::max(1, threads);
  std::vector<SearchScratch> sc(T);
  std::vector<SearchOut> so(T);
  std::atomic<int> err(0);
  parallel_for(B, T, [&](size_t b, int t) {
    SearchOut& o = so[t];
    int rc = greedy_search(ix, queries + b * ix->dim, k, L, filter, nfilter, sc[t], o, false);
    if (rc) { err.store(rc); return; }
    int cnt = 0;
    for (const Elem& e : o.result) {
      if (e.id == 1) continue;
      if (cnt >= k) break;
      out_ids[b * k + cnt] = e.id;
      out_dists[b * k + cnt] = e.dist;
      ++cnt;
    }
    for (int j = cnt; j < k; ++j) { out_ids[b * k + j] = 0; out_dists[b * k + j] = INFINITY; }
    out_counts[b] = uint32_t(cnt);
    if (out_hops) out_hops[b] = uint32_t(o.hops);
    if (out_ndist) out_ndist[b] = uint32_t(o.ndist);
    if (out_list_ids) {
      size_t n = o.result.size();
      for (int j = 0; j < L; ++j) {
        out_list_ids[b * L + j] = size_t(j) < n ? o.result[j].id : 0xFFFFFFFFu;
        out_list_dists[b * L + j] = size_t(j) < n ? o.result[j].dist : INFINITY;
      }
      if (out_list_len) out_list_len[b] = uint32_t(n);
    }
    if (out_vis_ids) {
      size_t n = std::min(o.visited.size(), size_t(vis_cap));
      for (size_t j = 0; j < n; ++j) {
        out_vis_ids[b * vis_cap + j] = o.visited[j].id;
        out_vis_dists[b * vis_cap + j] = o.visited[j].dist;
      }
      out_vis_len[b] = uint32_t(o.visited.size());
    }
  });
  return err.load();
}

// robustPrune on an explicit candidate list (ids + distances, already sorted as the
// caller wishes); returns the edge count, edges in edges_out (R slots).
int orc_robust_prune(void* h, uint32_t node, const uint32_t* cand_ids, const float* cand_dists, int n,
                     uint32_t* edges_out) {
  auto* ix = static_cast<Index*>(h);
  std::vector<Elem> cand(n);
  for (int i = 0; i < n; ++i) cand[i] = Elem{cand_ids[i], cand_dists[i], false, false};
  return robust_prune(ix, node, cand, edges_out, nullptr);
}

// Point-to-point distance through the store (DistanceFromPoint).
float orc_index_point_dist(void* h, uint32_t x, uint32_t y) {
  auto* ix = static_cast<Index*>(h);
  return PointDist(ix, x)(y);
}
// Query-to-point distances through the store (DistanceFromFloat), one closure per query.
void orc_index_query_dists(void* h, const float* query, const uint32_t* ids, size_t n, float* out) {
  auto* ix = static_cast<Index*>(h);
  QueryDist fn(ix, query);
  for (size_t i = 0; i < n; ++i) out[i] = fn(ids[i]);
}
// The ADC table DistanceFromFloat builds (product.go:255-263): M x K floats.
int orc_index_adc_table(void* h, const float* query, float* out) {
  auto* ix = static_cast<Index*>(h);
  QueryDist fn(ix, query);
  if (fn.mode != 2) return -1;
  std::memcpy(out, fn.table.data(), sizeof(float) * fn.table.size());
  return 0;
}

// IndexFlat.Search (shard/index/flat/flat.go:76-132) batched over queries. Iteration
// order = ascending node id (the reference iterates a Go map: nondeterministic on ties,
// flat_test.go:179-187). Skip if full and d >= worst (flat.go:99), strict '<' bubble
// (flat.go:117). Start node (id 1) is not part of a flat index: ids >= first_id only.
int orc_flat_search(void* h, const float* queries, size_t B, int k, uint32_t first_id, const uint32_t* filter,
                    size_t nfilter, uint32_t* out_ids, float* out_dists, uint32_t* out_counts, int threads) {
  auto* ix = static_cast<Index*>(h);
  parallel_for(B, std::max(1, threads), [&](size_t b, int) {
    QueryDist fn(ix, queries + b * ix->dim);
    std::vector<Elem> res;
    res.reserve(k);
    auto visit = [&](uint32_t id) {
      float d = fn(id);
      if (int(res.size()) == k && d >= res.back().dist) return;
      Elem e{id, d, false, false};
      if (int(res.size()) < k) res.push_back(e); else res.back() = e;
      for (size_t i = res.size() - 1; i > 0 && res[i].dist < res[i - 1].dist; --i) std::swap(res[i], res[i - 1]);
    };
    if (filter) { for (size_t i = 0; i < nfilter; ++i) if (filter[i] < ix->cap && ix->exists[filter[i]]) visit(filter[i]); }
    else for (uint32_t id = first_id; id < ix->cap; ++id) if (ix->exists[id]) visit(id);
    for (int j = 0; j < k; ++j) {
      out_ids[b * k + j] = size_t(j) < res.size() ? res[j].id : 0;
      out_dists[b * k + j] = size_t(j) < res.size() ? res[j].dist : INFINITY;
    }
    out_counts[b] = uint32_t(res.size());
  });
  return 0;
}

// Cross-shard merge (cluster/actions.go:357-376): concatenate per-shard results, sort
// by HybridScore = -dist (vamana.go:303) descending, truncate. The reference's sort is
// unstable; the oracle fixes ties as (dist asc, shard asc, rank asc).
// in_*: S x B x k, counts S x B. out: B x k.
void orc_merge_topk(const uint64_t* in_ids, const float* in_dists, const uint32_t* in_counts, int S, size_t B, int k,
                    uint64_t* out_ids, float* out_dists, uint32_t* out_counts) {
  for (size_t b = 0; b < B; ++b) {
    struct It { float score; int s; int r; uint64_t id; float d; };
    std::vector<It> all;
    for (int s = 0; s < S; ++s) {
      uint32_t c = in_counts[size_t(s) * B + b];
      for (uint32_t r = 0; r < c; ++r) {
        size_t o = (size_t(s) * B + b) * k + r;
        all.push_back(It{-1.0f * in_dists[o] * 1.0f, s, int(r), in_ids[o], in_dists[o]});
      }
    }
    std::stable_sort(all.begin(), all.end(), [](const It& a, const It& c) { return a.score > c.score; });
    size_t n = std::min(all.size(), size_t(k));
    for (int j = 0; j < k; ++j) {
      out_ids[b * k + j] = size_t(j) < n ? all[j].id : 0;
      out_dists[b * k + j] = size_t(j) < n ? all[j].d : INFINITY;
    }
    out_counts[b] = uint32_t(n);
  }
}

// Hybrid-score merge (indexManager.searchParallel, shard/index/search.go:259-298) for B requests of
// S sub-searches: the sets are the sub-searches' result ids (vamana.go:285-307 returns exactly
// those); FastOr / FastAnd; walk results in sub-search order; first occurrence appended, later ones
// add HybridScore (f32) and donate a distance if the first had none (NaN = nil); slices.SortFunc by
// HybridScore descending — unstable in Go, stable (first-appearance order) here.
// in_*: S x B x k, counts S x B; out_*: B x (S*k).
void orc_hybrid_merge(const uint64_t* in_ids, const float* in_h, const float* in_d, const uint32_t* in_counts, int S,
                      size_t B, int k, int disjunction, uint64_t* out_ids, float* out_h, float* out_d,
                      uint32_t* out_counts) {
  const size_t M = size_t(S) * k;
  for (size_t b = 0; b < B; ++b) {
    std::vector<std::vector<uint64_t>> sets(S);
    for (int s = 0; s < S; ++s)
      for (uint32_t r = 0; r < std::min<uint32_t>(in_counts[size_t(s) * B + b], k); ++r)
        sets[s].push_back(in_ids[(size_t(s) * B + b) * k + r]);
    auto in_final = [&](uint64_t id) {
      if (disjunction) return true;
      for (int s = 0; s < S; ++s)
        if (std::find(sets[s].begin(), sets[s].end(), id) == sets[s].end()) return false;
      return true;
    };
    struct Res { uint64_t id; float h; float d; };
    std::vector<Res> fin;
    for (int s = 0; s < S; ++s)
      for (uint32_t r = 0; r < std::min<uint32_t>(in_counts[size_t(s) * B + b], k); ++r) {
        const size_t o = (size_t(s) * B + b) * k + r;
        if (!in_final(in_ids[o])) continue;
        auto it = std::find_if(fin.begin(), fin.end(), [&](const Res& x) { return x.id == in_ids[o]; });
        if (it == fin.end()) fin.push_back(Res{in_ids[o], in_h[o], in_d[o]});
        else {
          it->h += in_h[o];
          if (std::isnan(it->d) && !std::isnan(in_d[o])) it->d = in_d[o];
        }
      }
    std::stable_sort(fin.begin(), fin.end(), [](const Res& a, const Res& c) { return a.h > c.h; });
    for (size_t j = 0; j < M; ++j) {
      out_ids[b * M + j] = j < fin.size() ? fin[j].id : 0;
      out_h[b * M + j] = j < fin.size() ? fin[j].h : -INFINITY;
      out_d[b * M + j] = j < fin.size() ? fin[j].d : INFINITY;
    }
    out_counts[b] = uint32_t(fin.size());
  }
}

// Per-shard request limit (cluster/actions.go:291-299).
int orc_shard_limit(int limit, int nshards, int maxSearchLimit) {
  int target = int(float(limit) * (1 / float(nshards)) * 1.42f + 10.0f);
  if (target > maxSearchLimit) target = maxSearchLimit;
  if (target > limit) target = limit;
  return target;
}

int orc_hw_threads() { return int(std::thread::hardware_concurrency()); }

}  // extern "C"
