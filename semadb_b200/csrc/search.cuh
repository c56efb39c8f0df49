// search.cuh — K1/K2/K3: batched Vamana greedy beam search, one warp per query.
//
// Restates greedySearch (shard/index/vamana/search.go:9-102) + DistSet.AddWithLimit
// (distset.go:166-200) for a whole batch of queries:
//   * persistent CTAs; each warp pulls query indices from a global counter;
//   * the searchSize-bounded candidate list, the exact visited set (open-addressed hash
//     of node ids) and the per-hop neighbour staging live in shared memory;
//   * per hop: one coalesced 256-byte adjacency-row load, parallel visited test-and-set,
//     ballot compaction in adjacency order, neighbour vector rows gathered with 128-bit
//     streaming loads (an 8-lane group per row, up to 32+ rows in flight per warp),
//     distances in the reference's exact summation order (common.cuh), then the
//     insertions applied sequentially in adjacency order with ballot/shift steps so
//     every tie behaves like the reference (reject only d > worst, overwrite the last
//     slot, bubble while strictly smaller).
// Algorithmic bytes per query = n_dist*row_bytes + n_hops*R*4 (SURVEY.md §8d); the
// kernel reports n_hops and n_dist per query.
// Evaluators: f32 rows (fixed dims pipelined, any dim generic), bit rows (hamming / jaccard),
// PQ codes against the query's ADC table in global or in shared memory (bulk async copy),
// dim-2 haversine rows (one lane per candidate, float64 math).
// Epilogue: the top-k goes to the caller's buffers (device, or mapped host memory) and, for a
// sharded search, straight into every peer GPU's gather buffer (PeerGather).
#pragma once
#include "common.cuh"

namespace sdb {

constexpr int LIST_SLOTS = 80;   // > max searchSize (75); lanes cover positions lane + 32j, j < 3
constexpr int CAND_SLOTS = 64;   // >= max degreeBound (64), 2 per lane
constexpr uint32_t EXPANDED_FLAG = 0x80000000u;
constexpr uint32_t ID_MASK = 0x7FFFFFFFu;
constexpr uint32_t COUNT_OVERFLOW = 0xFFFFFFFFu;  // out_counts marker: visited table overflowed

// Cross-shard exchange fused into the epilogue (replaces the fan-in of cluster/actions.go:357-376
// + one all-gather per result tensor): a query-warp stores its shard's top-k straight into every
// peer GPU's gather buffer over NVLink — peer-mapped pointers, slot [shard][query], ids tagged
// with the shard index — so that after one cross-GPU barrier every GPU holds all S lists.
constexpr int MAX_PEERS = 16;
struct PeerGather {
  uint32_t n;        // peers (0 = off), including this GPU
  uint32_t shard;    // this GPU's shard index
  uint32_t limit;    // per-shard result limit (actions.go:291-299), <= k
  uint64_t tag;      // shard << 40, or'ed into the node ids
  uint64_t* ids[MAX_PEERS];     // peer p's [S][B][k]
  float* dists[MAX_PEERS];      // peer p's [S][B][k]
  uint32_t* counts[MAX_PEERS];  // peer p's [S][B]
};

struct SearchArgs {
  PeerGather pg;
  // store
  const float* vec;        // [rows][vec_pitch]
  uint32_t vec_pitch;      // floats per row (multiple of 4)
  const uint64_t* bits;    // [rows][bits_pitch] (binary store)
  uint32_t bits_pitch;     // u64 per row (multiple of 2)
  uint32_t words;          // ceil(dim/64)
  const uint8_t* codes;    // [rows][codes_pitch] (product store)
  uint32_t codes_pitch;    // bytes per row (multiple of 16)
  const float* adc;        // [B][M*K] per-query ADC tables (product store)
  uint32_t pqM, pqK;
  const float* pq_cent;    // [M][K][sub] flatCentroids (EVAL_ADC_FLY: table entries computed on the fly)
  const float* bq_thr;     // [dim] binary threshold (query encode)
  int bit_metric;
  // graph
  const uint32_t* adj;     // [rows][R], INVALID_ID padded
  uint32_t R;
  const uint32_t* start_extra;  // edges of node 1 beyond R (normally none)
  uint32_t n_start_extra;
  uint32_t rows;
  // batch
  const float* queries;    // [B][dim]
  uint32_t dim;
  uint32_t B;
  uint32_t L, k;
  // outputs
  uint64_t* out_ids;       // [B][k]
  float* out_dists;        // [B][k]
  uint32_t* out_counts;    // [B]
  uint32_t* out_hops;      // [B]
  uint32_t* out_ndist;     // [B]
  // optional: visited (expanded) list in expansion order, for the insert path
  uint32_t* vis_ids;       // [B][vis_cap]
  float* vis_dists;
  uint32_t* vis_len;
  uint32_t vis_cap;
  // optional filters (search.go:33-51,93-95), one per request like shard/index/search.go:59-85:
  // filter f = ascending ids filter_ids[filter_off[f] .. filter_off[f+1]); query qi uses filter
  // query_filter[qi] (nullptr: every query uses filter 0). The first min(L, n) ids of a filter
  // are its seeds. filter_bits: optional dense bitmask over rows of filter 0 (shared-filter calls).
  const uint32_t* filter_ids;
  const uint32_t* filter_off;
  const int32_t* query_filter;
  const uint32_t* filter_bits;
  // optional work map: this launch covers queries qmap[0..n_work) (nullptr: 0..B-1). A batch that
  // mixes filtered and unfiltered requests runs as two launches over disjoint subsets.
  const uint32_t* qmap;
  uint32_t n_work;
  // RETRY launch: one exact visited bitmap over all rows per CTA, in global memory
  uint32_t* retry_bitmap;
  uint32_t bitmap_words;
  // work distribution: work_counter hands out batch slots; a query whose visited table
  // overflows is appended to retry_list and re-run by the RETRY launch (bigger table).
  uint32_t vt_slots;  // VisitedCompactN slot count for this launch
  uint32_t* work_counter;
  uint32_t* retry_list;
  uint32_t* retry_count;
  // optional per-query parameters {L, k, gather count limit, 0} (sdb_request), read by the REQ
  // variants only: nullptr = L, k and pg.limit for every query. With them, k is the stride of the
  // outputs and of the gather slots.
  const uint4* req;
};

// ---- exact visited set, compact form with a launch-time slot count ------------------------
// 16-bit entries in BUCKETS of four (one 64-bit shared-memory word): pi(id) = id*A mod 2^b is a
// bijection on the b-bit id space; span = ceil(2^b / buckets), home bucket = pi / span, remainder
// = pi % span, entry = 1 + remainder + disp*span (disp = bucket displacement, 0 = empty slot) —
// quotienting makes a 16-bit entry identify the id exactly. One 64-bit load shows a bucket's four
// entries, a SWAR compare finds the id or a free slot, one 64-bit CAS claims it: at the load
// factors of a search (<= 50 % typically, 87.5 % at most) almost every id resolves in its home
// bucket, where the linear-probe table of round 1 needed 4-6 vote-loop iterations per hop for the
// longest of its 64 chains (31 % of the hamming kernel's instructions, profiles/r02_k2_*).
// slots = 4 * buckets is chosen per launch (SearchArgs::vt_slots: 5888 keeps a dim-128 query-warp
// at 12.9 KB of shared memory; search.cu steps it up for workloads that visit more nodes).
// disp <= dmax = (65535 - span) / span; beyond that, above 87.5 % load, or when span does not fit
// 16 bits (more than ~96 M rows at 5888 slots) the query goes to the RETRY launch (exact bitmap).
struct VisitedCompactN {
  static __host__ __device__ constexpr size_t bytes(uint32_t slots) { return size_t(slots) * 2; }
  unsigned long long* t;
  uint32_t nbuckets, mask, span, magic, used, dmax, lim;
  bool failed, unusable;
  static constexpr unsigned long long ONES = 0x0001000100010001ull, HIGHS = 0x8000800080008000ull;
  __device__ __forceinline__ uint32_t limit() const { return lim; }
  __device__ __forceinline__ void init(unsigned char* base, uint32_t rows, uint32_t slots, uint32_t*, uint32_t) {
    t = reinterpret_cast<unsigned long long*>(base);
    nbuckets = slots / 4;
    uint32_t b = rows <= 2 ? 1 : 32 - __clz(rows - 1);
    if (b < 16) b = 16;
    mask = b >= 32 ? 0xFFFFFFFFu : ((1u << b) - 1);
    const uint64_t space = uint64_t(1) << b;
    span = uint32_t((space + nbuckets - 1) / nbuckets);
    magic = uint32_t((uint64_t(1) << 32) / span);
    used = uint32_t((space + span - 1) / span);  // buckets that can be a home
    unusable = span > 65534u;
    dmax = unusable ? 0 : (65535u - span) / span;
    if (dmax > 4096) dmax = 4096;
    lim = unusable ? 0 : used * 4 - used / 2;  // 87.5 % of the entries
  }
  __device__ __forceinline__ void clear(int lane) {
    uint4 z = make_uint4(0, 0, 0, 0);
    uint4* p = reinterpret_cast<uint4*>(t);
    for (uint32_t i = lane; i < nbuckets / 2; i += 32) p[i] = z;
    if ((nbuckets & 1u) && lane == 0) t[nbuckets - 1] = 0ull;
    failed = unusable;
  }
  __device__ __forceinline__ void home(uint32_t id, uint32_t& bucket, uint32_t& code) const {
    const uint32_t v = (id * 0x9E3779B1u) & mask;
    uint32_t q = __umulhi(v, magic);
    uint32_t r = v - q * span;
    if (r >= span) { ++q; r -= span; }  // the estimate is short by at most one
    bucket = q;
    code = 1 + r;
  }
  // which 16-bit lane of w equals c (bit 15 of that lane set in the result), 0 if none
  static __device__ __forceinline__ unsigned long long match16(unsigned long long w, uint32_t c) {
    const unsigned long long x = w ^ (ONES * c);
    return (x - ONES) & ~x & HIGHS;
  }
  // one probe step of one id: returns true when the id is resolved
  __device__ __forceinline__ bool step(uint32_t& bucket, uint32_t& code, uint32_t& disp, bool& isnew, bool& spill) {
    volatile unsigned long long* tw = t;
    const unsigned long long w = tw[bucket];
    if (match16(w, code)) return true;               // already visited
    const unsigned long long z = match16(w, 0u);      // free slots of the bucket
    if (z) {
      const int sh = (__ffsll((long long)z) - 1) & ~15;  // bit offset of the first free 16-bit slot
      const unsigned long long old = atomicCAS(const_cast<unsigned long long*>(tw) + bucket, w, w | ((unsigned long long)code << sh));
      if (old == w) { isnew = true; return true; }
      return false;                                    // the word changed under us: look again
    }
    bucket = bucket + 1 == used ? 0 : bucket + 1;     // bucket full of other ids
    code += span;
    if (++disp > dmax) { spill = true; return true; }
    return false;
  }
  // Two ids per lane (adjacency slots lane and lane+32) probed in one vote-driven loop — a
  // data-dependent `while` around the CAS makes ptxas emit WARPSYNC.COLLECTIVE trampolines for
  // every later shuffle.
  __device__ __forceinline__ void test_and_set2(uint32_t i0, bool a0, uint32_t i1, bool a1, bool& n0, bool& n1, int) {
    uint32_t b0, b1, c0, c1;
    home(i0, b0, c0);
    home(i1, b1, c1);
    uint32_t d0 = 0, d1 = 0;
    bool p0 = a0 && !unusable, p1 = a1 && !unusable, spill = false;
    n0 = false;
    n1 = false;
    while (__any_sync(SDB_FULL, p0 || p1)) {
      if (p0) p0 = !step(b0, c0, d0, n0, spill);
      if (p1) p1 = !step(b1, c1, d1, n1, spill);
    }
    if (__any_sync(SDB_FULL, spill)) failed = true;
  }
  // Read-only hint for the speculative row prefetch: false only if id is certainly in the set
  // (home bucket and the next one, no loop, no vote); "true" may be wrong, which costs one wasted
  // prefetch.
  __device__ __forceinline__ bool maybe_new(uint32_t id) const {
    uint32_t bucket, c;
    home(id, bucket, c);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const unsigned long long w = t[bucket];
      if (match16(w, c)) return false;
      if (match16(w, 0u)) return true;
      bucket = bucket + 1 == used ? 0 : bucket + 1;
      c += span;
    }
    return true;
  }
};

// ---- exact visited set of the RETRY launch: one bit per row, in global memory ------------
// The reference's visited set never fills up (a bitset sized by maxNodeId, distset.go:41,
// 140-155). A query whose compact shared-memory table overflowed is re-run against this
// bitmap — one per resident CTA of the RETRY launch, cleared per query — so a search always
// completes exactly, however many nodes it visits; the overflow marker never reaches a caller.
struct VisitedBitmap {
  static __host__ __device__ constexpr size_t bytes(uint32_t) { return 0; }
  uint32_t* t;
  uint32_t words;
  bool failed;
  __device__ __forceinline__ uint32_t limit() const { return 0xFFFFFFFFu; }
  __device__ __forceinline__ void init(unsigned char*, uint32_t, uint32_t, uint32_t* g, uint32_t gwords) {
    t = g + size_t(blockIdx.x) * gwords;
    words = gwords;
  }
  __device__ __forceinline__ void clear(int lane) {
    uint4 z = make_uint4(0, 0, 0, 0);
    uint4* p = reinterpret_cast<uint4*>(t);
    for (uint32_t i = lane; i < words / 4; i += 32) p[i] = z;
    failed = false;
    __syncwarp();
  }
  __device__ __forceinline__ bool test_and_set(uint32_t id, bool active, int) {
    if (!active) return false;
    const uint32_t bit = 1u << (id & 31);
    return (atomicOr(t + (id >> 5), bit) & bit) == 0;
  }
  __device__ __forceinline__ void test_and_set2(uint32_t i0, bool a0, uint32_t i1, bool a1, bool& n0, bool& n1, int lane) {
    n0 = test_and_set(i0, a0, lane);
    n1 = test_and_set(i1, a1, lane);
    __syncwarp();
  }
  __device__ __forceinline__ bool maybe_new(uint32_t id) const { return ((t[id >> 5] >> (id & 31)) & 1u) == 0; }
};

// ---- bounded candidate list (distset.go:133-200) in shared memory ------------------
struct CandList {
  uint32_t* id;  // EXPANDED_FLAG in the top bit
  float* dist;
  int len;
  int cap;
  bool nan_seen;  // a NaN distance reached this list: only the sequential form is exact from then on
  // Insert one element with AddWithLimit semantics; caller has already applied the
  // "full && d > worst" rejection. Warp-synchronous; all lanes call with the same args.
  __device__ __forceinline__ void insert(uint32_t nid, float d, int lane) {
    const bool full = (len == cap);
    const int n_items = full ? cap - 1 : len;  // full: last slot is overwritten first
    // bubble: new element stops right after the last p with !(d < dist[p])
    int pos = 0;
#pragma unroll
    for (int j = 2; j >= 0; --j) {
      int p = lane + 32 * j;
      bool ok = (p < n_items) && !(d < dist[p]);
      uint32_t b = __ballot_sync(SDB_FULL, ok);
      if (b && pos == 0) pos = 32 * j + (32 - __clz(b));
    }
    // shift [pos, n_items) up by one
    uint32_t mv_id[3];
    float mv_d[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      int p = lane + 32 * j;
      if (p >= pos && p < n_items) { mv_id[j] = id[p]; mv_d[j] = dist[p]; }
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      int p = lane + 32 * j;
      if (p >= pos && p < n_items) { id[p + 1] = mv_id[j]; dist[p + 1] = mv_d[j]; }
    }
    if (lane == 0) { id[pos] = nid; dist[pos] = d; }
    if (!full) ++len;
    __syncwarp();
  }

  // Batch form of AddWithLimit (distset.go:166-200) for n staged candidates, arrival order =
  // index. Let U = list ∪ candidates ordered by (distance, list-before-candidates, arrival).
  // If the elements of U at ranks cap-1 and cap have different distances (or |U| <= cap),
  // applying insert() one candidate at a time yields exactly the first cap elements of U in
  // that order: an element with d <= theta (the rank cap-1 distance) is never rejected
  // (worst >= theta whenever the list is full) and never evicted (that would need cap+1
  // elements with d <= theta); equal distances keep arrival order (strict '<' bubble).
  // If a tie straddles the cut the reference lets the newest equal win the last slot
  // (distset.go:184-194); that one slot is fixed up exactly (see below), which matters for
  // integer distances (hamming, PQ) where such ties are everywhere; with TIEFIX = false (float
  // metrics, ties rare) a tie returns false instead. Also returns false, with the list
  // untouched, if a candidate distance is NaN (then, and for the rest of the query, the caller
  // applies the sequential form) or fewer than min_m candidates survive (the sequential form
  // is cheaper).
  template <bool TIEFIX>
  __device__ __forceinline__ bool merge(const uint32_t* cid, const float* cdist, int n, int lane, uint32_t lt, int min_m) {
    const int len0 = len;
    const bool full = (len0 == cap);
    const float worst = full ? dist[cap - 1] : 0.0f;
    const float d0 = lane < n ? cdist[lane] : 0.0f;
    const float d1 = lane + 32 < n ? cdist[lane + 32] : 0.0f;
    const bool s0 = lane < n && !(full && d0 > worst);
    const bool s1 = lane + 32 < n && !(full && d1 > worst);
    const uint32_t b0 = __ballot_sync(SDB_FULL, s0), b1 = __ballot_sync(SDB_FULL, s1);
    const int m = __popc(b0) + __popc(b1);
    if (m == 0) return true;
    if (__any_sync(SDB_FULL, (s0 && d0 != d0) || (s1 && d1 != d1))) nan_seen = true;
    if (nan_seen || m < min_m) return false;
    // position among the old items: number of items with dist <= d (newcomers go after equals)
    int lo0 = 0, hi0 = len0, lo1 = 0, hi1 = len0;
#pragma unroll
    for (int it = 0; it < 7; ++it) {  // len0 <= 96 < 128
      const int m0 = (lo0 + hi0) >> 1, m1 = (lo1 + hi1) >> 1;
      const float x0 = dist[min(m0, LIST_SLOTS - 1)], x1 = dist[min(m1, LIST_SLOTS - 1)];
      if (lo0 < hi0) { if (x0 <= d0) lo0 = m0 + 1; else hi0 = m0; }
      if (lo1 < hi1) { if (x1 <= d1) lo1 = m1 + 1; else hi1 = m1; }
    }
    // rank among the surviving candidates by (distance, arrival)
    int r0 = 0, r1 = 0;
    if (m > 1) {
      for (uint32_t bb = b0; bb; bb &= bb - 1) {
        const int c = __ffs(bb) - 1;
        const float dc = __shfl_sync(SDB_FULL, d0, c);
        r0 += (dc < d0) || (dc == d0 && c < lane);
        r1 += (dc <= d1);
      }
      for (uint32_t bb = b1; bb; bb &= bb - 1) {
        const int c = __ffs(bb) - 1;
        const float dc = __shfl_sync(SDB_FULL, d1, c);
        r0 += (dc < d0);
        r1 += (dc < d1) || (dc == d1 && c < lane);
      }
    }
    const int f0 = s0 ? lo0 + r0 : 0x7FFF, f1 = s1 ? lo1 + r1 : 0x7FFF;
    // which final positions are taken by candidates (positions < 96 are all that matter)
    uint32_t x[3];
#pragma unroll
    for (int w = 0; w < 3; ++w) {
      x[w] = ((f0 >> 5) == w ? (1u << (f0 & 31)) : 0u) | ((f1 >> 5) == w ? (1u << (f1 & 31)) : 0u);
      x[w] = __reduce_or_sync(SDB_FULL, x[w]);
    }
    // old item landing at final position P = lane + 32j is item P - (candidates below P)
    uint32_t oid[3];
    float od[3];
    bool take[3];
    int below = 0;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int P = lane + 32 * j;
      const bool occ = (x[j] >> lane) & 1u;
      const int i = P - below - __popc(x[j] & lt);
      take[j] = !occ && P <= cap && i < len0;
      oid[j] = 0;
      od[j] = 0.0f;
      if (take[j]) { oid[j] = id[i]; od[j] = dist[i]; }
      below += __popc(x[j]);
    }
    // Tie across the cut: ranks cap-1 (last kept) and cap (first dropped) share a distance
    // theta. Sequential AddWithLimit then differs from the stable order in exactly one slot:
    // once the list is all <= theta, a newcomer with d == theta overwrites the last slot
    // (distset.go:184-194) and a newcomer with d < theta evicts it. So the last slot ends up
    // holding the last candidate with d == theta that arrives after the last *strict* insert
    // (a candidate with d < the worst of its time), if there is one. The last strict insert
    // is the later of: the candidate whose arrival brings the number of elements <= theta to
    // cap (every <= theta candidate up to it met a worst > theta), and the last candidate
    // with d < theta. Everything else equals the stable order computed above.
    int x_last = -1;
    float theta = 0.0f;
    if (len0 + m > cap) {
      float dcut[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int P = cap - 1 + e, j = P >> 5, l = P & 31;
        const float mine = j == 0 ? od[0] : (j == 1 ? od[1] : od[2]);
        float v = __shfl_sync(SDB_FULL, mine, l);
        const uint32_t h0 = __ballot_sync(SDB_FULL, f0 == P), h1 = __ballot_sync(SDB_FULL, f1 == P);
        if (h0) v = __shfl_sync(SDB_FULL, d0, __ffs(h0) - 1);
        if (h1) v = __shfl_sync(SDB_FULL, d1, __ffs(h1) - 1);
        dcut[e] = v;
      }
      if (dcut[0] == dcut[1]) {
        // float metrics: ties are rare — hand the hop to the sequential form (list untouched)
        if (!TIEFIX) return false;
        theta = dcut[0];
        // old items with dist <= theta (uniform binary search)
        int lo = 0, hi = len0;
#pragma unroll
        for (int it = 0; it < 7; ++it) {
          const int mid = (lo + hi) >> 1;
          const float xm = dist[min(mid, LIST_SLOTS - 1)];
          if (lo < hi) { if (xm <= theta) lo = mid + 1; else hi = mid; }
        }
        const int need = cap - lo;  // candidates <= theta still needed to fill the list
        const uint32_t le0 = __ballot_sync(SDB_FULL, s0 && d0 <= theta), le1 = __ballot_sync(SDB_FULL, s1 && d1 <= theta);
        const uint32_t ls0 = __ballot_sync(SDB_FULL, s0 && d0 < theta), ls1 = __ballot_sync(SDB_FULL, s1 && d1 < theta);
        uint32_t eq0 = le0 & ~ls0, eq1 = le1 & ~ls1;
        int c_t = -1;
        if (need > 0) {
          const int n0 = __popc(le0);
          c_t = need <= n0 ? int(__fns(le0, 0, need)) : 32 + int(__fns(le1, 0, need - n0));
        }
        const int i1 = ls1 ? 63 - __clz(ls1) : (ls0 ? 31 - __clz(ls0) : -1);
        const int t_last = max(c_t, i1);
        // keep only d == theta candidates that arrive after t_last
        if (t_last >= 0) {
          eq0 = t_last >= 31 ? 0u : (eq0 & ~((2u << t_last) - 1u));
          if (t_last >= 32) eq1 = t_last >= 63 ? 0u : (eq1 & ~((2u << (t_last - 32)) - 1u));
        }
        x_last = eq1 ? 63 - __clz(eq1) : (eq0 ? 31 - __clz(eq0) : -1);
      }
    }
    __syncwarp();
    const int newlen = min(cap, len0 + m);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int P = lane + 32 * j;
      if (take[j] && P < newlen) { id[P] = oid[j]; dist[P] = od[j]; }
    }
    if (f0 < newlen) { id[f0] = cid[lane]; dist[f0] = d0; }
    if (f1 < newlen) { id[f1] = cid[lane + 32]; dist[f1] = d1; }
    len = newlen;
    __syncwarp();
    if (x_last >= 0) {
      if (lane == 0) { id[cap - 1] = cid[x_last]; dist[cap - 1] = theta; }
      __syncwarp();
    }
    return true;
  }
};

// ---- distance evaluators -----------------------------------------------------------
// Each evaluates cdist[c] = dist(query, row cid[c]) for c in [0, n), warp-cooperatively.

// f32 rows, dim = 32*TRIPS exactly. An 8-lane group owns a row: lane g loads the float4 at
// element 32t + 4g of every trip (one full 128-byte line per group per load instruction) and
// so holds partial sums 4g..4g+3 of the asm's 32. Row sets (4 rows per warp-wide load) are
// software-pipelined: SETS sets stay in flight and set s+SETS is issued as soon as set s has
// been consumed. Queries of <= 4 trips live in registers (read straight from global).
// Measured on B200 (profiles/r01_ab_k1.txt): narrower groups (4 or 2 lanes per row => fewer
// shuffles, 32- or 64-byte pieces of 8 or 16 rows per load) run 1.4x / 2.7x slower — the L1
// processes one 128-byte line per wavefront, so lines per instruction is what counts; parking
// the partial sums in shared memory and folding them in one lane also lost to the shuffles.
template <int METRIC, int TRIPS, int SETS>
struct FloatEvalFixed {
  static constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
  static constexpr bool QREG = (TRIPS <= 4);
  float4 q[QREG ? TRIPS : 1];
  const float* qs;
  __device__ __forceinline__ void load_query(const float* qsmem, const float* qg, int lane) {
    qs = qsmem;
    if (QREG) {
#pragma unroll
      for (int t = 0; t < TRIPS; ++t) q[t] = ldg_f4(qg + 32 * t + 4 * (lane & 7));
    }
  }
  __device__ __forceinline__ void issue(const SearchArgs& a, const uint32_t* cid, int n, int s, int g, int grp,
                                        float4 (&v)[TRIPS]) {
    // groups past the end re-read the hop's first candidate row (this warp's own, cache-hot;
    // no branch, result discarded) so every load is unconditional. Not the query's own row,
    // which may live in mapped host memory, and not one fixed row for everybody: a single
    // line hammered by every warp of the GPU cost C1 (L2-resident) two thirds of its QPS.
    const int ci = s * 4 + grp;
    const float* row = a.vec + size_t(cid[ci < n ? ci : 0]) * a.vec_pitch + 4 * g;
#pragma unroll
    for (int t = 0; t < TRIPS; ++t) v[t] = ldg_f4_stream(row + 32 * t);
  }
  __device__ __forceinline__ void consume(float* cdist, int n, int s, int g, int grp, const float4 (&v)[TRIPS]) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int t = 0; t < TRIPS; ++t) {
      const float4 x = QREG ? q[t] : *reinterpret_cast<const float4*>(qs + 32 * t + 4 * g);
      trip_accum<L2>(x, v[t], acc);
    }
    const float r = group_reduce(acc, 0.0f);
    const int ci = s * 4 + grp;
    if (g == 0 && ci < n) cdist[ci] = metric_epilogue<METRIC>(r);
  }
  __device__ __forceinline__ void eval(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane) {
    const int g = lane & 7, grp = lane >> 3;
    const int nsets = (n + 3) >> 2;
    float4 v[SETS][TRIPS];
#pragma unroll
    for (int u = 0; u < SETS; ++u)
      if (u < nsets) issue(a, cid, n, u, g, grp, v[u]);
    for (int base = 0; base < nsets; base += SETS) {
#pragma unroll
      for (int u = 0; u < SETS; ++u) {
        const int s = base + u;
        if (s >= nsets) break;  // warp-uniform
        consume(cdist, n, s, g, grp, v[u]);
        if (s + SETS < nsets) issue(a, cid, n, s + SETS, g, grp, v[u]);
      }
    }
    __syncwarp();
  }
};

// f32 rows, any dim: runtime trips + scalar tail, query in shared memory.
template <int METRIC>
struct FloatEvalGeneric {
  static constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
  const float* qs;
  __device__ __forceinline__ void load_query(const float* qsmem, int) { qs = qsmem; }
  __device__ __forceinline__ void eval(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane) {
    const int g = lane & 7, grp = lane >> 3;
    const int trips = a.dim >> 5;
    const int tail0 = trips << 5;
    for (int base = 0; base < n; base += 4) {
      int ci = base + grp;
      bool act = ci < n;
      const float* row = a.vec + size_t(act ? cid[ci] : cid[0]) * a.vec_pitch;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      int t = 0;
      for (; t + 8 <= trips; t += 8) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = ldg_f4_stream(row + 32 * (t + u) + 4 * g);
#pragma unroll
        for (int u = 0; u < 8; ++u)
          trip_accum<L2>(*reinterpret_cast<const float4*>(qs + 32 * (t + u) + 4 * g), v[u], acc);
      }
      for (; t < trips; ++t) {
        float4 v = ldg_f4_stream(row + 32 * t + 4 * g);
        trip_accum<L2>(*reinterpret_cast<const float4*>(qs + 32 * t + 4 * g), v, acc);
      }
      float tail = 0.0f;
      if (g == 0)
        for (int i = tail0; i < int(a.dim); ++i) tail = tail_accum<L2>(qs[i], __ldg(row + i), tail);
      float r = group_reduce(acc, tail);
      if (g == 0 && act) cdist[ci] = metric_epilogue<METRIC>(r);
    }
    __syncwarp();
  }
};

// Bit-packed rows (binaryQuantizer.DistanceFromFloat, binary.go:187-201): the query is
// encoded once (binary.go:103-129) into shared memory; hamming / jaccard by popcount
// (distance.go:45-67). An 8-lane group owns a row, 16 bytes per lane per 128-byte chunk (one
// full line per group per load); NCH chunks cover rows of up to NCH*1024 bits. Row sets are
// pipelined like FloatEvalFixed (SETS sets = 4*SETS rows in flight). Integer sums: the
// cross-lane reduction order is free.
template <int BMETRIC, int NCH, int SETS>
struct BitEval {
  uint64_t q[NCH][2];  // this lane's slice of the encoded query
  __device__ __forceinline__ void encode_query(const SearchArgs& a, const float* qsmem, uint64_t* qbits, int lane) {
    // bit i%64 of word i/64 = q[i] > thr[i]; qsmem = the query in GLOBAL (or mapped host) memory, read
    // once, coalesced — a shared-memory copy of the floats (4 KB at 1024 dims) would only cost residency
    for (uint32_t w = 0; w < a.bits_pitch; ++w) {
      uint64_t word = 0;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t i = w * 64 + h * 32 + lane;
        bool on = (i < a.dim) && (__ldg(qsmem + (i < a.dim ? i : 0)) > __ldg(a.bq_thr + (i < a.dim ? i : 0)));
        uint32_t b = __ballot_sync(SDB_FULL, on);
        word |= uint64_t(b) << (32 * h);
      }
      if (lane == 0) qbits[w] = word;
    }
    __syncwarp();
    const int g = lane & 7;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const uint32_t w = c * 16 + 2 * g;
      q[c][0] = w < a.bits_pitch ? qbits[w] : 0;
      q[c][1] = w + 1 < a.bits_pitch ? qbits[w + 1] : 0;
    }
  }
  __device__ __forceinline__ void issue(const SearchArgs& a, const uint32_t* cid, int n, int s, int g, int grp,
                                        uint4 (&v)[NCH]) {
    // groups past the end re-read the first candidate's row (result discarded)
    const int ci = s * 4 + grp;
    const uint64_t* row = a.bits + size_t(cid[ci < n ? ci : 0]) * a.bits_pitch;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const uint32_t w = c * 16 + 2 * g;
      v[c] = w < a.bits_pitch ? ldg_u4_stream(row + w) : make_uint4(0, 0, 0, 0);
    }
  }
  __device__ __forceinline__ void consume(float* cdist, int n, int s, int g, int grp, const uint4 (&v)[NCH]) {
    int x = 0, u = 0;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const uint64_t r0 = (uint64_t(v[c].y) << 32) | v[c].x, r1 = (uint64_t(v[c].w) << 32) | v[c].z;
      if (BMETRIC == METRIC_JACCARD) {
        x += __popcll(q[c][0] & r0) + __popcll(q[c][1] & r1);
        u += __popcll(q[c][0] | r0) + __popcll(q[c][1] | r1);
      } else {
        x += __popcll(q[c][0] ^ r0) + __popcll(q[c][1] ^ r1);
      }
    }
#pragma unroll
    for (int o = 4; o >= 1; o >>= 1) {
      x += __shfl_down_sync(SDB_FULL, x, o, 8);
      if (BMETRIC == METRIC_JACCARD) u += __shfl_down_sync(SDB_FULL, u, o, 8);
    }
    const int ci = s * 4 + grp;
    if (g == 0 && ci < n) cdist[ci] = bits_finish(BMETRIC, x, u);
  }
  template <class Hook>
  __device__ __forceinline__ void eval(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane, Hook&& hook) {
    const int g = lane & 7, grp = lane >> 3;
    const int nsets = (n + 3) >> 2;
    uint4 v[SETS][NCH];
#pragma unroll
    for (int u = 0; u < SETS; ++u)
      if (u < nsets) issue(a, cid, n, u, g, grp, v[u]);
    hook();  // this hop's first rows are in flight: speculative prefetches for the next hop ride along
    for (int base = 0; base < nsets; base += SETS) {
#pragma unroll
      for (int u = 0; u < SETS; ++u) {
        const int s = base + u;
        if (s >= nsets) break;  // warp-uniform
        consume(cdist, n, s, g, grp, v[u]);
        if (s + SETS < nsets) issue(a, cid, n, s + SETS, g, grp, v[u]);
      }
    }
    __syncwarp();
  }
};

// Rows of up to 1024 bits whose pitch is a multiple of 32 bytes (NCH = 0 selects this form): FOUR
// lanes own a row, 32 bytes per lane in one 256-bit load (LDG.E.256), eight rows per warp-wide
// load, two shuffle steps per reduction — half the instructions per row of the 8-lane form, which
// is what the hamming search is bound by once the visited probe is cheap (profiles/r02_k2_*: the
// evaluator was 41 % of its instructions). SETS sets of 8 rows stay in flight.
template <int BMETRIC, int SETS>
struct BitEval<BMETRIC, 0, SETS> {
  uint64_t q[4];  // this lane's 32-byte slice of the encoded query
  __device__ __forceinline__ void encode_query(const SearchArgs& a, const float* qsmem, uint64_t* qbits, int lane) {
    for (uint32_t w = 0; w < a.bits_pitch; ++w) {
      uint64_t word = 0;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t i = w * 64 + h * 32 + lane;
        bool on = (i < a.dim) && (__ldg(qsmem + (i < a.dim ? i : 0)) > __ldg(a.bq_thr + (i < a.dim ? i : 0)));
        uint32_t b = __ballot_sync(SDB_FULL, on);
        word |= uint64_t(b) << (32 * h);
      }
      if (lane == 0) qbits[w] = word;
    }
    __syncwarp();
    const uint32_t w0 = 4u * (lane & 3);
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = w0 + j < a.bits_pitch ? qbits[w0 + j] : 0;
  }
  __device__ __forceinline__ void issue(const SearchArgs& a, const uint32_t* cid, int n, int s, int h, int grp, uint4 (&v)[2]) {
    const int ci = s * 8 + grp;  // groups past the end re-read the first candidate's row (result discarded)
    const uint64_t* row = a.bits + size_t(cid[ci < n ? ci : 0]) * a.bits_pitch;
    if (4u * h < a.bits_pitch) ldg_u8_stream(row + 4 * h, v[0], v[1]);
    else { v[0] = make_uint4(0, 0, 0, 0); v[1] = v[0]; }
  }
  __device__ __forceinline__ void consume(float* cdist, int n, int s, int h, int grp, const uint4 (&v)[2]) {
    const uint64_t r[4] = {(uint64_t(v[0].y) << 32) | v[0].x, (uint64_t(v[0].w) << 32) | v[0].z,
                           (uint64_t(v[1].y) << 32) | v[1].x, (uint64_t(v[1].w) << 32) | v[1].z};
    int x = 0, u = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (BMETRIC == METRIC_JACCARD) { x += __popcll(q[j] & r[j]); u += __popcll(q[j] | r[j]); }
      else x += __popcll(q[j] ^ r[j]);
    }
#pragma unroll
    for (int o = 2; o >= 1; o >>= 1) {
      x += __shfl_down_sync(SDB_FULL, x, o, 4);
      if (BMETRIC == METRIC_JACCARD) u += __shfl_down_sync(SDB_FULL, u, o, 4);
    }
    const int ci = s * 8 + grp;
    if (h == 0 && ci < n) cdist[ci] = bits_finish(BMETRIC, x, u);
  }
  template <class Hook>
  __device__ __forceinline__ void eval(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane, Hook&& hook) {
    const int h = lane & 3, grp = lane >> 2;
    const int nsets = (n + 7) >> 3;
    uint4 v[SETS][2];
#pragma unroll
    for (int u = 0; u < SETS; ++u)
      if (u < nsets) issue(a, cid, n, u, h, grp, v[u]);
    hook();
    for (int base = 0; base < nsets; base += SETS) {
#pragma unroll
      for (int u = 0; u < SETS; ++u) {
        const int s = base + u;
        if (s >= nsets) break;  // warp-uniform
        consume(cdist, n, s, h, grp, v[u]);
        if (s + SETS < nsets) issue(a, cid, n, s + SETS, h, grp, v[u]);
      }
    }
    __syncwarp();
  }
};

// PQ codes (productQuantizer.DistanceFromFloat, product.go:238-277): per-query ADC table
// (built by a separate kernel, product.go:255-263) read through L1/L2; one lane per
// candidate sums M table entries sequentially in f32 (product.go:271-275).
struct AdcEval {
  const float* table;  // [M*K] for this query (global)
  template <class Hook>
  __device__ __forceinline__ void eval(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane, Hook&& hook) {
    hook();
    for (int c = lane; c < n; c += 32) {
      const uint8_t* code = a.codes + size_t(cid[c]) * a.codes_pitch;
      float d = 0.0f;
      for (uint32_t i0 = 0; i0 < a.pqM; i0 += 16) {
        uint4 v = ldg_u4_stream(code + i0);
        uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          uint32_t i = i0 + j;
          if (i < a.pqM) {
            uint32_t cj = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
            d = __fadd_rn(d, __ldg(table + i * a.pqK + cj));
          }
        }
      }
      cdist[c] = d;
    }
    __syncwarp();
  }
};

// PQ codes with the query's ADC table resident in shared memory (the table is what every
// distance touches: M lookups per candidate, 288 k per query at C4 — through L1/L2 that was the
// bound). The table is pulled from global memory once per query by bulk async copies
// (cp.async.bulk, completion on an mbarrier). One lane owns two candidates (adjacency slots
// lane, lane+32): their code rows (NCH 16-byte chunks each) are all in flight before the first
// lookup, and the two sums advance as independent sequential f32 chains in sub-vector order
// (product.go:271-275), so the result is the same float the global-table path and the reference
// produce.
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_addr(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
               "l"(src), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}

template <int NCH>
struct AdcEvalSmem {
  const float* table;  // [M*K] for this query (shared memory)
  // pull the query's table into shared memory; returns after it has landed
  __device__ __forceinline__ void load_table(float* tab, const float* src, uint32_t nfloats, uint64_t* bar, uint32_t& phase,
                                             int lane) {
    table = tab;
    // earlier generic-proxy reads of the old table are ordered before the async-proxy writes
    __syncwarp();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if ((nfloats & 3u) == 0) {
      const uint32_t bytes = nfloats * 4;
      constexpr uint32_t CHUNK = 8192;
      if (lane == 0) mbar_expect_tx(bar, bytes);
      __syncwarp();
      for (uint32_t off = uint32_t(lane) * CHUNK; off < bytes; off += 32 * CHUNK)
        bulk_g2s(reinterpret_cast<unsigned char*>(tab) + off, reinterpret_cast<const unsigned char*>(src) + off,
                 min(CHUNK, bytes - off), bar);
      mbar_wait(bar, phase);
      phase ^= 1u;
    } else {  // table rows not 16-byte sized: plain copy
      for (uint32_t i = lane; i < nfloats; i += 32) tab[i] = __ldg(src + i);
    }
    __syncwarp();
  }
  // TWO: the hop staged more than 32 candidates, lanes run a second chain for slot lane+32.
  // K256: K = 256 (the reference's maximum and the C4 shape): the table offset of sub-vector i
  // is the compile-time constant i*1024 B, so a lookup is shift/mask + LDS + FADD.
  template <bool TWO, bool K256, class Hook>
  __device__ __forceinline__ void chains(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane, Hook&& hook) {
    const bool h0 = lane < n, h1 = TWO && lane + 32 < n;
    const uint8_t* r0 = a.codes + size_t(h0 ? cid[lane] : cid[0]) * a.codes_pitch;
    const uint8_t* r1 = a.codes + size_t(h1 ? cid[lane + 32] : cid[0]) * a.codes_pitch;
    const uint32_t nch = (a.pqM + 15) >> 4;
    const uint32_t K = K256 ? 256u : a.pqK;
    float d0 = 0.0f, d1 = 0.0f;
    for (uint32_t cb = 0; cb < nch; cb += NCH) {
      uint4 v0[NCH], v1[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const bool in = cb + c < nch;  // warp-uniform
        v0[c] = in ? ldg_u4_stream(r0 + (cb + c) * 16) : make_uint4(0, 0, 0, 0);
        if (TWO) v1[c] = in ? ldg_u4_stream(r1 + (cb + c) * 16) : make_uint4(0, 0, 0, 0);
      }
      if (cb == 0) hook();  // code rows in flight: speculative prefetches for the next hop ride along
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const uint32_t w0[4] = {v0[c].x, v0[c].y, v0[c].z, v0[c].w};
        const uint32_t w1[4] = {TWO ? v1[c].x : 0u, TWO ? v1[c].y : 0u, TWO ? v1[c].z : 0u, TWO ? v1[c].w : 0u};
        const uint32_t ibase = (cb + c) * 16;
        if (ibase + 16 <= a.pqM) {
          const float* t = table + ibase * K;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const uint32_t c0 = (w0[j >> 2] >> (8 * (j & 3))) & 0xFFu;
            d0 = __fadd_rn(d0, t[j * K + c0]);
            if (TWO) {
              const uint32_t c1 = (w1[j >> 2] >> (8 * (j & 3))) & 0xFFu;
              d1 = __fadd_rn(d1, t[j * K + c1]);
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const uint32_t i = ibase + j;
            if (i < a.pqM) {
              const uint32_t c0 = (w0[j >> 2] >> (8 * (j & 3))) & 0xFFu;
              d0 = __fadd_rn(d0, table[i * K + c0]);
              if (TWO) {
                const uint32_t c1 = (w1[j >> 2] >> (8 * (j & 3))) & 0xFFu;
                d1 = __fadd_rn(d1, table[i * K + c1]);
              }
            }
          }
        }
      }
    }
    if (h0) cdist[lane] = d0;
    if (h1) cdist[lane + 32] = d1;
    __syncwarp();
  }
  template <class Hook>
  __device__ __forceinline__ void eval(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane, Hook&& hook) {
    if (a.pqK == 256) {
      if (n > 32) chains<true, true>(a, cid, cdist, n, lane, hook);
      else chains<false, true>(a, cid, cdist, n, lane, hook);
    } else {
      if (n > 32) chains<true, false>(a, cid, cdist, n, lane, hook);
      else chains<false, false>(a, cid, cdist, n, lane, hook);
    }
  }
};

// PQ codes without a materialised table. The reference fills dists[i*K+j] = distFn(x_i, centroid_ij)
// for all M*K entries of a query and then sums M lookups per point (product.go:255-277). An entry
// depends only on (query, i, j): computing it where it is needed — the same sequential FMA chain
// over the sub-vector the table kernel runs (short_dist_thread), so the same float — removes the
// per-query table (96 KB at C4) from shared memory, where it capped residency at two query-warps
// per SM and left the search latency-bound at 3 % warp occupancy (profiles/r02_k3_*). The
// codebook (M*K*sub floats, 786 KB at C4) is shared by every query and stays L2-resident; a
// lookup becomes one 32-byte sector read + sub FMAs, and twelve query-warps per SM hide it.
// One lane owns a candidate (two when the hop staged more than 32); the M terms are summed in
// sub-vector order in f32 (product.go:271-275). SUB = sub-vector length (4, 8 or 16 floats).
template <int METRIC, int SUB>
struct AdcEvalFly {
  static constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
  static constexpr int V4 = SUB / 4;
  const float* qs;  // the query in shared memory
  // one centroid (SUB floats, SUB*4-byte aligned): 256-bit loads where the record allows — the
  // lookups are scattered, so the L1 pays one wavefront per lane per load instruction
  __device__ __forceinline__ void load_entry(const float* p, float4 (&c)[V4]) const {
    if (V4 == 1) {
      c[0] = ldg_f4(p);
    } else {
#pragma unroll
      for (int v = 0; v < V4; v += 2) ldg_f8(p + 4 * v, c[v], c[(v + 1) < V4 ? v + 1 : v]);
    }
  }
  __device__ __forceinline__ float term(const float4 (&c)[V4], uint32_t i) const {
    float t = 0.0f;
#pragma unroll
    for (int v = 0; v < V4; ++v) {
      const float4 q = *reinterpret_cast<const float4*>(qs + i * SUB + 4 * v);
      t = tail_accum<L2>(q.x, c[v].x, t);
      t = tail_accum<L2>(q.y, c[v].y, t);
      t = tail_accum<L2>(q.z, c[v].z, t);
      t = tail_accum<L2>(q.w, c[v].w, t);
    }
    return metric_epilogue<METRIC>(t);
  }
  // LPC lanes share a candidate (hops that stage few candidates — the usual case on a PQ graph,
  // 6-12 of 64 neighbours are new — would otherwise leave most lanes idle through the M-term
  // loop): within each 16-byte chunk of the code row lane s of the group computes the terms of
  // code words s*WPL .. s*WPL+WPL-1 (4 sub-vectors per word), then the 16 terms are added in
  // sub-vector order through shuffles, so the sum is the same sequential f32 chain. TWO (LPC = 1
  // only): a second chain for adjacency slot lane + 32.
  template <int LPC, bool TWO, class Hook>
  __device__ __forceinline__ void chains(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane, Hook&& hook) {
    constexpr int WPL = 4 / LPC;  // code words per lane per chunk
    const int s = lane % LPC, c = lane / LPC;
    const bool h0 = c < n, h1 = TWO && lane + 32 < n;
    const uint8_t* r0 = a.codes + size_t(h0 ? cid[c] : cid[0]) * a.codes_pitch + s * WPL * 4;
    const uint8_t* r1 = a.codes + size_t(h1 ? cid[lane + 32] : cid[0]) * a.codes_pitch;
    const uint32_t nch = (a.pqM + 15) >> 4;
    const uint32_t K = a.pqK;
    float d0 = 0.0f, d1 = 0.0f;
    auto load_words = [&](const uint8_t* p, uint32_t (&w)[WPL]) {
      if (WPL == 4) {
        const uint4 v = ldg_u4_stream(p);
        w[0] = v.x; w[WPL > 1 ? 1 : 0] = v.y; w[WPL > 2 ? 2 : 0] = v.z; w[WPL > 3 ? 3 : 0] = v.w;
      } else if (WPL == 2) {
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
        w[0] = v.x; w[WPL > 1 ? 1 : 0] = v.y;
      } else {
        w[0] = __ldg(reinterpret_cast<const uint32_t*>(p));
      }
    };
    uint32_t nx0[WPL], nx1[WPL];
    load_words(r0, nx0);
    if (TWO) load_words(r1, nx1);
    hook();  // first code chunks in flight: speculative prefetches for the next hop ride along
    for (uint32_t cb = 0; cb < nch; ++cb) {
      uint32_t w0[WPL], w1[WPL];
#pragma unroll
      for (int k = 0; k < WPL; ++k) { w0[k] = nx0[k]; w1[k] = TWO ? nx1[k] : 0u; }
      if (cb + 1 < nch) {  // next 16 code bytes while this chunk's centroids are fetched
        load_words(r0 + (cb + 1) * 16, nx0);
        if (TWO) load_words(r1 + (cb + 1) * 16, nx1);
      }
      const uint32_t ibase = cb * 16 + s * WPL * 4;
      float t0[WPL * 4], t1[WPL * 4];
#pragma unroll
      for (int k = 0; k < WPL; ++k) {
        // the lane's word k covers sub-vectors ibase + 4k .. +3; past M (only when M % 16 != 0, LPC = 1)
        // the word is skipped warp-uniformly
        if (LPC == 1 && ibase + 4 * k >= a.pqM) {
#pragma unroll
          for (int j = 0; j < 4; ++j) { t0[4 * k + j] = 0.0f; t1[4 * k + j] = 0.0f; }
          continue;
        }
        float4 c0[4][V4], c1[4][V4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t i = ibase + 4 * k + j;
          const uint32_t k0 = (w0[k] >> (8 * j)) & 0xFFu;
          load_entry(a.pq_cent + (size_t(i) * K + k0) * SUB, c0[j]);
          if (TWO) {
            const uint32_t k1 = (w1[k] >> (8 * j)) & 0xFFu;
            load_entry(a.pq_cent + (size_t(i) * K + k1) * SUB, c1[j]);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t i = ibase + 4 * k + j;
          t0[4 * k + j] = term(c0[j], i);
          if (TWO) t1[4 * k + j] = term(c1[j], i);
        }
      }
      // the chunk's terms in sub-vector order: word x of the chunk lives in lane x / WPL of the group
      const uint32_t left = a.pqM - cb * 16;  // sub-vectors of this chunk that exist (>= 16 except in the last)
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        if (LPC == 1 && uint32_t(4 * x) >= left) break;  // warp-uniform
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float v0 = t0[4 * (x % WPL) + j];
          if (LPC > 1) v0 = __shfl_sync(SDB_FULL, v0, (lane - s) + x / WPL);
          d0 = __fadd_rn(d0, v0);
          if (TWO) d1 = __fadd_rn(d1, t1[4 * x + j]);
        }
      }
    }
    if (h0 && s == 0) cdist[c] = d0;
    if (h1) cdist[lane + 32] = d1;
    __syncwarp();
  }
  template <class Hook>
  __device__ __forceinline__ void eval(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane, Hook&& hook) {
    const bool whole = (a.pqM & 15u) == 0;  // groups need whole 16-sub-vector chunks
    if (n > 32) chains<1, true>(a, cid, cdist, n, lane, hook);
    else if (n > 16 || !whole) chains<1, false>(a, cid, cdist, n, lane, hook);
    else if (n > 8) chains<2, false>(a, cid, cdist, n, lane, hook);
    else chains<4, false>(a, cid, cdist, n, lane, hook);
  }
};

// dim-2 haversine rows (latitude, longitude in degrees; distance.go:33-43). A row is 8 bytes of a
// 16-byte pitch, so the 8-lane-per-line layout of the f32 evaluators would leave 7 of 8 lanes idle:
// here one lane owns a candidate (adjacency slot c in lane c % 32, a second one for c >= 32), both
// rows are loaded before either distance is computed, and the query's terms (radians, cos(lat)) are
// computed once per query into registers. haversine_from is haversine_thread's body with the query
// as x, so every distance is the float sdb_index_query_dists and the flat scan produce.
struct GeoEval {
  HaversineX q;
  __device__ __forceinline__ void load_query(const float* qg) { q = haversine_terms(__ldg(qg), __ldg(qg + 1)); }
  template <class Hook>
  __device__ __forceinline__ void eval(const SearchArgs& a, const uint32_t* cid, float* cdist, int n, int lane, Hook&& hook) {
    const bool h0 = lane < n, h1 = lane + 32 < n;
    float2 r0 = make_float2(0.f, 0.f), r1 = make_float2(0.f, 0.f);
    if (h0) r0 = __ldg(reinterpret_cast<const float2*>(a.vec + size_t(cid[lane]) * a.vec_pitch));
    if (h1) r1 = __ldg(reinterpret_cast<const float2*>(a.vec + size_t(cid[lane + 32]) * a.vec_pitch));
    hook();
    if (h0) cdist[lane] = haversine_from(q, r0.x, r0.y);
    if (h1) cdist[lane + 32] = haversine_from(q, r1.x, r1.y);
    __syncwarp();
  }
};

enum EvalKind : int { EVAL_FLOAT_FIXED = 0, EVAL_FLOAT_GENERIC = 1, EVAL_BITS = 2, EVAL_ADC = 3, EVAL_ADC_SMEM = 4, EVAL_ADC_FLY = 5, EVAL_GEO = 6 };

// ---- shared-memory layout per query-warp ------------------------------------------------
template <class VT, bool FILTER>
__host__ __device__ constexpr size_t warp_smem_bytes(uint32_t qfloats, uint32_t qwords, uint32_t vt_slots,
                                                     uint32_t table_floats = 0) {
  return ((VT::bytes(vt_slots) + 15) / 16) * 16 + LIST_SLOTS * 8 + (FILTER ? LIST_SLOTS * 8 : 0) + CAND_SLOTS * 8 +
         ((size_t(qfloats) * 4 + 15) / 16) * 16 + ((size_t(qwords) * 8 + 15) / 16) * 16 +
         (table_floats ? 16 + ((size_t(table_floats) * 4 + 15) / 16) * 16 : 0);
}

// ---- the kernel ---------------------------------------------------------------------
// One warp per CTA, one query per warp at a time; MINB = CTAs per SM the register budget
// must allow (launch bounds).
// SETS: FloatEvalFixed pipeline depth; MERGE_MIN > 0: use the batch form of AddWithLimit
// (CandList::merge) when at least that many candidates survive.
// XTRA: the start node has edges beyond R (a.start_extra) — compiled in only when it does.
// REQ: per-query L / k / gather limit from a.req (request batches); false = the launch-wide values,
// compiled without a trace of the per-query path.
template <int KIND, int METRIC, int TRIPS, int SETS, int MERGE_MIN, class VT, bool FILTER, bool RETRY, int MINB,
          bool XTRA, bool PF, bool REQ>
__global__ void __launch_bounds__(32, MINB) beam_search_kernel(SearchArgs a, uint32_t qfloats, uint32_t qwords) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  unsigned char* base = smem_raw;
  VT vt;
  vt.init(base, a.rows, a.vt_slots, a.retry_bitmap, a.bitmap_words);
  base += ((VT::bytes(a.vt_slots) + 15) / 16) * 16;
  CandList list;
  list.id = reinterpret_cast<uint32_t*>(base);
  list.dist = reinterpret_cast<float*>(base + LIST_SLOTS * 4);
  base += LIST_SLOTS * 8;
  CandList res;  // filter mode: k-bounded result set (search.go:33-35)
  res.id = list.id;
  res.dist = list.dist;
  if (FILTER) {
    res.id = reinterpret_cast<uint32_t*>(base);
    res.dist = reinterpret_cast<float*>(base + LIST_SLOTS * 4);
    base += LIST_SLOTS * 8;
  }
  uint32_t* cid = reinterpret_cast<uint32_t*>(base);
  float* cdist = reinterpret_cast<float*>(base + CAND_SLOTS * 4);
  base += CAND_SLOTS * 8;
  float* qs = reinterpret_cast<float*>(base);
  base += ((size_t(qfloats) * 4 + 15) / 16) * 16;
  uint64_t* qbits = reinterpret_cast<uint64_t*>(base);
  base += ((size_t(qwords) * 8 + 15) / 16) * 16;
  uint64_t* tbar = reinterpret_cast<uint64_t*>(base);  // EVAL_ADC_SMEM: mbarrier + the query's ADC table
  float* tab = reinterpret_cast<float*>(base + 16);
  uint32_t tphase = 0;
  if (KIND == EVAL_ADC_SMEM) {
    if (lane == 0) mbar_init(tbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();
  }
  const uint32_t lt = (1u << lane) - 1;
  // speculative L2 prefetch of the runner-up's rows: the small-row evaluators only (see the hop loop)
  constexpr bool PFROWS = PF && (KIND == EVAL_BITS || KIND == EVAL_ADC_SMEM || KIND == EVAL_ADC || KIND == EVAL_ADC_FLY);

  for (;;) {
    uint32_t qi = 0;
    if (lane == 0) {
      qi = atomicAdd(a.work_counter, 1u);
      if (RETRY) qi = qi < *a.retry_count ? a.retry_list[qi] : 0xFFFFFFFFu;
      else if (a.qmap) qi = qi < a.n_work ? a.qmap[qi] : 0xFFFFFFFFu;
    }
    qi = __shfl_sync(SDB_FULL, qi, 0);
    if (qi >= a.B) break;

    // ---- per-query setup
    vt.clear(lane);
    if (KIND != EVAL_ADC && KIND != EVAL_ADC_SMEM && KIND != EVAL_BITS && KIND != EVAL_GEO) {
      const float* qg = a.queries + size_t(qi) * a.dim;
      for (uint32_t i = lane; i < qfloats; i += 32) qs[i] = i < a.dim ? __ldg(qg + i) : 0.0f;
    }
    __syncwarp();
    constexpr bool FIXED = (KIND == EVAL_FLOAT_FIXED);
    FloatEvalFixed<METRIC, (FIXED ? TRIPS : 1), (FIXED ? SETS : 1)> ev_fixed;
    FloatEvalGeneric<METRIC> ev_gen;
    constexpr bool BITS = (KIND == EVAL_BITS);
    BitEval<(BITS ? METRIC : METRIC_HAMMING), (BITS ? TRIPS : 1), (BITS ? SETS : 1)> ev_bits;
    AdcEval ev_adc;
    AdcEvalSmem<(KIND == EVAL_ADC_SMEM ? TRIPS : 1)> ev_adcs;
    constexpr bool FLY = (KIND == EVAL_ADC_FLY);
    AdcEvalFly<(FLY && METRIC == METRIC_EUCLIDEAN ? METRIC_EUCLIDEAN : METRIC_DOT), (FLY ? TRIPS : 4)> ev_fly;
    if (FLY) ev_fly.qs = qs;
    GeoEval ev_geo;
    if (KIND == EVAL_GEO) ev_geo.load_query(a.queries + size_t(qi) * a.dim);
    if (KIND == EVAL_ADC_SMEM)
      ev_adcs.load_table(tab, a.adc + size_t(qi) * a.pqM * a.pqK, a.pqM * a.pqK, tbar, tphase, lane);
    if (KIND == EVAL_FLOAT_FIXED) ev_fixed.load_query(qs, a.queries + size_t(qi) * a.dim, lane);
    if (KIND == EVAL_FLOAT_GENERIC) ev_gen.load_query(qs, lane);
    if (KIND == EVAL_BITS) ev_bits.encode_query(a, a.queries + size_t(qi) * a.dim, qbits, lane);
    if (KIND == EVAL_ADC) ev_adc.table = a.adc + size_t(qi) * a.pqM * a.pqK;
    auto no_hook = []() {};
    auto evaluate_h = [&](int n, auto&& hook) {
      if (KIND == EVAL_FLOAT_FIXED) ev_fixed.eval(a, cid, cdist, n, lane);
      if (KIND == EVAL_FLOAT_GENERIC) ev_gen.eval(a, cid, cdist, n, lane);
      if (KIND == EVAL_BITS) ev_bits.eval(a, cid, cdist, n, lane, hook);
      if (KIND == EVAL_ADC) ev_adc.eval(a, cid, cdist, n, lane, hook);
      if (KIND == EVAL_ADC_SMEM) ev_adcs.eval(a, cid, cdist, n, lane, hook);
      if (KIND == EVAL_ADC_FLY) ev_fly.eval(a, cid, cdist, n, lane, hook);
      if (KIND == EVAL_GEO) ev_geo.eval(a, cid, cdist, n, lane, hook);
    };
    auto evaluate = [&](int n) { evaluate_h(n, no_hook); };

    list.len = 0;
    list.cap = int(REQ ? __ldg(&a.req[qi].x) : a.L);
    list.nan_seen = false;
    res.len = 0;
    res.cap = int(REQ ? __ldg(&a.req[qi].y) : a.k);
    res.nan_seen = false;
    uint32_t hops = 0, ndist = 0, nvisited = 0;
    bool overflow = false;

    // AddWithLimit of the staged candidates cid/cdist[0..n) into `dst`, sequentially in
    // order (distset.go:166-200 after the visited test and the distance evaluation).
    auto add_with_limit = [&](CandList& dst, int n) {
      float d0 = lane < n ? cdist[lane] : 0.0f;
      float d1 = lane + 32 < n ? cdist[lane + 32] : 0.0f;
      int next = 0;
      for (;;) {
        const bool full = dst.len == dst.cap;
        const float worst = full ? dst.dist[dst.cap - 1] : 0.0f;
        bool e0 = lane >= next && lane < n && !(full && d0 > worst);
        bool e1 = lane + 32 >= next && lane + 32 < n && !(full && d1 > worst);
        uint32_t m0 = __ballot_sync(SDB_FULL, e0), m1 = __ballot_sync(SDB_FULL, e1);
        int c;
        if (m0) c = __ffs(m0) - 1;
        else if (m1) c = 32 + __ffs(m1) - 1;
        else break;
        float dc = __shfl_sync(SDB_FULL, c < 32 ? d0 : d1, c & 31);
        dst.insert(cid[c], dc, lane);
        next = c + 1;
      }
    };

    // stage ids i0/i1 (adjacency order c = lane, lane+32) that pass the visited
    // test-and-set into cid[]; returns how many
    auto visit_and_stage = [&](uint32_t i0, bool a0, uint32_t i1, bool a1) -> int {
      bool new0, new1;
      vt.test_and_set2(i0, a0, i1, a1, new0, new1, lane);
      uint32_t b0 = __ballot_sync(SDB_FULL, new0), b1 = __ballot_sync(SDB_FULL, new1);
      const int t0 = __popc(b0);
      if (new0) cid[__popc(b0 & lt)] = i0;
      if (new1) cid[t0 + __popc(b1 & lt)] = i1;
      __syncwarp();
      return t0 + __popc(b1);
    };

    // this query's filter: ascending ids fl[0..fn), the first min(fn, L) of them are the seeds (L of
    // this query: list.cap)
    const uint32_t* fl = nullptr;
    uint32_t fn = 0;
    if (FILTER) {
      const uint32_t f = a.query_filter ? uint32_t(__ldg(a.query_filter + qi)) : 0u;
      const uint32_t fb = __ldg(a.filter_off + f);
      fl = a.filter_ids + fb;
      fn = __ldg(a.filter_off + f + 1) - fb;
    }
    if (FILTER) {
      // searchSet.Add(filterPoints...) (plain append, search.go:49) and
      // resultSet.AddWithLimit(filterPoints...) (search.go:50)
      const int nf = int(min(fn, REQ ? uint32_t(list.cap) : a.L));
      for (int b0 = 0; b0 < nf; b0 += CAND_SLOTS) {
        const int n = min(CAND_SLOTS, nf - b0);
        uint32_t i0 = lane < n ? __ldg(fl + b0 + lane) : 0;
        uint32_t i1 = lane + 32 < n ? __ldg(fl + b0 + lane + 32) : 0;
        const int nn = visit_and_stage(i0, lane < n, i1, lane + 32 < n);
        nvisited += nn;
        ndist += nn;
        evaluate(nn);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          int c = lane + 32 * j;
          if (c < nn) {
            list.id[list.len + c] = cid[c];
            list.dist[list.len + c] = cdist[c];
          }
        }
        list.len += nn;
        __syncwarp();
        add_with_limit(res, nn);  // resultSet has its own visited set; seeds are unique
      }
    }

    // searchSet.AddWithLimit(startNode) (search.go:57-61)
    if (visit_and_stage(START_ID, lane == 0, 0, false) > 0) {
      ++nvisited;
      ++ndist;
      evaluate(1);
      add_with_limit(list, 1);
    }

    // a table that cannot hold this store's ids at all (span beyond 16 bits) refuses every probe:
    // the query goes to the RETRY launch before it has searched anything
    if (vt.failed) overflow = true;
    // main loop (search.go:65-98). pf_*: adjacency row of the runner-up candidate, fetched
    // one hop early; used if that candidate is indeed expanded next.
    uint32_t pf_id = INVALID_ID, pf_n0 = INVALID_ID, pf_n1 = INVALID_ID;
    for (; !overflow;) {
      const int lim = min(list.len, REQ ? list.cap : int(a.L));
      int pos = -1, pos2 = -1, pos3 = -1;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        int p = lane + 32 * j;
        bool un = (p < lim) && !(list.id[p] & EXPANDED_FLAG);
        uint32_t b = __ballot_sync(SDB_FULL, un);
        if (b && pos < 0) {
          pos = 32 * j + __ffs(b) - 1;
          b &= b - 1;
        }
        if (b && pos >= 0 && pos2 < 0) {
          pos2 = 32 * j + __ffs(b) - 1;
          b &= b - 1;
        }
        if (PFROWS && b && pos2 >= 0 && pos3 < 0) pos3 = 32 * j + __ffs(b) - 1;
      }
      if (pos < 0) break;
      const uint32_t e = list.id[pos];
      const float edist = list.dist[pos];
      const uint32_t e2 = pos2 >= 0 ? list.id[pos2] : INVALID_ID;
      const uint32_t e3 = (PFROWS && pos3 >= 0) ? list.id[pos3] : INVALID_ID;
      __syncwarp();
      if (lane == 0) list.id[pos] = e | EXPANDED_FLAG;
      if (a.vis_ids != nullptr && lane == 0) {
        if (hops < a.vis_cap) {
          a.vis_ids[size_t(qi) * a.vis_cap + hops] = e;
          a.vis_dists[size_t(qi) * a.vis_cap + hops] = edist;
        }
      }
      ++hops;
      // neighbours, adjacency order c = lane, lane+32
      uint32_t n0, n1;
      if (e == pf_id) {
        n0 = pf_n0;
        n1 = pf_n1;
      } else {
        const uint32_t* arow = a.adj + size_t(e) * a.R;
        n0 = lane < int(a.R) ? __ldg(arow + lane) : INVALID_ID;
        n1 = lane + 32 < int(a.R) ? __ldg(arow + lane + 32) : INVALID_ID;
      }
      pf_id = e2;
      if (e2 != INVALID_ID) {
        const uint32_t* prow = a.adj + size_t(e2) * a.R;
        pf_n0 = lane < int(a.R) ? __ldg(prow + lane) : INVALID_ID;
        pf_n1 = lane + 32 < int(a.R) ? __ldg(prow + lane + 32) : INVALID_ID;
      }
      // Small rows (bit rows, PQ codes) leave this kernel latency-bound on one warp's dependent
      // chain adjacency row -> visited test -> row gather, not HBM-bound (profiles/r01_k2_*,
      // r02_k3_*). Speculation two levels deep takes DRAM latency off that chain:
      //  * the third unexpanded candidate's adjacency row is pulled into L2 now, so that when it is
      //    the runner-up next hop its register prefetch above is an L2 hit;
      //  * once this hop's own rows are in flight (the evaluators call the hook), the rows of the
      //    runner-up's not-yet-visited neighbours are pulled into L2: if the runner-up is expanded
      //    next — the common case once the list has settled — its gather hits L2.
      // Wrong guesses cost bandwidth this kernel has to spare (< 20 % of HBM in use), never results.
      if (PFROWS && e3 != INVALID_ID && lane < int((a.R * 4 + 127) / 128)) prefetch_l2(a.adj + size_t(e3) * a.R + lane * 32);
      auto pf_rows = [&]() {
        if (!PFROWS || pf_id == INVALID_ID) return;
        const uint32_t ids2[2] = {pf_n0, pf_n1};
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const uint32_t id = ids2[j];
          if (id == INVALID_ID || !vt.maybe_new(id)) continue;
          const unsigned char* row = (KIND == EVAL_BITS) ? reinterpret_cast<const unsigned char*>(a.bits + size_t(id) * a.bits_pitch)
                                                         : a.codes + size_t(id) * a.codes_pitch;
          const uint32_t bytes = (KIND == EVAL_BITS) ? a.bits_pitch * 8 : a.codes_pitch;
          const uint32_t first = uint32_t(reinterpret_cast<uintptr_t>(row) & 127u);
          for (uint32_t o = 0; o < first + bytes; o += 128) prefetch_l2(row - first + o);
        }
      };
      // searchSet.AddWithLimit(neighbours...) (search.go:90), 64 adjacency slots at a time: the
      // row itself, then — for the start node only — its edges beyond R (orphans re-attached
      // after deletes, prune.go:137-151; normally none). One copy of the hop body.
      for (uint32_t x0 = 0;; x0 += CAND_SLOTS) {
        const int nnew = visit_and_stage(n0, n0 != INVALID_ID, n1, n1 != INVALID_ID);
        nvisited += nnew;
        ndist += nnew;
        if (nvisited > vt.limit() || vt.failed) { overflow = true; break; }
        if (nnew > 0) {
          if (x0 == 0) evaluate_h(nnew, pf_rows);
          else evaluate(nnew);
          // integer-valued / coarse distances; geo: points at one address (exact duplicates) tie exactly
          constexpr bool TIEFIX = (KIND == EVAL_BITS || KIND == EVAL_ADC || KIND == EVAL_ADC_SMEM || KIND == EVAL_ADC_FLY || KIND == EVAL_GEO);
          if (MERGE_MIN == 0 || !list.template merge<TIEFIX>(cid, cdist, nnew, lane, lt, MERGE_MIN)) add_with_limit(list, nnew);
        }
        if (!XTRA || e != START_ID || x0 >= a.n_start_extra) break;
        const uint32_t j0 = x0 + lane, j1 = x0 + 32 + lane;
        n0 = j0 < a.n_start_extra ? __ldg(a.start_extra + j0) : INVALID_ID;
        n1 = j1 < a.n_start_extra ? __ldg(a.start_extra + j1) : INVALID_ID;
      }
      if (overflow) break;
      if (FILTER) {
        // resultSet.AddWithLimit(distElem.Point) if the expanded node passes the filter
        // (search.go:93-95). resultSet dedupes with its own visited set, which holds the
        // seeds (search.go:50) and every node added here; a node is expanded at most once.
        // filter.Contains(node.Id): the shared filter's dense bitmask when there is one, else a
        // 32-way search of the query's ascending id list (4 rounds for a million ids)
        bool in_filter;
        if (a.filter_bits != nullptr) {
          in_filter = (__ldg(a.filter_bits + (e >> 5)) >> (e & 31)) & 1u;
        } else {
          uint32_t lo = 0, hi = fn;  // invariant: if e is in the list its index is in [lo, hi)
          while (hi - lo > 32) {
            const uint32_t stride = (hi - lo + 31) / 32;
            const uint32_t at = lo + uint32_t(lane) * stride;
            const bool le = at < hi && __ldg(fl + at) <= e;
            const uint32_t b = __ballot_sync(SDB_FULL, le);
            if (b == 0) { hi = lo; break; }  // e is below the first pivot
            const uint32_t c = 31 - __clz(b);  // pivots ascend: the set lanes form a prefix
            lo = lo + c * stride;
            hi = min(lo + stride, hi);
          }
          const bool eq = lo + lane < hi && __ldg(fl + lo + lane) == e;
          in_filter = __any_sync(SDB_FULL, eq);
        }
        if (in_filter) {
          // the seeds are already in resultSet (search.go:50): ascending list => e is a seed
          // iff it is not above the last seed
          const uint32_t ns = min(fn, REQ ? uint32_t(list.cap) : a.L);
          const bool seeded = ns > 0 && e <= __ldg(fl + ns - 1);
          if (!seeded) {
            if (lane == 0) { cid[0] = e; cdist[0] = edist; }
            __syncwarp();
            add_with_limit(res, 1);
          }
        }
      }
    }

    // ---- results (vamana.go:285-307): drop STARTID, first k items
    CandList& out = FILTER ? res : list;
    if (overflow) {
      if (lane == 0) {
        a.out_counts[qi] = COUNT_OVERFLOW;
        a.out_hops[qi] = hops;
        a.out_ndist[qi] = ndist;
        if (!RETRY) a.retry_list[atomicAdd(a.retry_count, 1u)] = qi;
      }
    } else {
      // this query's k; a.k is the row stride
      const int qk = REQ ? res.cap : int(a.k);
      int written = 0;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        int p = lane + 32 * j;
        uint32_t nid = p < out.len ? (out.id[p] & ID_MASK) : START_ID;
        bool keep = (p < out.len) && (nid != START_ID);
        uint32_t b = __ballot_sync(SDB_FULL, keep);
        int r = written + __popc(b & lt);
        if (keep && r < qk) {
          const float dd = out.dist[p];
          a.out_ids[size_t(qi) * a.k + r] = uint64_t(nid);
          a.out_dists[size_t(qi) * a.k + r] = dd;
          if (a.pg.n) {
            const size_t o = (size_t(a.pg.shard) * a.B + qi) * a.k + r;
            for (uint32_t s = 0; s < a.pg.n; ++s) {
              a.pg.ids[s][o] = uint64_t(nid) | a.pg.tag;
              a.pg.dists[s][o] = dd;
            }
          }
        }
        written += __popc(b);
      }
      int cnt = min(written, qk);
      for (int r = cnt + lane; r < int(a.k); r += 32) {
        a.out_ids[size_t(qi) * a.k + r] = 0;
        a.out_dists[size_t(qi) * a.k + r] = __int_as_float(0x7f800000);
        if (a.pg.n) {
          const size_t o = (size_t(a.pg.shard) * a.B + qi) * a.k + r;
          for (uint32_t s = 0; s < a.pg.n; ++s) {
            a.pg.ids[s][o] = 0;
            a.pg.dists[s][o] = __int_as_float(0x7f800000);
          }
        }
      }
      if (a.pg.n && lane < int(a.pg.n)) {
        const int plim = REQ ? int(__ldg(&a.req[qi].z)) : int(a.pg.limit);
        a.pg.counts[lane][size_t(a.pg.shard) * a.B + qi] = uint32_t(min(cnt, plim));
      }
      if (lane == 0) {
        a.out_counts[qi] = uint32_t(cnt);
        a.out_hops[qi] = hops;
        a.out_ndist[qi] = ndist;
        if (a.vis_len) a.vis_len[qi] = hops;
      }
    }
    __syncwarp();
  }
}

}  // namespace sdb
