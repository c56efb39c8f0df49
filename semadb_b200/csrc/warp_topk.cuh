// warp_topk.cuh — a k-slot list sorted by (distance asc, id asc) held in the registers of one warp.
//
// Slot p = lane + 32 j, NS slots per lane (1 for k <= 32, 3 up to k = 96). An insertion is NS
// ballots' worth of compares and two shuffles per slot row, no shared-memory round trip. A
// candidate that does not beat the current k-th (kept in a uniform register pair) is dropped by
// the lane that holds it. Because (distance, id) is a total order over distinct ids, the list
// after any sequence of offers is the top-k of everything offered, whatever the order: the
// reference's flat scan (flat.go:99-119, ascending ids) keeps the same list.
// Every member function is warp-synchronous: all 32 lanes call it.
#pragma once
#include "common.cuh"

namespace sdb {

template <int NS>
struct WarpTopK {
  // The list itself is locals of the calling kernel (declared by SDB_WARP_TOPK_STATE): a struct that
  // owned the arrays would live in local memory at NS = 3. This view holds references to them, in
  // the order of their first use in insert(), which keeps rescore_warp_kernel's code as it was when
  // insert / offer were lambdas in its body.
  const int& lane;
  uint32_t& len;
  float (&kd)[NS];
  uint32_t (&ki)[NS];
  const uint32_t& k;
  const int& wj;
  float& wd;  // the k-th entry once the list is full (uniform)
  const int& wl;
  uint32_t& wi;

  // offer (d, id), held by every lane, to the sorted list
  __device__ __forceinline__ void insert(float d, uint32_t id) {
    uint32_t pos = 0;
#pragma unroll
    for (int j = 0; j < NS; ++j) {
      const uint32_t p = lane + 32 * j;
      const bool before = p < len && (kd[j] < d || (kd[j] == d && ki[j] < id));
      pos += __popc(__ballot_sync(SDB_FULL, before));
    }
    if (pos >= k) return;
#pragma unroll
    for (int j = NS - 1; j >= 0; --j) {  // slots >= pos move up by one; the rows below are still unmodified
      float pd = __shfl_up_sync(SDB_FULL, kd[j], 1);
      uint32_t pi = __shfl_up_sync(SDB_FULL, ki[j], 1);
      if (j > 0) {
        const float cd = __shfl_sync(SDB_FULL, kd[j > 0 ? j - 1 : 0], 31);
        const uint32_t ci = __shfl_sync(SDB_FULL, ki[j > 0 ? j - 1 : 0], 31);
        if (lane == 0) { pd = cd; pi = ci; }
      }
      const uint32_t p = lane + 32 * j;
      if (p > pos) { kd[j] = pd; ki[j] = pi; }
      else if (p == pos) { kd[j] = d; ki[j] = id; }
    }
    if (len < k) ++len;
    if (len == k) {
      float sd = kd[0];
      uint32_t si = ki[0];
#pragma unroll
      for (int j = 1; j < NS; ++j)
        if (j == wj) { sd = kd[j]; si = ki[j]; }
      wd = __shfl_sync(SDB_FULL, sd, wl);
      wi = __shfl_sync(SDB_FULL, si, wl);
    }
  }

  // the lanes that hold a fresh (d, id) (have = true) offer it if it can enter the list
  __device__ __forceinline__ void offer(float d, uint32_t id, bool have) {
    const bool want = have && (len < k || d < wd || (d == wd && id < wi));
    uint32_t m = __ballot_sync(SDB_FULL, want);
    while (m) {
      const int src = __ffs(m) - 1;
      m &= m - 1;
      insert(__shfl_sync(SDB_FULL, d, src), __shfl_sync(SDB_FULL, id, src));
    }
  }
};

}  // namespace sdb

// The registers of an empty list for k results, NS slots per lane; `name` is then a WarpTopK over them.
#define SDB_WARP_TOPK_STATE(name, NS, k, lane)                         \
  float name##_kd[NS];                                                 \
  uint32_t name##_ki[NS];                                              \
  _Pragma("unroll") for (int j_ = 0; j_ < NS; ++j_) {                  \
    name##_kd[j_] = 0.0f;                                              \
    name##_ki[j_] = 0u;                                                \
  }                                                                    \
  uint32_t name##_len = 0;                                             \
  float name##_wd = 0.0f;                                              \
  uint32_t name##_wi = 0u;                                             \
  const int name##_wj = int((k) - 1) >> 5, name##_wl = int((k) - 1) & 31; \
  ::sdb::WarpTopK<NS> name{lane, name##_len, name##_kd, name##_ki, k, name##_wj, name##_wd, name##_wl, name##_wi}
