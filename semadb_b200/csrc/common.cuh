// common.cuh — shared device helpers for the semadb_b200 kernels (sm_100a).
//
// Float distances reproduce the summation order of the reference's AVX2/FMA kernels
// (distance/asm/dot.s:16-54, distance/asm/euclidean.s:20-64) bit for bit:
//   element i of a 32-float trip goes to partial sum (i%32) via one fused multiply-add
//   per trip; the <32 tail is a sequential scalar FMA chain; the reduction is
//   v[l] = ((a0[l]+a1[l])+a2[l])+a3[l], w[l] = v[l]+v[l+4], w[0] += tail,
//   result = (w0+w1)+(w2+w3).
// An 8-lane group owns one row: lane g loads float4 at element 32t+4g (one 128-byte
// line per trip per group, fully coalesced) and so holds partial sums 4g..4g+3.
// Compile with -fmad=false: every FMA is written explicitly.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sdb {

constexpr int METRIC_EUCLIDEAN = 0;
constexpr int METRIC_DOT = 1;
constexpr int METRIC_COSINE = 2;
constexpr int METRIC_HAMMING = 3;
constexpr int METRIC_JACCARD = 4;
constexpr int METRIC_HAVERSINE = 5;

constexpr uint32_t INVALID_ID = 0xFFFFFFFFu;
constexpr uint32_t START_ID = 1u;  // vamana.go:28

#define SDB_FULL 0xFFFFFFFFu

__device__ __forceinline__ float4 ldg_f4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
// streaming 128-bit load: vector rows have no reuse within a query; keep them out of L1
__device__ __forceinline__ float4 ldg_f4_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
// 256-bit read-only load (sm_100: LDG.E.256): one instruction — one L1 wavefront per touched line —
// for a 32-byte record instead of two
__device__ __forceinline__ void ldg_f8(const float* p, float4& a, float4& b) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(p));
}
// streaming 256-bit load (32-byte aligned): two uint4 halves
__device__ __forceinline__ void ldg_u8_stream(const void* p, uint4& a, uint4& b) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
               : "l"(p));
}
__device__ __forceinline__ uint4 ldg_u4_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// One 32-float trip for the lane's 4 partial sums. L2: d = x - y; acc = fma(d, d, acc)
// (euclidean.s:24-31). Dot: acc = fma(x, y, acc) (dot.s:20-27).
template <bool L2>
__device__ __forceinline__ void trip_accum(const float4& x, const float4& y, float4& acc) {
  if (L2) {
    float d0 = __fsub_rn(x.x, y.x), d1 = __fsub_rn(x.y, y.y), d2 = __fsub_rn(x.z, y.z), d3 = __fsub_rn(x.w, y.w);
    acc.x = __fmaf_rn(d0, d0, acc.x);
    acc.y = __fmaf_rn(d1, d1, acc.y);
    acc.z = __fmaf_rn(d2, d2, acc.z);
    acc.w = __fmaf_rn(d3, d3, acc.w);
  } else {
    acc.x = __fmaf_rn(x.x, y.x, acc.x);
    acc.y = __fmaf_rn(x.y, y.y, acc.y);
    acc.z = __fmaf_rn(x.z, y.z, acc.z);
    acc.w = __fmaf_rn(x.w, y.w, acc.w);
  }
}

template <bool L2>
__device__ __forceinline__ float tail_accum(float x, float y, float t) {
  if (L2) {
    float d = __fsub_rn(x, y);
    return __fmaf_rn(d, d, t);
  }
  return __fmaf_rn(x, y, t);
}

// Reduction across the 8-lane group (dot.s:45-54 / euclidean.s:55-64). Valid in the
// group's lane 0 only. All 32 lanes must call it (full-mask shuffles).
__device__ __forceinline__ float group_reduce(float4 acc, float tail) {
  float4 s = acc;
#pragma unroll
  for (int a = 1; a <= 3; ++a) {
    s.x = __fadd_rn(s.x, __shfl_down_sync(SDB_FULL, acc.x, 2 * a, 8));
    s.y = __fadd_rn(s.y, __shfl_down_sync(SDB_FULL, acc.y, 2 * a, 8));
    s.z = __fadd_rn(s.z, __shfl_down_sync(SDB_FULL, acc.z, 2 * a, 8));
    s.w = __fadd_rn(s.w, __shfl_down_sync(SDB_FULL, acc.w, 2 * a, 8));
  }
  float w0 = __fadd_rn(s.x, __shfl_down_sync(SDB_FULL, s.x, 1, 8));
  float w1 = __fadd_rn(s.y, __shfl_down_sync(SDB_FULL, s.y, 1, 8));
  float w2 = __fadd_rn(s.z, __shfl_down_sync(SDB_FULL, s.z, 1, 8));
  float w3 = __fadd_rn(s.w, __shfl_down_sync(SDB_FULL, s.w, 1, 8));
  w0 = __fadd_rn(w0, tail);
  return __fadd_rn(__fadd_rn(w0, w1), __fadd_rn(w2, w3));
}

// distance.go:19-25: dot distance = -dot, cosine = 1 - dot.
template <int METRIC>
__device__ __forceinline__ float metric_epilogue(float s) {
  if (METRIC == METRIC_DOT) return -s;
  if (METRIC == METRIC_COSINE) return __fsub_rn(1.0f, s);
  return s;
}

// Whole-thread (sequential) version of the same order, for kernels where one thread
// owns a pair (flat scan tiles, k-means, PQ tables). x, y readable by this thread.
template <bool L2>
__device__ __forceinline__ float ordered_dist_thread(const float* __restrict__ x, const float* __restrict__ y, int n) {
  float acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.0f;
  int blocks = n >> 5;
  for (int t = 0; t < blocks; ++t) {
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = tail_accum<L2>(x[t * 32 + i], y[t * 32 + i], acc[i]);
  }
  float tail = 0.0f;
  for (int i = blocks << 5; i < n; ++i) tail = tail_accum<L2>(x[i], y[i], tail);
  float w[4];
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    float v0 = __fadd_rn(__fadd_rn(__fadd_rn(acc[l], acc[8 + l]), acc[16 + l]), acc[24 + l]);
    float v1 = __fadd_rn(__fadd_rn(__fadd_rn(acc[4 + l], acc[12 + l]), acc[20 + l]), acc[28 + l]);
    w[l] = __fadd_rn(v0, v1);
  }
  w[0] = __fadd_rn(w[0], tail);
  return __fadd_rn(__fadd_rn(w[0], w[1]), __fadd_rn(w[2], w[3]));
}

// Short vectors (n < 32, e.g. PQ sub-vectors): only the scalar tail path runs in the
// reference, i.e. a plain sequential FMA chain from +0.
template <bool L2>
__device__ __forceinline__ float short_dist_thread(const float* __restrict__ x, const float* __restrict__ y, int n) {
  float t = 0.0f;
  for (int i = 0; i < n; ++i) t = tail_accum<L2>(x[i], y[i], t);
  return t;
}

template <int METRIC>
__device__ __forceinline__ float float_dist_thread(const float* __restrict__ x, const float* __restrict__ y, int n) {
  constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
  float s = (n < 32) ? short_dist_thread<L2>(x, y, n) : ordered_dist_thread<L2>(x, y, n);
  return metric_epilogue<METRIC>(s);
}

// distance.go:33-43 (float64 math like the reference), split so that a caller with one fixed x
// (the beam search's query) computes x's terms once: haversine_terms(x) then haversine_from(x, y).
struct HaversineX {
  double lat, lon, coslat;  // radians; cos(lat)
};
constexpr double HAV_DEG_TO_RAD = 3.14159265358979323846 / 180.0;
__device__ __forceinline__ HaversineX haversine_terms(float x0, float x1) {
  HaversineX h;
  h.lat = double(x0) * HAV_DEG_TO_RAD;
  h.lon = double(x1) * HAV_DEG_TO_RAD;
  h.coslat = cos(h.lat);
  return h;
}
__device__ __forceinline__ float haversine_from(const HaversineX& x, float y0, float y1) {
  const double earthRadius = 6371000.0;
  double laty = double(y0) * HAV_DEG_TO_RAD, lony = double(y1) * HAV_DEG_TO_RAD;
  double dlat = x.lat - laty, dlon = x.lon - lony;
  double sdlat = sin(dlat / 2), sdlon = sin(dlon / 2);
  double a = sdlat * sdlat + x.coslat * cos(laty) * sdlon * sdlon;
  double c = 2 * asin(sqrt(a));
  return float(earthRadius * c);
}
__device__ __forceinline__ float haversine_thread(const float* x, const float* y) {
  return haversine_from(haversine_terms(x[0], x[1]), y[0], y[1]);
}

// distance.go:45-67 on u64 words.
__device__ __forceinline__ float bits_finish(int metric, int a /*xor or and count*/, int b /*or count*/) {
  if (metric == METRIC_JACCARD) {
    if (b == 0) return 0.0f;
    return __fsub_rn(1.0f, __fdiv_rn(float(a), float(b)));
  }
  return float(a);
}

}  // namespace sdb
