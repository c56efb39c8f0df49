// flat_tc.cu — K5 on tensor cores: IndexFlat.Search (shard/index/flat/flat.go:76-132) for a batch
// of queries over an f32 store, exact results, dense contraction on the tensor pipe.
//
// bf16 products cannot be final distances (1e-5 tolerance, SURVEY.md §7.3-⑥), so the tensor
// cores only *generate candidates*, with a guarantee:
//   1. an upper bound tau_q of every query's k-th smallest distance. Default (tcgen05 path, "two-pass
//      form"): the GEMM runs in minimum mode over a sample of the point tiles spread over the id
//      range; the k smallest of a query's per-group minima belong to k different points, so the
//      k-th of them plus the error bound is such a tau_q (kth_thresh_kernel) — no exact work, one
//      candidate pass over all points, one re-score. Level scheme (mma.sync pass; SDB_FLAT_LEVELS=1
//      selects it on the tcgen05 path too, for tests):
//      exact top-k over the first 128 points, then steps 2-3 level by level over disjoint point
//      ranges growing x8 (last level up to x16); a level's candidate list is seeded with the exact
//      top-k of everything before it, so its re-score is the exact top-k of the whole prefix;
//   2. a bf16 GEMM (fp32 accumulate) scores every (query, point) pair: a(q,x) = |x|^2 - 2 q~.x~
//      (+|q|^2) for squared-L2, -q~.x~ for dot/cosine. |a - d| <= eps_q, a bound from the bf16
//      unit roundoff 2^-8 and the largest point norm: eps_q = c1 |q| xmax + c2 (|q|^2 + xmax^2)
//      (two-pass form: the c1 term per pair, c1 |q| |x_j|, carried by the GEMM itself; squared-L2
//      stores are centred first, which shrinks both norms). Every pair with a < tau_q + eps_q is
//      appended to the query's candidate list — a superset of the true top-k, because a true
//      top-k member has d <= tau_q;
//   3. candidates are re-scored with the reference's exact summation order (common.cuh) and the
//      top-k taken by (distance asc, id asc) — flat.go:99,117 with ascending-id iteration.
// A query whose candidate list overflows at any level falls back to the exact scan. The result is
// therefore bit-identical to flat.cu's, and tests compare the two.
//
// Two forms of the GEMM + filter, same candidates:
//   * tc5_filter_kernel (default, dim <= 384): tcgen05.mma M128xN256xK16 from TMA-fed (SWIZZLE_128B)
//     shared memory into TMEM, warp-specialised, bias and threshold folded into the GEMM as a K
//     extension so the epilogue is a sign test — see the comment above the kernel;
//   * tc_filter_kernel (dim > 384, SDB_FLAT_MMA_SYNC=1): mma.sync.m16n8k16 bf16, CTA tile 128 x 128,
//     8 warps of 64x32, K chunks of 64 double-buffered with cp.async, ldmatrix fragments,
//     accumulators in registers.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "index.cuh"
#include "warp_topk.cuh"

namespace sdb {

namespace {

constexpr int TM = 128, TN = 128, TK = 64;
constexpr int TPAD = 8;                 // bf16 elements of row padding (16 B): conflict-free ldmatrix
constexpr int TROW = TK + TPAD;         // 72 bf16 = 144 B per smem row
constexpr int TC_THREADS = 256;
constexpr uint32_t CAND_CAP = 4096;     // candidate ids kept per query
constexpr uint32_t LEVEL0 = 128;        // points scanned exactly to bound the k-th distance
                                        // 1M points: 128 -> 4k -> 131k -> all runs in 5.45 ms, 1024 -> 32k -> all in 5.85 ms
constexpr uint32_t LEVEL_RATIO = 32;    // each tensor-core level covers 32x more points than the one before
constexpr size_t TC_SMEM = size_t(2) * (TM + TN) * TROW * 2 + TN * 4;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// rows of f32 -> bf16 [n][pitch]: columns [0, kp) = scale * v (zero padded; scale is a power of two,
// so the rounding is that of v), columns [kp, pitch) = 0 (the K extension, filled in by
// bias_kernel / thresh_kernel); squared norms of the unscaled rows (fp32, sequential per lane then
// tree: the norm only feeds the candidate bound, not a result)
// mu != nullptr (squared-L2 only): rows are centred, v = src - mu. Distances do not change under a
// common translation, while the candidate bound scales with |q - mu| |x - mu| instead of |q| |x|
// (mu itself need not be exact: any vector is a valid translation, results are re-scored exactly).
__global__ void to_bf16_kernel(const float* src, uint32_t src_pitch, uint32_t dim, uint32_t n, uint32_t n_pad,
                               __nv_bfloat16* dst, uint32_t kp, uint32_t pitch, float scale, float* norms, const float* mu) {
  const uint32_t row = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (row >= n_pad) return;
  float s = 0.0f;
  for (uint32_t i = lane; i < pitch; i += 32) {
    float v = (row < n && i < dim) ? src[size_t(row) * src_pitch + i] - (mu ? mu[i] : 0.0f) : 0.0f;
    s += v * v;
    dst[size_t(row) * pitch + i] = __float2bfloat16_rn(scale * v);
  }
  for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(SDB_FULL, s, o);
  if (lane == 0 && norms) norms[row] = s;
}

// v = hi + mid + lo with three bf16 pieces (24 significant bits: exact for an f32)
__device__ __forceinline__ void split3(float v, __nv_bfloat16& hi, __nv_bfloat16& mid, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  const float r1 = v - __bfloat162float(hi);
  mid = __float2bfloat16_rn(r1);
  lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
}
constexpr float T5_NO_POINT = 3.0e38f;   // bias of a row that holds no point: never passes
constexpr float T5_PASS_ALL = 1.0e38f;   // threshold of a query without a bound yet: every point passes
constexpr float T5_PASS_NONE = -1.0e38f; // padding query rows
// bf16 unit round-off 2^-8 on both factors of a product: |fl(q_i) fl(x_i) - q_i x_i| <= (2u + u^2) |q_i x_i|, summed with
// Cauchy-Schwarz: <= 0.007828 |q| |x| for the dot product, twice that for the -2 q.x of the squared-L2 score
constexpr float T5_C1 = 0.0157f;
constexpr float T5_UP = 1.00001f;  // covers the fp32 rounding of the norms and of the square roots

// tcgen05 pass: the per-point bias and the per-query threshold ride in the GEMM as a K extension,
//   x~ = [ x (bf16) | b_hi b_mid b_lo  1 1 1 | 0 ... ]      b = |x|^2 (squared-L2) or 0 (dot, cosine)
//   q~ = [ s*q      |  1    1     1   -t_hi -t_mid -t_lo | 0 ... ]   s = -2 or -1, t = threshold
// so the accumulator is score - threshold and the filter is its sign bit. Rows that hold no point
// (deleted, never set, beyond the last id) get b = 3e38: never negative against any threshold.
// Seventh extension column (two-pass form): x~ carries |x_j| (rounded up), q~ carries +-c |q| (rounded
// up in magnitude): the accumulator becomes score +- c |q| |x_j|, the bf16 error bound of THIS pair
// instead of the one of the largest row.
__global__ void bias_kernel(const float* xn, const uint8_t* exists, uint32_t rows, uint32_t rows_pad, int l2, float* bias,
                            __nv_bfloat16* x16, uint32_t kp, uint32_t pitch) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows_pad) return;
  const float b = (i >= 2 && i < rows && exists[i]) ? (l2 ? xn[i] : 0.0f) : T5_NO_POINT;
  bias[i] = b;
  __nv_bfloat16 h, m, l;
  split3(b, h, m, l);
  __nv_bfloat16* e = x16 + size_t(i) * pitch + kp;
  const __nv_bfloat16 one = __float2bfloat16_rn(1.0f);
  e[0] = h; e[1] = m; e[2] = l; e[3] = one; e[4] = one; e[5] = one;
  // the row's norm, rounded up: the two-pass form charges every point its own share c |q| |x_j| of the error bound
  e[6] = b < T5_NO_POINT ? __float2bfloat16_ru(sqrtf(xn[i]) * T5_UP) : __float2bfloat16_rn(0.0f);
}

__global__ void xmax_kernel(const float* xn, const uint8_t* exists, uint32_t first, uint32_t end, uint32_t* out_bits) {
  uint32_t i = first + blockIdx.x * blockDim.x + threadIdx.x;
  float v = 0.0f;
  if (i < end && exists[i]) v = xn[i];
  for (int o = 16; o >= 1; o >>= 1) v = fmaxf(v, __shfl_xor_sync(SDB_FULL, v, o));
  if ((threadIdx.x & 31) == 0 && v > 0.0f) atomicMax(out_bits, __float_as_uint(v));  // v >= 0: bits are ordered
}

// per-query pass threshold in "score space": squared-L2 score = xn - 2 acc, dot/cosine score = -acc
__global__ void thresh_kernel(const float* sample_d, const uint32_t* sample_cnt, uint32_t k, const float* qn,
                              const uint32_t* xmax_bits, int metric, uint32_t dim, uint32_t B, uint32_t B_pad, float* thr,
                              __nv_bfloat16* q16, uint32_t kp, uint32_t pitch) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= B_pad) return;
  auto put = [&](float t_plain, float t_ext) {  // thr[]: mma.sync pass; K extension of q16: tcgen05 pass
    thr[q] = t_plain;
    __nv_bfloat16 h, m, l;
    split3(-t_ext, h, m, l);
    __nv_bfloat16* e = q16 + size_t(q) * pitch + kp;
    const __nv_bfloat16 one = __float2bfloat16_rn(1.0f);
    e[0] = one; e[1] = one; e[2] = one; e[3] = h; e[4] = m; e[5] = l;
    e[6] = __float2bfloat16_rn(0.0f);  // level scheme: the bound of the largest row, inside t
  };
  if (q >= B) { put(-INFINITY, T5_PASS_NONE); return; }  // padding rows never pass
  if (sample_cnt[q] < k) { put(INFINITY, T5_PASS_ALL); return; }
  const float tau = sample_d[size_t(q) * k + (k - 1)];
  const float x2 = __uint_as_float(*xmax_bits), q2 = qn[q];
  const float nq = sqrtf(q2), nx = sqrtf(x2);
  const float c1 = T5_C1;                         // bf16 unit roundoff 2^-8 on both factors of -2 q.x
  const float c2 = float(dim + 32) * 4.8e-7f;     // fp32 accumulation of the GEMM (tensor cores may truncate), the K
                                                  // extension, the norms and the exact kernel
  float t;
  if (metric == METRIC_EUCLIDEAN) t = tau + (c1 * nq * nx + c2 * (q2 + x2)) - q2;
  else if (metric == METRIC_DOT) t = tau + (0.5f * c1 + c2) * nq * nx;
  else t = tau + (0.5f * c1 + c2) * nq * nx - 1.0f;  // cosine distance = 1 - dot
  // strictly above t: the tcgen05 pass keeps score - threshold < 0, the mma.sync pass score <= threshold
  const float tt = fminf(t + fabsf(t) * 1e-6f + 1e-30f, T5_PASS_ALL);
  put(tt, tt);
}

// ---- centring (squared-L2): mean of an evenly strided sample of the stored rows, fixed summation order
constexpr uint32_t MU_PARTS = 64;
__global__ void mean_partial_kernel(const float* vec, uint32_t vec_pitch, uint32_t dim, const uint8_t* exists, uint32_t first,
                                    uint32_t end, uint32_t stride, uint32_t per_part, float* partial, uint32_t* cnt) {
  const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x, part = blockIdx.y;
  float s = 0.0f;
  uint32_t c = 0;
  for (uint32_t i = 0; i < per_part; ++i) {
    const uint64_t r = uint64_t(first) + (uint64_t(part) * per_part + i) * stride;
    if (r >= end) break;
    if (!exists[r]) continue;
    ++c;
    if (d < dim) {
      const float v = vec[size_t(r) * vec_pitch + d];
      if (isfinite(v)) s += v;  // a stray inf / NaN row must not poison the translation of every row
    }
  }
  if (d < dim) partial[size_t(part) * dim + d] = s;
  if (d == 0) cnt[part] = c;
}
__global__ void mean_final_kernel(const float* partial, const uint32_t* cnt, uint32_t dim, float* mu) {
  const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= dim) return;
  float s = 0.0f;
  uint32_t c = 0;
  for (uint32_t p = 0; p < MU_PARTS; ++p) { s += partial[size_t(p) * dim + d]; c += cnt[p]; }
  const float m = c ? s / float(c) : 0.0f;
  mu[d] = isfinite(m) ? m : 0.0f;
}

// K extension of the query rows for the minimum-mode pass: threshold 0 and +c |q| against the
// points' norms, so the accumulator is approximate score + c |q| |x_j| >= exact score - (fp32 terms)
__global__ void ext_min_kernel(__nv_bfloat16* q16, uint32_t kp, uint32_t pitch, uint32_t B, uint32_t B_pad, const float* qn, int l2) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= B_pad) return;
  __nv_bfloat16* e = q16 + size_t(q) * pitch + kp;
  const __nv_bfloat16 one = __float2bfloat16_rn(1.0f), zero = __float2bfloat16_rn(0.0f);
  e[0] = one; e[1] = one; e[2] = one; e[3] = zero; e[4] = zero; e[5] = zero;
  e[6] = q < B ? __float2bfloat16_ru((l2 ? T5_C1 : 0.5f * T5_C1) * sqrtf(qn[q]) * T5_UP) : zero;
}

// Threshold of the candidate pass from the minimum-mode pass over a sample of the points. With
// a_j the approximate score, e_j = c |q| |x_j| the bf16 share of the error bound of the pair and
// F the fp32 share (accumulation, norms, the exact kernel): exact_j <= a_j + e_j + F. The minimum
// mode kept m = min (a_j + e_j) per group; the k smallest group minima belong to k different
// points (the groups are disjoint), so the k-th exact score over ALL points is <= m_k + F, and
// every point that good has a_j - e_j <= m_k + 2F = t: the candidate pass keeps a_j - e_j - t < 0.
// One warp per query: k rounds of warp-wide minimum extraction over the <= 512 group minima
// held in registers.
constexpr uint32_t KTH_MAX_GROUPS = 512;
__global__ void __launch_bounds__(128) kth_thresh_kernel(const float* gmin, uint32_t gmin_pitch, uint32_t G, uint32_t k, const float* qn,
                                                         const uint32_t* xmax_bits, int metric, uint32_t dim, uint32_t B,
                                                         uint32_t B_pad, float* thr, __nv_bfloat16* q16, uint32_t kp, uint32_t pitch,
                                                         uint32_t* cand_cnt) {
  const uint32_t q = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (q >= B_pad) return;
  float t_out;
  if (q >= B) {
    t_out = T5_PASS_NONE;  // padding rows never pass
  } else {
    float v[KTH_MAX_GROUPS / 32];
#pragma unroll
    for (uint32_t i = 0; i < KTH_MAX_GROUPS / 32; ++i) {
      const uint32_t g = lane + 32 * i;
      v[i] = g < G ? gmin[size_t(g) * gmin_pitch + q] : INFINITY;
      if (!(v[i] == v[i])) v[i] = INFINITY;  // NaN (inf - inf in a degenerate row): no information
    }
    float mk = INFINITY;
    for (uint32_t r = 0; r < k; ++r) {
      float m = v[0];
      int mi = 0;
#pragma unroll
      for (int i = 1; i < int(KTH_MAX_GROUPS / 32); ++i)
        if (v[i] < m) { m = v[i]; mi = i; }
      float w = m;
      for (int o = 16; o >= 1; o >>= 1) w = fminf(w, __shfl_xor_sync(SDB_FULL, w, o));
      const uint32_t holders = __ballot_sync(SDB_FULL, m == w);
      if (lane == __ffs(holders) - 1) {
#pragma unroll
        for (int i = 0; i < int(KTH_MAX_GROUPS / 32); ++i)
          if (i == mi) v[i] = INFINITY;
      }
      mk = w;
      if (!(w < 1.0e37f)) break;  // fewer than k groups hold a point
    }
    if (!(mk < 1.0e37f)) {
      t_out = T5_PASS_ALL;
    } else {
      const float x2 = __uint_as_float(*xmax_bits), q2 = qn[q];
      const float nq = sqrtf(q2), nx = sqrtf(x2);
      const float c2 = float(dim + 32) * 4.8e-7f;  // as in thresh_kernel
      const float F = metric == METRIC_EUCLIDEAN ? c2 * (q2 + x2) : c2 * nq * nx;
      const float t = mk + 2.0f * F;
      t_out = fminf(t + fabsf(t) * 1e-6f + 1e-30f, T5_PASS_ALL);
    }
  }
  if (lane == 0) {
    thr[q] = t_out;
    __nv_bfloat16 h, m, l;
    split3(-t_out, h, m, l);
    __nv_bfloat16* e = q16 + size_t(q) * pitch + kp;
    const __nv_bfloat16 one = __float2bfloat16_rn(1.0f);
    e[0] = one; e[1] = one; e[2] = one; e[3] = h; e[4] = m; e[5] = l;
    const float ce = (metric == METRIC_EUCLIDEAN ? T5_C1 : 0.5f * T5_C1) * sqrtf(q < B ? qn[q] : 0.0f) * T5_UP;
    e[6] = __hneg(__float2bfloat16_ru(ce));
    if (q < B) cand_cnt[q] = 0;
  }
}

struct TcArgs {
  const __nv_bfloat16* q16;   // [B_pad][pitch]: scale * q, then the K extension
  const __nv_bfloat16* x16;   // [rows_pad][pitch]
  uint32_t pitch;             // kp + 64
  const float* xn;            // [rows_pad]
  const float* thr;           // [B_pad]
  const uint8_t* exists;
  uint32_t kp, first_id, end_id, tiles_per_cta;
  int l2;                     // squared-L2: score = xn - 2 acc; else score = -acc
  uint32_t* cand; uint32_t* cand_cnt;  // [B][CAND_CAP], [B]
  uint32_t B;
  uint32_t rows_alloc;        // rows of x16 / bias (tcgen05 path: point tiles may reach past end_id)
  const float* bias;          // [rows_alloc] tcgen05 path
  // tcgen05 path, minimum mode (gmin != nullptr): no candidates; the smallest accumulator of every
  // (query, group of `fold` point tiles, column half) goes to gmin[group * gmin_pitch + query]
  float* gmin;
  uint32_t gmin_pitch, fold;
  uint32_t tile_stride;       // minimum mode: tile t covers the points from first_id + t * tile_stride * 256 (an evenly
                              // spread sample instead of a prefix); 0 or 1 = contiguous
};

__global__ void __launch_bounds__(TC_THREADS, 2) tc_filter_kernel(TcArgs a) {
  extern __shared__ __align__(16) unsigned char tc_smem[];
  __nv_bfloat16(*sA)[TM * TROW] = reinterpret_cast<__nv_bfloat16(*)[TM * TROW]>(tc_smem);
  __nv_bfloat16(*sB)[TN * TROW] = reinterpret_cast<__nv_bfloat16(*)[TN * TROW]>(tc_smem + size_t(2) * TM * TROW * 2);
  float* s_xn = reinterpret_cast<float*>(tc_smem + size_t(2) * (TM + TN) * TROW * 2);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 2, wn = warp & 3;  // 2 x 4 warps, warp tile 64 x 32
  const uint32_t q0 = blockIdx.x * TM;
  const uint32_t nk = a.kp / TK;
  // this thread's 8 query rows and their thresholds
  float thr[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int h = 0; h < 2; ++h) thr[i][h] = a.thr[q0 + wm * 64 + i * 16 + (lane >> 2) + h * 8];

  const uint32_t tile0 = blockIdx.y * a.tiles_per_cta;
  for (uint32_t t = 0; t < a.tiles_per_cta; ++t) {
    const uint32_t p0 = a.first_id + (tile0 + t) * TN;
    if (p0 >= a.end_id) break;
    float acc[4][4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.0f;
    auto load_chunk = [&](int buf, uint32_t kc) {
      // 128 rows x 128 B per operand = 1024 16-byte pieces each: 4 per thread per operand
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int piece = tid + r * TC_THREADS, row = piece >> 3, seg = piece & 7;
        cp_async16(&sA[buf][row * TROW + seg * 8], a.q16 + size_t(q0 + row) * a.pitch + kc * TK + seg * 8);
        cp_async16(&sB[buf][row * TROW + seg * 8], a.x16 + size_t(p0 + row) * a.pitch + kc * TK + seg * 8);
      }
      cp_async_commit();
    };
    load_chunk(0, 0);
    if (tid < TN) s_xn[tid] = a.xn[p0 + tid];
    for (uint32_t kc = 0; kc < nk; ++kc) {
      const int buf = kc & 1;
      if (kc + 1 < nk) {
        load_chunk(buf ^ 1, kc + 1);
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
#pragma unroll
      for (int ks = 0; ks < TK / 16; ++ks) {
        uint32_t af[4][4], bf[2][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = wm * 64 + i * 16 + (lane & 15), col = ks * 16 + (lane >> 4) * 8;
          ldmatrix_x4(af[i], &sA[buf][row * TROW + col]);
        }
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {  // two n8 blocks per ldmatrix.x4
          const int mat = lane >> 3;
          const int row = wn * 32 + jj * 16 + (lane & 7) + (mat >> 1) * 8, col = ks * 16 + (mat & 1) * 8;
          ldmatrix_x4(bf[jj], &sB[buf][row * TROW + col]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) mma_bf16(acc[i][j], af[i], bf[j >> 1][(j & 1) * 2], bf[j >> 1][(j & 1) * 2 + 1]);
      }
      __syncthreads();
    }
    // ---- filter: keep (query, point) pairs whose approximate score is under the threshold
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int c2 = 0; c2 < 2; ++c2) {
        const int col = wn * 32 + j * 8 + (lane & 3) * 2 + c2;
        const float xn = a.l2 ? s_xn[col] : 0.0f;  // q16 holds -2 q (squared-L2) or -q: score = acc + bias
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float score = acc[i][j][h * 2 + c2] + xn;
            if (score <= thr[i][h]) {
              const uint32_t pid = p0 + col;
              const uint32_t q = q0 + wm * 64 + i * 16 + (lane >> 2) + h * 8;
              if (pid < a.end_id && a.exists[pid] && q < a.B) {
                const uint32_t slot = atomicAdd(&a.cand_cnt[q], 1u);
                if (slot < CAND_CAP) a.cand[size_t(q) * CAND_CAP + slot] = pid;
              }
            }
          }
      }
    }
    __syncthreads();  // s_xn is rewritten by the next tile
  }
}


// ================================================================================================
// tcgen05 form of the candidate pass (the default for dim <= 384): the same bf16 GEMM + threshold
// filter as tc_filter_kernel, on the 5th-generation tensor cores, with the bias (|x|^2) and the
// per-query threshold folded into the GEMM as a K extension (bias_kernel / thresh_kernel) so the
// accumulator is score - threshold and the filter is a sign test.
//   * warp 0 (one lane): TMA producer. The CTA's 128-query tile of q16 is loaded once
//     (pitch/64 boxes of 128 rows x 128 B, SWIZZLE_128B); point tiles of 256 rows stream through
//     a ring of 32 KB stages (one 64-wide K block per stage), cp.async.bulk.tensor + mbarrier.
//   * warp 1 (one lane): issues tcgen05.mma.kind::f16 M128 x N256 x K16 (bf16 in, f32 out),
//     A and B straight from shared memory through matrix descriptors; the accumulator of a point
//     tile is 256 TMEM columns, two tiles (512 columns = all of TMEM) are in flight so the
//     filter of tile t overlaps the MMAs of tile t+1. tcgen05.commit frees a stage / publishes
//     an accumulator.
//   * warps 2..9: epilogue. A thread owns one query (TMEM lane) and half of the tile's columns:
//     tcgen05.ld 32 columns at a time, one funnel shift per element gathers the sign bits, the
//     rare survivors are parked in shared memory and appended to the query's candidate list
//     with one atomicAdd per flush. No block-wide barrier in the steady state.
// One CTA per SM (~200 KB of shared memory, all 512 TMEM columns).
constexpr int T5_M = 128;   // UMMA M = query rows per MMA = TMEM lanes
// Query tiles per CTA x points per tile (UMMA N); T5_QT * T5_N = 256 accumulator columns per stage.
// Measured on B200, 10k x 1M x 128: 1 x 256 runs the pass in 2.9 ms, 2 x 128 (two query tiles
// sharing each point stage: half the L2->SM traffic, but N = 128 MMAs re-read A from shared
// memory twice as often) in 3.5 ms — the pass is not L2-bound.
constexpr int T5_QT = 1;
constexpr int T5_N = 256;
constexpr int T5_KB = 64;
constexpr int T5_THREADS = 320;
constexpr int T5_EPI_THREADS = 256;
constexpr uint32_t T5_QBLK_BYTES = T5_M * 128;  // one K block of one query tile
constexpr uint32_t T5_XBLK_BYTES = T5_N * 128;  // one K block of a point tile = one stage
constexpr uint32_t T5_IDESC = (1u << 4)                      // D format f32
                              | (1u << 7) | (1u << 10)        // A, B format bf16; both K-major
                              | (uint32_t(T5_N >> 3) << 17)   // N
                              | (uint32_t(T5_M >> 4) << 24);  // M

__device__ __forceinline__ void t5_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void t5_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void t5_mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// bounded wait: a protocol error traps instead of hanging the GPU
__device__ __forceinline__ void t5_mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spins = 0; !done; ++spins) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (spins > (1u << 26)) __trap();
  }
}
__device__ __forceinline__ void t5_tma_load_2d(uint32_t dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
               : "memory");
}
// K-major operand, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart (SBO), version 1
__device__ __forceinline__ uint64_t t5_smem_desc(uint32_t addr) {
  return uint64_t((addr & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) |
         (uint64_t(2) << 61);
}
__device__ __forceinline__ void t5_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(T5_IDESC), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void t5_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void t5_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void t5_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void t5_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void t5_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

constexpr int T5_HITS = 6;    // survivors per half-buffer (two halves per epilogue thread)
constexpr int T5_ESTAGES = 2;  // ring of extension blocks
constexpr uint32_t T5_QEXT_BYTES = T5_M * 32;   // extension block of the query tile: 16 bf16 = 32 B per row
constexpr uint32_t T5_XEXT_BYTES = T5_N * 32;   // extension block of a point tile
struct T5Smem {  // offsets from the 1024-byte aligned base
  uint32_t q, qe, x, xe, hits, bars, tmem_slot, total;
  int stages;
};
// nkb = data K blocks (64 wide); the extension travels as a 16-wide block of 32-byte rows
// (SWIZZLE_32B) in its own small ring: a quarter of the bytes a 64-wide block would move
__host__ __device__ inline T5Smem t5_layout(uint32_t nkb, int stages) {
  T5Smem L;
  L.stages = stages;
  L.q = 0;
  L.qe = T5_QT * nkb * T5_QBLK_BYTES;
  L.x = L.qe + ((T5_QT * T5_QEXT_BYTES + 1023u) & ~1023u);
  L.xe = L.x + uint32_t(stages) * T5_XBLK_BYTES;
  L.hits = L.xe + T5_ESTAGES * T5_XEXT_BYTES;
  L.bars = L.hits + T5_EPI_THREADS * 2 * T5_HITS * 4;
  L.tmem_slot = L.bars + (2 * uint32_t(stages) + 2 * T5_ESTAGES + 5) * 8;
  L.total = L.tmem_slot + 16;
  return L;
}

// K-major operand with 32-byte rows (one K16 step wide), 32-byte swizzle: 8-row groups 256 B apart
__device__ __forceinline__ uint64_t t5_smem_desc_sw32(uint32_t addr) {
  return uint64_t((addr & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(256 >> 4) << 32) | (uint64_t(1) << 46) |
         (uint64_t(6) << 61);
}

__global__ void __launch_bounds__(T5_THREADS, 1)
tc5_filter_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                  const __grid_constant__ CUtensorMap map_qe, const __grid_constant__ CUtensorMap map_xe, TcArgs a, int stages) {
  extern __shared__ unsigned char t5_raw[];
  const uint32_t raw = smem_u32(t5_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  unsigned char* gbase = t5_raw + (base - raw);
  const uint32_t nkb = a.kp / T5_KB;  // data K blocks; the extension block (bias, threshold) has its own ring
  const T5Smem L = t5_layout(nkb, stages);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // barriers: full[s], empty[s], q_full, tmem_full[2], tmem_empty[2]
  auto bar_full = [&](int s) { return base + L.bars + uint32_t(s) * 8; };
  auto bar_empty = [&](int s) { return base + L.bars + uint32_t(stages + s) * 8; };
  const uint32_t bar_q = base + L.bars + uint32_t(2 * stages) * 8;
  auto bar_tfull = [&](int i) { return base + L.bars + uint32_t(2 * stages + 1 + i) * 8; };
  auto bar_tempty = [&](int i) { return base + L.bars + uint32_t(2 * stages + 3 + i) * 8; };
  auto bar_efull = [&](int i) { return base + L.bars + uint32_t(2 * stages + 5 + i) * 8; };
  auto bar_eempty = [&](int i) { return base + L.bars + uint32_t(2 * stages + 5 + T5_ESTAGES + i) * 8; };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gbase + L.tmem_slot);

  const uint32_t q0 = blockIdx.x * (T5_M * T5_QT);
  const uint32_t tile_begin = blockIdx.y * a.tiles_per_cta;
  const uint32_t ntiles_total = (a.end_id - a.first_id + T5_N - 1) / T5_N;
  const uint32_t tile_end = min(tile_begin + a.tiles_per_cta, ntiles_total);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      t5_mbar_init(bar_full(s), 1);
      t5_mbar_init(bar_empty(s), 1);
    }
    t5_mbar_init(bar_q, 1);
    for (int i = 0; i < 2; ++i) {
      t5_mbar_init(bar_tfull(i), 1);
      t5_mbar_init(bar_tempty(i), T5_EPI_THREADS / 32);
    }
    for (int i = 0; i < T5_ESTAGES; ++i) {
      t5_mbar_init(bar_efull(i), 1);
      t5_mbar_init(bar_eempty(i), 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // TMEM: all 512 columns (two 256-column accumulators)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(base + L.tmem_slot), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  t5_fence_before();
  __syncthreads();
  t5_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      t5_mbar_expect_tx(bar_q, T5_QT * (nkb * T5_QBLK_BYTES + T5_QEXT_BYTES));
      for (uint32_t qt = 0; qt < T5_QT; ++qt) {
        for (uint32_t kb = 0; kb < nkb; ++kb)
          t5_tma_load_2d(base + L.q + (qt * nkb + kb) * T5_QBLK_BYTES, &map_q, int32_t(kb * T5_KB), int32_t(q0 + qt * T5_M), bar_q);
        t5_tma_load_2d(base + L.qe + qt * T5_QEXT_BYTES, &map_qe, int32_t(a.kp), int32_t(q0 + qt * T5_M), bar_q);
      }
      int s = 0, es = 0;
      uint32_t ph = 0, eph = 0;
      const uint32_t tstride = a.tile_stride ? a.tile_stride : 1u;
      for (uint32_t t = tile_begin; t < tile_end; ++t) {
        const int32_t p0 = int32_t(a.first_id + t * tstride * T5_N);
        for (uint32_t kb = 0; kb < nkb; ++kb) {
          t5_mbar_wait(bar_empty(s), ph ^ 1u);
          t5_mbar_expect_tx(bar_full(s), T5_XBLK_BYTES);
          t5_tma_load_2d(base + L.x + uint32_t(s) * T5_XBLK_BYTES, &map_x, int32_t(kb * T5_KB), p0, bar_full(s));
          if (++s == stages) { s = 0; ph ^= 1u; }
        }
        t5_mbar_wait(bar_eempty(es), eph ^ 1u);
        t5_mbar_expect_tx(bar_efull(es), T5_XEXT_BYTES);
        t5_tma_load_2d(base + L.xe + uint32_t(es) * T5_XEXT_BYTES, &map_xe, int32_t(a.kp), p0, bar_efull(es));
        if (++es == T5_ESTAGES) { es = 0; eph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      t5_mbar_wait(bar_q, 0);
      t5_fence_after();
      int s = 0, es = 0;
      uint32_t ph = 0, eph = 0;
      uint32_t it = 0;
      for (uint32_t t = tile_begin; t < tile_end; ++t, ++it) {
        const uint32_t acc = it & 1u, aph = (it >> 1) & 1u;
        t5_mbar_wait(bar_tempty(acc), aph ^ 1u);  // the epilogue has drained this accumulator
        t5_fence_after();
        const uint32_t d_tmem = tmem_base + acc * (T5_QT * T5_N);
        for (uint32_t kb = 0; kb < nkb; ++kb) {
          t5_mbar_wait(bar_full(s), ph);
          t5_fence_after();
          const uint64_t bdesc = t5_smem_desc(base + L.x + uint32_t(s) * T5_XBLK_BYTES);
          for (uint32_t qt = 0; qt < T5_QT; ++qt) {
            const uint64_t adesc = t5_smem_desc(base + L.q + (qt * nkb + kb) * T5_QBLK_BYTES);
#pragma unroll
            for (uint32_t k = 0; k < T5_KB / 16; ++k)  // +32 B per K step inside the swizzle row
              t5_mma(d_tmem + qt * T5_N, adesc + 2 * k, bdesc + 2 * k, (kb | k) != 0 ? 1u : 0u);
          }
          t5_commit(bar_empty(s));  // stage free once these MMAs have read it
          if (++s == stages) { s = 0; ph ^= 1u; }
        }
        // the K extension (bias, threshold): one K16 step from the 32-byte-row ring
        t5_mbar_wait(bar_efull(es), eph);
        t5_fence_after();
        for (uint32_t qt = 0; qt < T5_QT; ++qt)
          t5_mma(d_tmem + qt * T5_N, t5_smem_desc_sw32(base + L.qe + qt * T5_QEXT_BYTES),
                 t5_smem_desc_sw32(base + L.xe + uint32_t(es) * T5_XEXT_BYTES), 1u);
        t5_commit(bar_eempty(es));
        if (++es == T5_ESTAGES) { es = 0; eph ^= 1u; }
        t5_commit(bar_tfull(acc));  // accumulator complete
      }
    }
  } else {
    // ===== epilogue: sign filter =====
    // The accumulator already is score - threshold (K extension): a pair survives iff its sign
    // bit is set. One funnel shift per element collects the 32 sign bits of a chunk. No
    // block-level synchronisation: a warp that is busy appending survivors never holds the other
    // seven back; the only coupling is the accumulator hand-off with the MMA warp.
    const int e = warp - 2;                 // 0..7
    const int quad = warp & 3;              // TMEM lanes 32*quad .. 32*quad+31 are this warp's
    const int qt = T5_QT == 2 ? (e >> 2) : 0;        // query tile of this warp
    const int col0 = T5_QT == 2 ? 0 : (e >> 2) * 128;  // its 128 of the tile's columns
    const int etid = threadIdx.x - 64;      // 0..255
    const uint32_t q = q0 + uint32_t(qt) * T5_M + uint32_t(quad) * 32 + lane;
    const bool q_ok = q < a.B;
    // Two half-buffers per thread. A full half reserves its slots with an atomicAdd whose return
    // value is NOT consumed yet: the thread goes on filtering into the other half, and copies the
    // reserved half out at the next flush, when the round trip (~1 us) has long completed. (Waiting
    // for every atomicAdd was 40 % of the samples of a candidate-dense level.)
    uint32_t* hit_buf = reinterpret_cast<uint32_t*>(gbase + L.hits) + etid * (2 * T5_HITS);
    uint32_t* my_hits = hit_buf;
    int nh = 0, cur_half = 0, pend_n = 0;
    uint32_t pend_slot = 0;
    auto drain_pending = [&]() {  // copy out the half reserved by the previous flush
      const uint32_t* src = hit_buf + (cur_half ^ 1) * T5_HITS;
      uint32_t slot = pend_slot;
      for (int i = 0; i < pend_n; ++i, ++slot)
        if (slot < CAND_CAP) a.cand[size_t(q) * CAND_CAP + slot] = src[i];
      pend_n = 0;
    };
    auto flush_hits = [&]() {
      drain_pending();
      if (nh && q_ok) {
        pend_slot = atomicAdd(&a.cand_cnt[q], uint32_t(nh));
        pend_n = nh;
      }
      cur_half ^= 1;
      my_hits = hit_buf + cur_half * T5_HITS;
      nh = 0;
    };
    uint32_t it = 0;
    if (a.gmin) {
      // ===== minimum mode: the thresholds are zero, the accumulator is the approximate score; keep
      // the smallest one per (query, group of `fold` tiles, column half). The launch makes
      // tiles_per_cta a multiple of fold, so every group belongs to one thread: plain stores.
      float gm = INFINITY;
      for (uint32_t t = tile_begin; t < tile_end; ++t, ++it) {
        const uint32_t acc = it & 1u, aph = (it >> 1) & 1u;
        t5_mbar_wait(bar_tfull(acc), aph);
        t5_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t(quad * 32) << 16) + acc * (T5_QT * T5_N) + uint32_t(qt) * T5_N + uint32_t(col0);
        uint32_t v[2][32];
        t5_ld32(taddr, v[0]);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          t5_wait_ld();
          if (c + 1 < 4) t5_ld32(taddr + uint32_t(c + 1) * 32, v[(c + 1) & 1]);
          float m0 = INFINITY, m1 = INFINITY, m2 = INFINITY, m3 = INFINITY;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            m0 = fminf(m0, __uint_as_float(v[c & 1][j]));
            m1 = fminf(m1, __uint_as_float(v[c & 1][j + 1]));
            m2 = fminf(m2, __uint_as_float(v[c & 1][j + 2]));
            m3 = fminf(m3, __uint_as_float(v[c & 1][j + 3]));
          }
          gm = fminf(gm, fminf(fminf(m0, m1), fminf(m2, m3)));
        }
        t5_fence_before();
        __syncwarp();
        if (lane == 0) t5_mbar_arrive(bar_tempty(acc));
        if ((t + 1) % a.fold == 0 || t + 1 == tile_end) {
          if (q_ok) a.gmin[size_t((t / a.fold) * 2 + uint32_t(e >> 2)) * a.gmin_pitch + q] = gm;
          gm = INFINITY;
        }
      }
    } else
    for (uint32_t t = tile_begin; t < tile_end; ++t, ++it) {
      const uint32_t acc = it & 1u, aph = (it >> 1) & 1u;
      const uint32_t p0 = a.first_id + t * T5_N;
      t5_mbar_wait(bar_tfull(acc), aph);
      t5_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t(quad * 32) << 16) + acc * (T5_QT * T5_N) + uint32_t(qt) * T5_N + uint32_t(col0);
      uint32_t v[2][32];
      t5_ld32(taddr, v[0]);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        t5_wait_ld();
        if (c + 1 < 4) t5_ld32(taddr + uint32_t(c + 1) * 32, v[(c + 1) & 1]);
        uint32_t mask = 0;  // bit 31 - j = sign of column j
#pragma unroll
        for (int j = 0; j < 32; ++j) mask = __funnelshift_l(v[c & 1][j], mask, 1);
        // survivors are rare (~k * LEVEL_RATIO per query per level): park them in this thread's
        // shared-memory list; one atomicAdd per flush instead of one global round trip per hit
        while (mask) {
          const int j = __clz(mask);
          mask &= ~(0x80000000u >> j);
          my_hits[nh++] = p0 + uint32_t(col0) + uint32_t(c) * 32 + uint32_t(j);
          if (nh == T5_HITS) flush_hits();
        }
      }
      t5_fence_before();
      __syncwarp();
      if (lane == 0) t5_mbar_arrive(bar_tempty(acc));
    }
    flush_hits();
    drain_pending();
  }
  t5_fence_before();
  __syncthreads();
  if (warp == 1) {
    t5_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

PFN_cuTensorMapEncodeTiled_v12000 t5_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

// [rows][pitch] bf16 row-major -> boxes of box_rows x box_cols elements: 64 columns with the
// 128-byte swizzle (data K blocks), 16 columns with the 32-byte swizzle (the K extension)
int t5_make_map(CUtensorMap* map, const void* ptr, uint32_t rows, uint32_t pitch, uint32_t box_rows, uint32_t box_cols) {
  auto fn = t5_encode_fn();
  if (!fn) return fail(SDB_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t gdim[2] = {pitch, rows};
  cuuint64_t gstride[1] = {cuuint64_t(pitch) * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SDB_ERR_CUDA, "cuTensorMapEncodeTiled failed: " + std::to_string(int(r)));
  return SDB_OK;
}

// the query tile (all K blocks + the extension) stays resident next to at least two point stages
bool t5_eligible(uint32_t kp) { return kp <= 384 && !getenv("SDB_FLAT_MMA_SYNC"); }

int launch_tc5_filter(sdb_index* ix, TcArgs ta, uint32_t B_pad, cudaStream_t stream) {
  const uint32_t nkb = ta.kp / T5_KB;
  const uint32_t fixed = t5_layout(nkb, 0).total + 1024;
  int stages = int((227u * 1024u - fixed) / T5_XBLK_BYTES);
  if (stages > 8) stages = 8;
  const T5Smem L = t5_layout(nkb, stages);
  const size_t smem = size_t(L.total) + 1024;
  CUtensorMap mq, mx, mqe, mxe;
  int rc;
  if ((rc = t5_make_map(&mq, ta.q16, B_pad, ta.pitch, T5_M, T5_KB)) || (rc = t5_make_map(&mx, ta.x16, ta.rows_alloc, ta.pitch, T5_N, T5_KB)) ||
      (rc = t5_make_map(&mqe, ta.q16, B_pad, ta.pitch, T5_M, 16)) || (rc = t5_make_map(&mxe, ta.x16, ta.rows_alloc, ta.pitch, T5_N, 16)))
    return rc;
  static size_t attr_smem_dev[64] = {};  // cudaFuncSetAttribute is per device
  size_t& attr_smem = attr_smem_dev[ix->device & 63];
  if (attr_smem < smem) {
    SDB_CUDA(cudaFuncSetAttribute(tc5_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    attr_smem = smem;
  }
  const uint32_t qtiles = B_pad / (T5_M * T5_QT);
  const uint32_t ntiles = (ta.end_id - ta.first_id + T5_N - 1) / T5_N;
  // one CTA per SM: split the point range so that the CTAs fill whole waves of sm_count (the
  // fewest waves >= 3 whose last wave is at least 97 % full; each CTA keeps >= 4 tiles)
  uint32_t ysplit = 1;
  {
    const uint32_t sms = uint32_t(ix->sm_count);
    const uint32_t ymax = std::max<uint32_t>(1, std::min<uint32_t>(64, ntiles / 4));  // >= 4 tiles per CTA
    double best = -1.0;
    for (uint32_t y = 1; y <= ymax; ++y) {
      const uint32_t ctas = qtiles * y, waves = (ctas + sms - 1) / sms;
      const double eff = double(ctas) / (double(waves) * sms);
      if (eff > best) { best = eff; ysplit = y; }
      if (eff >= 0.97 && waves >= 3) { ysplit = y; break; }
    }
  }
  ta.tiles_per_cta = (ntiles + ysplit - 1) / ysplit;
  if (ta.gmin) ta.tiles_per_cta = (ta.tiles_per_cta + ta.fold - 1) / ta.fold * ta.fold;  // a group never spans two CTAs
  ysplit = (ntiles + ta.tiles_per_cta - 1) / ta.tiles_per_cta;
  tc5_filter_kernel<<<dim3(qtiles, ysplit), T5_THREADS, smem, stream>>>(mq, mx, mqe, mxe, ta, stages);
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

// Levels cover disjoint point ranges: a level's candidate list starts with the exact top-k of
// everything before it, so its re-score yields the exact top-k of the whole prefix.
__global__ void seed_cand_kernel(const uint64_t* prev_ids, const uint32_t* prev_cnt, uint32_t k, uint32_t B, uint32_t* cand,
                                 uint32_t* cand_cnt) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= B) return;
  const uint32_t c = min(prev_cnt[q], k);
  for (uint32_t i = 0; i < c; ++i) cand[size_t(q) * CAND_CAP + i] = uint32_t(prev_ids[size_t(q) * k + i]);
  cand_cnt[q] = c;
}

// Exact re-score, one WARP per query (four queries per CTA, no block-wide barrier): the candidates'
// rows are gathered 16 at a time (an 8-lane group per row, all 16 row loads of a lane in flight),
// scored with the reference's summation order, and offered to a k-slot list sorted by (distance asc,
// id asc) that lives in REGISTERS (WarpTopK, warp_topk.cuh). A candidate that does not beat the
// current k-th is dropped by the lane that holds it, so the warp-wide insertion runs
// ~k ln(n/k) times per query. implicit_n > 0: the candidates are the implicit_n points first_id,
// first_id+1, ... (level 0 of the level scheme: no list in memory). cand_total: optional running
// sum of the list lengths (the sdb_flat_last_stats diagnostic).
constexpr int RW_WARPS = 4;
template <int METRIC, int NS>
__global__ void __launch_bounds__(32 * RW_WARPS) rescore_warp_kernel(
    const float* vec, uint32_t vec_pitch, uint32_t dim, const float* queries, uint32_t B, const uint32_t* cand,
    const uint32_t* cand_cnt, uint32_t k, uint64_t* out_ids, float* out_d, uint32_t* out_cnt, uint32_t* overflow_list,
    uint32_t* overflow_cnt, uint32_t* overflow_flag, int last_level, uint32_t first_id, uint32_t implicit_n,
    const uint8_t* exists, unsigned long long* cand_total) {
  extern __shared__ __align__(16) float s_qall[];  // [RW_WARPS][dim rounded up to 4]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, g = lane & 7, grp = lane >> 3;
  const uint32_t q = blockIdx.x * RW_WARPS + wid;
  if (q >= B) return;
  const uint32_t dpad = (dim + 3) & ~3u;
  float* s_q = s_qall + size_t(wid) * dpad;
  const uint32_t n = implicit_n ? implicit_n : cand_cnt[q];
  if (cand_total && lane == 0 && !implicit_n) atomicAdd(cand_total, static_cast<unsigned long long>(n));
  if (!implicit_n && n > CAND_CAP) {
    // Levels cover disjoint point ranges, so a list that overflowed at any level has lost
    // candidates for good: the query goes to the exact scan after the last level (once: the
    // per-query flag). Its outputs of this level stay as they were (the previous bound).
    if (lane == 0) {
      if (atomicExch(&overflow_flag[q], 1u) == 0u) overflow_list[atomicAdd(overflow_cnt, 1u)] = q;
      if (last_level) out_cnt[q] = 0;
    }
    return;
  }
  for (uint32_t i = lane; i < dpad; i += 32) s_q[i] = i < dim ? queries[size_t(q) * dim + i] : 0.0f;
  __syncwarp();
  constexpr bool L2 = (METRIC == METRIC_EUCLIDEAN);
  const int trips = dim >> 5;
  SDB_WARP_TOPK_STATE(top, NS, k, lane);
  auto cand_id = [&](uint32_t c) -> uint32_t { return implicit_n ? first_id + c : cand[size_t(q) * CAND_CAP + c]; };
  uint32_t c0 = 0;
  if (trips <= 4) {
    for (; c0 < n; c0 += 16) {
      float4 y[4][4];
      uint32_t pid[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t c = c0 + u * 4 + grp;
        pid[u] = cand_id(c < n ? c : 0);
        const float* row = vec + size_t(pid[u]) * vec_pitch + 4 * g;
#pragma unroll
        for (int t = 0; t < 4; ++t) y[u][t] = t < trips ? ldg_f4_stream(row + 32 * t) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t c = c0 + u * 4 + grp;
        const float* row = vec + size_t(pid[u]) * vec_pitch;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int t = 0; t < 4; ++t)
          if (t < trips) trip_accum<L2>(*reinterpret_cast<const float4*>(s_q + 32 * t + 4 * g), y[u][t], acc);
        float tail = 0.0f;
        if (g == 0)
          for (uint32_t i = trips << 5; i < dim; ++i) tail = tail_accum<L2>(s_q[i], __ldg(row + i), tail);
        const float r = metric_epilogue<METRIC>(group_reduce(acc, tail));
        const bool have = g == 0 && c < n && (!implicit_n || exists[pid[u]]);
        top.offer(r, pid[u], have);
      }
    }
  }
  for (; c0 < n; c0 += 4) {
    const uint32_t c = c0 + grp;
    const bool act = c < n;
    const uint32_t pid = cand_id(act ? c : 0);
    const float* row = vec + size_t(pid) * vec_pitch;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int t = 0; t < trips; ++t) {
      const float4 x = *reinterpret_cast<const float4*>(s_q + 32 * t + 4 * g);
      const float4 yy = ldg_f4(row + 32 * t + 4 * g);
      trip_accum<L2>(x, yy, acc);
    }
    float tail = 0.0f;
    if (g == 0)
      for (uint32_t i = trips << 5; i < dim; ++i) tail = tail_accum<L2>(s_q[i], __ldg(row + i), tail);
    const float r = metric_epilogue<METRIC>(group_reduce(acc, tail));
    top.offer(r, pid, g == 0 && act && (!implicit_n || exists[pid]));
  }
#pragma unroll
  for (int j = 0; j < NS; ++j) {
    const uint32_t r = lane + 32 * j;
    if (r < k) {
      out_ids[size_t(q) * k + r] = r < top.len ? uint64_t(top.ki[j]) : 0;
      out_d[size_t(q) * k + r] = r < top.len ? top.kd[j] : __int_as_float(0x7f800000);
    }
  }
  if (lane == 0) out_cnt[q] = top.len;
}

}  // namespace

__global__ void gather_queries_kernel(const uint32_t* list, uint32_t n, const float* src, uint32_t dim, float* dst) {
  const uint32_t i = blockIdx.x;
  if (i >= n) return;
  for (uint32_t t = threadIdx.x; t < dim; t += blockDim.x) dst[size_t(i) * dim + t] = src[size_t(list[i]) * dim + t];
}
__global__ void scatter_results_kernel(const uint32_t* list, uint32_t n, uint32_t k, const uint64_t* ids, const float* d,
                                       const uint32_t* cnt, uint64_t* out_ids, float* out_d, uint32_t* out_cnt) {
  const uint32_t i = blockIdx.x;
  if (i >= n) return;
  const uint32_t q = list[i];
  for (uint32_t t = threadIdx.x; t < k; t += blockDim.x) {
    out_ids[size_t(q) * k + t] = ids[size_t(i) * k + t];
    out_d[size_t(q) * k + t] = d[size_t(i) * k + t];
  }
  if (threadIdx.x == 0) out_cnt[q] = cnt[i];
}

// growth of the levels: intermediate levels multiply the covered prefix by LEVEL_MID, the last level
// may cover up to LEVEL_LAST times the prefix before it (a level's re-score handles ~k * ratio
// candidates per query; the intermediate re-scores only serve the next threshold, so they are kept
// small). Measured on 10k x 1M x 128 (host buffers in and out), mid,last: 32,32 4.64 ms; 16,32 4.83;
// 8,32 4.19; 8,64 4.25; 4,32 4.40; 8,16 4.13 ms
static constexpr uint32_t LEVEL_MID = 8, LEVEL_LAST = 16;

bool flat_tc_eligible(const sdb_index* ix, uint32_t k, bool filtered) {
  if (getenv("SDB_FLAT_EXACT")) return false;
  if (filtered || ix->quant_active()) return false;
  if (ix->store_metric != SDB_METRIC_EUCLIDEAN && ix->store_metric != SDB_METRIC_DOT && ix->store_metric != SDB_METRIC_COSINE)
    return false;
  const uint32_t end_id = std::max<uint32_t>(2, ix->max_node_id + 1);
  return end_id - 2 >= LEVEL0 * LEVEL_RATIO && k <= 75;
}

int launch_flat_tc(sdb_index* ix, uint32_t B, const float* d_queries, uint32_t k, uint64_t* d_out_ids, float* d_out_dists,
                   uint32_t* d_out_counts, cudaStream_t stream) {
  const uint32_t dim = ix->p.dim, kp = (dim + TK - 1) / TK * TK;
  const uint32_t first_id = 2, end_id = std::max<uint32_t>(2, ix->max_node_id + 1);
  const uint32_t rows_pad = ix->rows + T5_N;  // the last point tile may read past end_id
  const uint32_t B_pad = (B + 255) / 256 * 256;  // a multiple of both kernels' query tiles
  const bool debug = getenv("SDB_DEBUG_FLAT") != nullptr;
  int rc;
  // ---- bf16 shadow of the store (rebuilt when the store changed)
  const uint32_t pitch = kp + T5_KB;  // one more 64-wide K block: the extension (bias / threshold pieces)
  const bool l2 = ix->store_metric == SDB_METRIC_EUCLIDEAN;
  // squared-L2: the shadow holds x - mu (mu = mean of a sample of the rows), see to_bf16_kernel
  if (ix->tc_epoch != ix->vec_epoch || ix->d_x16.n < size_t(rows_pad) * pitch) {
    if ((rc = ix->d_x16.ensure(size_t(rows_pad) * pitch)) || (rc = ix->d_xn.ensure(rows_pad)) || (rc = ix->d_bias.ensure(rows_pad)))
      return rc;
    if (l2) {
      if ((rc = ix->d_mu.ensure(size_t(MU_PARTS + 1) * dim + MU_PARTS))) return rc;
      float* partial = ix->d_mu.p + dim;
      uint32_t* cnt = reinterpret_cast<uint32_t*>(ix->d_mu.p + size_t(MU_PARTS + 1) * dim);
      const uint32_t span = end_id - first_id;
      const uint32_t stride = std::max<uint32_t>(1, span / 65536);
      const uint32_t per_part = ((span + stride - 1) / stride + MU_PARTS - 1) / MU_PARTS;
      mean_partial_kernel<<<dim3((dim + 127) / 128, MU_PARTS), 128, 0, stream>>>(ix->d_vec, ix->vec_pitch, dim, ix->d_exists, first_id,
                                                                                 end_id, stride, per_part, partial, cnt);
      mean_final_kernel<<<(dim + 127) / 128, 128, 0, stream>>>(partial, cnt, dim, ix->d_mu.p);
      ix->launches += 2;
    }
    to_bf16_kernel<<<(rows_pad + 7) / 8, 256, 0, stream>>>(ix->d_vec, ix->vec_pitch, dim, ix->rows, rows_pad,
                                                          reinterpret_cast<__nv_bfloat16*>(ix->d_x16.p), kp, pitch, 1.0f, ix->d_xn.p,
                                                          l2 ? ix->d_mu.p : nullptr);
    bias_kernel<<<(rows_pad + 255) / 256, 256, 0, stream>>>(ix->d_xn.p, ix->d_exists, ix->rows, rows_pad, l2 ? 1 : 0, ix->d_bias.p,
                                                            reinterpret_cast<__nv_bfloat16*>(ix->d_x16.p), kp, pitch);
    // largest squared norm of a stored row (of the centred rows for squared-L2): part of the candidate bound
    if ((rc = ix->d_xmax.ensure(1))) return rc;
    SDB_CUDA(cudaMemsetAsync(ix->d_xmax.p, 0, sizeof(uint32_t), stream));
    xmax_kernel<<<(end_id - first_id + 255) / 256, 256, 0, stream>>>(ix->d_xn.p, ix->d_exists, first_id, end_id, ix->d_xmax.p);
    ix->launches += 3;
    SDB_CUDA(cudaGetLastError());
    ix->tc_epoch = ix->vec_epoch;
  }
  const uint32_t* d_xmax = ix->d_xmax.p;
  if ((rc = ix->d_q16.ensure(size_t(B_pad) * pitch)) || (rc = ix->d_qn.ensure(B_pad)) || (rc = ix->d_thr.ensure(B_pad)) ||
      (rc = ix->d_cand.ensure(size_t(B) * CAND_CAP)) || (rc = ix->d_candcnt.ensure(size_t(B) * 3 + 8)) ||
      (rc = ix->d_sample_ids.ensure(size_t(B) * k)) || (rc = ix->d_sample_d.ensure(size_t(B) * k)) ||
      (rc = ix->d_sample_cnt.ensure(B)))
    return rc;
  uint32_t* d_cnt = ix->d_candcnt.p;            // [B] candidate counts
  uint32_t* d_ovf_list = ix->d_candcnt.p + B;   // [B] overflowed queries
  uint32_t* d_misc = ix->d_candcnt.p + 2 * size_t(B);  // [1] overflow count, [2..3] candidates of the last level
  uint32_t* d_ovf_flag = d_misc + 8;                   // [B] query already on the overflow list
  SDB_CUDA(cudaMemsetAsync(d_misc, 0, (8 + size_t(B)) * sizeof(uint32_t), stream));
  to_bf16_kernel<<<(B_pad + 7) / 8, 256, 0, stream>>>(d_queries, dim, dim, B, B_pad, reinterpret_cast<__nv_bfloat16*>(ix->d_q16.p),
                                                     kp, pitch, l2 ? -2.0f : -1.0f, ix->d_qn.p, l2 ? ix->d_mu.p : nullptr);
  ix->launches += 1;
  SDB_CUDA(cudaGetLastError());
  static bool attr_set_dev[64] = {};  // cudaFuncSetAttribute is per device
  bool& attr_set = attr_set_dev[ix->device & 63];
  if (!attr_set) {
    SDB_CUDA(cudaFuncSetAttribute(tc_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(TC_SMEM)));
    // the re-score kernel keeps queries in dynamic shared memory: RW_WARPS rows pass the 48 KB
    // default from dim 3 073
    const int wmax = int(RW_WARPS * MAX_DIM * sizeof(float));
    for (auto kern : {rescore_warp_kernel<METRIC_EUCLIDEAN, 1>, rescore_warp_kernel<METRIC_EUCLIDEAN, 3>,
                      rescore_warp_kernel<METRIC_DOT, 1>, rescore_warp_kernel<METRIC_DOT, 3>,
                      rescore_warp_kernel<METRIC_COSINE, 1>, rescore_warp_kernel<METRIC_COSINE, 3>})
      SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, wmax));
    attr_set = true;
  }
  // ---- exact re-score + top-k, one warp per query (rescore_warp_kernel)
  const size_t wsmem = size_t(RW_WARPS) * ((dim + 3) & ~3u) * sizeof(float);
  unsigned long long* d_cand_total = reinterpret_cast<unsigned long long*>(d_misc + 2);  // summed by the last re-score
  auto rescore_warp = [&](uint64_t* o_ids, float* o_d, uint32_t* o_c, int last, uint32_t impl_first, uint32_t impl_n) {
    const uint32_t grid = (B + RW_WARPS - 1) / RW_WARPS;
    unsigned long long* tot = last ? d_cand_total : nullptr;
#define SDB_RW_LAUNCH(M, NS)                                                                                                   \
  rescore_warp_kernel<M, NS><<<grid, 32 * RW_WARPS, wsmem, stream>>>(ix->d_vec, ix->vec_pitch, dim, d_queries, B, ix->d_cand.p, d_cnt, k, \
                                                                     o_ids, o_d, o_c, d_ovf_list, d_misc + 1, d_ovf_flag, last,  \
                                                                     impl_first, impl_n, ix->d_exists, tot)
    const bool small = k <= 32;
    switch (ix->store_metric) {
      case SDB_METRIC_EUCLIDEAN:
        if (small) SDB_RW_LAUNCH(METRIC_EUCLIDEAN, 1); else SDB_RW_LAUNCH(METRIC_EUCLIDEAN, 3);
        break;
      case SDB_METRIC_DOT:
        if (small) SDB_RW_LAUNCH(METRIC_DOT, 1); else SDB_RW_LAUNCH(METRIC_DOT, 3);
        break;
      default:
        if (small) SDB_RW_LAUNCH(METRIC_COSINE, 1); else SDB_RW_LAUNCH(METRIC_COSINE, 3);
        break;
    }
#undef SDB_RW_LAUNCH
  };
  const uint32_t npts = end_id - first_id;
  // ---- two-pass form (tcgen05 path, the default): a minimum-mode pass over a sample prefix gives
  // every query an upper bound of its k-th distance without any exact work (kth_thresh_kernel),
  // then ONE candidate pass over all points and ONE exact re-score. The level scheme below (exact
  // top-k of a growing prefix, four candidate passes + five re-scores at 1M points) remains for
  // the mma.sync pass and as SDB_FLAT_LEVELS=1.
  uint32_t tiles_a = 0, fold = 1;
  const uint32_t whole_tiles = npts / T5_N;
  if (t5_eligible(kp) && !getenv("SDB_FLAT_LEVELS")) {
    uint32_t div = 8;  // sample = 1/8 of the points: ~8 k candidates per query before the error margin
    if (const char* e = getenv("SDB_FLAT_SAMPLE_DIV")) { const int v = atoi(e); if (v >= 1 && v <= 4096) div = uint32_t(v); }
    const uint32_t whole = whole_tiles;  // whole tiles only
    tiles_a = std::min(whole, std::max<uint32_t>({whole / div, 2 * k, 32u}));
    fold = (2 * tiles_a + KTH_MAX_GROUPS - 1) / KTH_MAX_GROUPS;
    if (fold) tiles_a = tiles_a / fold * fold;
    if (tiles_a < k) tiles_a = 0;  // fewer groups than k: no bound from the minima
  }
  if (tiles_a) {
    const uint32_t G = 2 * tiles_a / fold;
    if ((rc = ix->d_gmin.ensure(size_t(G) * B_pad))) return rc;
    ext_min_kernel<<<(B_pad + 127) / 128, 128, 0, stream>>>(reinterpret_cast<__nv_bfloat16*>(ix->d_q16.p), kp, pitch, B, B_pad,
                                                            ix->d_qn.p, l2 ? 1 : 0);
    TcArgs ta{};
    ta.q16 = reinterpret_cast<const __nv_bfloat16*>(ix->d_q16.p);
    ta.x16 = reinterpret_cast<const __nv_bfloat16*>(ix->d_x16.p);
    ta.xn = ix->d_xn.p; ta.thr = ix->d_thr.p; ta.exists = ix->d_exists;
    ta.kp = kp; ta.pitch = pitch; ta.l2 = l2;
    ta.cand = ix->d_cand.p; ta.cand_cnt = d_cnt; ta.B = B;
    ta.rows_alloc = rows_pad; ta.bias = ix->d_bias.p;
    ta.first_id = first_id; ta.end_id = first_id + tiles_a * T5_N;
    ta.gmin = ix->d_gmin.p; ta.gmin_pitch = B_pad; ta.fold = fold;
    ta.tile_stride = whole_tiles / tiles_a;  // the sample tiles are spread over the whole id range
    if ((rc = launch_tc5_filter(ix, ta, B_pad, stream))) return rc;
    kth_thresh_kernel<<<(B_pad + 3) / 4, 128, 0, stream>>>(ix->d_gmin.p, B_pad, G, k, ix->d_qn.p, d_xmax, ix->store_metric, dim, B, B_pad,
                                                          ix->d_thr.p, reinterpret_cast<__nv_bfloat16*>(ix->d_q16.p), kp, pitch, d_cnt);
    ta.end_id = end_id;
    ta.gmin = nullptr; ta.gmin_pitch = 0; ta.fold = 1; ta.tile_stride = 1;
    if ((rc = launch_tc5_filter(ix, ta, B_pad, stream))) return rc;
    rescore_warp(d_out_ids, d_out_dists, d_out_counts, 1, 0, 0);
    ix->launches += 5;
    SDB_CUDA(cudaGetLastError());
    if (debug) {
      std::vector<uint32_t> h(B);
      cudaStreamSynchronize(stream);
      cudaMemcpy(h.data(), d_cnt, B * sizeof(uint32_t), cudaMemcpyDeviceToHost);
      uint64_t tot = 0;
      uint32_t mx = 0;
      for (uint32_t v : h) { tot += v; mx = std::max(mx, v); }
      fprintf(stderr, "[sdb] flat tc two-pass: sample %u points in %u groups, %.1f candidates/query (max %u, cap %u)\n",
              tiles_a * T5_N, G, double(tot) / B, mx, CAND_CAP);
    }
  } else {
  // ---- level 0: exact scan of the first LEVEL0 points bounds every query's k-th distance
  rescore_warp(ix->d_sample_ids.p, ix->d_sample_d.p, ix->d_sample_cnt.p, 0, first_id, std::min<uint32_t>(LEVEL0, end_id - first_id));
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  // ---- levels 1..: tensor-core pass over a 32x larger prefix, thresholds from the level before
  const uint32_t qtiles = B_pad / TM;
  uint64_t covered = LEVEL0;
  uint32_t lvl_begin = first_id + uint32_t(covered);  // levels cover disjoint ranges [lvl_begin, lvl_end)
  while (covered < npts) {
    covered = covered * LEVEL_LAST >= npts ? npts : std::min<uint64_t>(npts, covered * LEVEL_MID);
    // whole 256-point tiles: what a level scans past its nominal end is not scanned again
    uint64_t span = (first_id + covered - lvl_begin + 255) / 256 * 256;
    const bool last = lvl_begin + span >= end_id;
    const uint32_t lvl_end = last ? end_id : lvl_begin + uint32_t(span);
    covered = lvl_end - first_id;
    // thresholds from the previous level's exact top-k
    thresh_kernel<<<(B_pad + 127) / 128, 128, 0, stream>>>(ix->d_sample_d.p, ix->d_sample_cnt.p, k, ix->d_qn.p, d_xmax,
                                                           ix->store_metric, dim, B, B_pad, ix->d_thr.p,
                                                           reinterpret_cast<__nv_bfloat16*>(ix->d_q16.p), kp, pitch);
    seed_cand_kernel<<<(B + 127) / 128, 128, 0, stream>>>(ix->d_sample_ids.p, ix->d_sample_cnt.p, k, B, ix->d_cand.p, d_cnt);
    TcArgs ta{};
    ta.q16 = reinterpret_cast<const __nv_bfloat16*>(ix->d_q16.p);
    ta.x16 = reinterpret_cast<const __nv_bfloat16*>(ix->d_x16.p);
    ta.xn = ix->d_xn.p; ta.thr = ix->d_thr.p; ta.exists = ix->d_exists;
    ta.kp = kp; ta.pitch = pitch; ta.first_id = lvl_begin; ta.end_id = lvl_end;
    ta.l2 = l2;
    ta.cand = ix->d_cand.p; ta.cand_cnt = d_cnt; ta.B = B;
    const uint32_t ntiles = (lvl_end - lvl_begin + TN - 1) / TN;
    // ~6 waves of CTAs (2 resident per SM) so the last wave's imbalance stays small
    uint32_t ysplit = std::max<uint32_t>(1, (uint32_t(ix->sm_count) * 12 + qtiles - 1) / qtiles);
    ysplit = std::min(ysplit, ntiles);
    ta.tiles_per_cta = (ntiles + ysplit - 1) / ysplit;
    ysplit = (ntiles + ta.tiles_per_cta - 1) / ta.tiles_per_cta;
    ta.rows_alloc = rows_pad;
    ta.bias = ix->d_bias.p;
    if (t5_eligible(kp)) {
      if ((rc = launch_tc5_filter(ix, ta, B_pad, stream))) return rc;
    } else {
      tc_filter_kernel<<<dim3(qtiles, ysplit), TC_THREADS, TC_SMEM, stream>>>(ta);
    }
    SDB_CUDA(cudaGetLastError());
    // exact re-score + top-k of the level; the last level writes the caller's outputs
    uint64_t* o_ids = last ? d_out_ids : ix->d_sample_ids.p;
    float* o_d = last ? d_out_dists : ix->d_sample_d.p;
    uint32_t* o_c = last ? d_out_counts : ix->d_sample_cnt.p;
    rescore_warp(o_ids, o_d, o_c, last ? 1 : 0, 0, 0);
    ix->launches += 3;
    SDB_CUDA(cudaGetLastError());
    if (debug) {
      std::vector<uint32_t> h(B);
      cudaStreamSynchronize(stream);
      cudaMemcpy(h.data(), d_cnt, B * sizeof(uint32_t), cudaMemcpyDeviceToHost);
      uint64_t tot = 0;
      uint32_t mx = 0;
      for (uint32_t v : h) { tot += v; mx = std::max(mx, v); }
      fprintf(stderr, "[sdb] flat tc level over %u points: %u queries, %.1f candidates/query (max %u, cap %u)\n",
              lvl_end - lvl_begin, B, double(tot) / B, mx, CAND_CAP);
    }
    lvl_begin = lvl_end;
  }
  }  // level scheme
  // ---- queries whose candidate list overflowed at some level: the exact scan of the list the
  // re-score built (d_ovf_list, count d_misc[1]). Enqueued every time and split by the count on the
  // device, so nothing here waits for the host: two near-empty launches when nothing overflowed.
  if ((rc = launch_flat_exact_list(ix, B, d_queries, k, d_ovf_list, d_misc + 1, d_out_ids, d_out_dists, d_out_counts, stream,
                                   first_id, end_id)))
    return rc;
  // [1] overflow count, [2..3] candidates the last level kept, summed over the batch by the last
  // re-score: a 16-byte copy into page-locked memory behind the last kernel, read by
  // flat_stats_settle once the call has completed
  if ((rc = ix->h_flat_misc.ensure(4))) return rc;
  if (!ix->flat_stats_ev) SDB_CUDA(cudaEventCreateWithFlags(&ix->flat_stats_ev, cudaEventDisableTiming));
  SDB_CUDA(cudaMemcpyAsync(ix->h_flat_misc.p, d_misc, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
  SDB_CUDA(cudaEventRecord(ix->flat_stats_ev, stream));
  ix->flat_stats_pending = true;
  ix->flat_last_path = t5_eligible(kp) ? 2 : 1;
  if (debug) {
    SDB_CUDA(cudaStreamSynchronize(stream));
    fprintf(stderr, "[sdb] flat tc: %u of %u queries overflowed -> exact scan\n", ix->h_flat_misc.p[1], B);
  }
  return SDB_OK;
}

int flat_stats_settle(sdb_index* ix) {
  if (!ix->flat_stats_pending) return SDB_OK;
  SDB_CUDA(cudaEventSynchronize(ix->flat_stats_ev));
  const uint32_t* h = ix->h_flat_misc.p;
  ix->flat_last_candidates = uint64_t(h[2]) | (uint64_t(h[3]) << 32);
  ix->flat_last_overflow = h[1];
  ix->flat_stats_pending = false;
  return SDB_OK;
}

}  // namespace sdb

extern "C" int sdb_flat_last_stats(sdb_index* ix, int32_t* path, uint64_t* candidates, uint32_t* overflowed) {
  if (!ix) return sdb::fail(SDB_ERR_INVALID, "null index");
  std::lock_guard<std::mutex> g(ix->mu);
  SDB_CUDA(cudaSetDevice(ix->device));
  if (int rc = sdb::flat_stats_settle(ix)) return rc;  // waits for a device-entry call still in flight
  if (path) *path = ix->flat_last_path;
  if (candidates) *candidates = ix->flat_last_candidates;
  if (overflowed) *overflowed = ix->flat_last_overflow;
  return SDB_OK;
}
