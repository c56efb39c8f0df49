// search_launch.cuh — launch plumbing of the beam-search kernel variants (search.cuh), shared by
// the translation units that instantiate them: search.cu (dispatcher, bit and PQ stores) and
// search_l2.cu / search_dot.cu / search_cos.cu (one f32 metric each, so the four compile in parallel),
// search_geo.cu (dim-2 haversine rows).
#pragma once
#include "search.cuh"

#include "index.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>

namespace sdb {
namespace launch {

template <int KIND, int METRIC, int TRIPS, int SETS, int MERGE_MIN, class VT, bool FILTER, bool RETRY, int MINB, bool XTRA,
          bool PF, bool REQ>
int launch_variant_x(sdb_index* ix, const SearchArgs& a, cudaStream_t stream) {
  auto kern = beam_search_kernel<KIND, METRIC, TRIPS, SETS, MERGE_MIN, VT, FILTER, RETRY, MINB, XTRA, PF, REQ>;
  // FloatEvalFixed keeps short queries (<= 4 float4 per lane) in registers: no shared copy
  constexpr bool QREG = (KIND == EVAL_FLOAT_FIXED) && TRIPS <= 4;
  const uint32_t qfloats = (KIND == EVAL_ADC || KIND == EVAL_ADC_SMEM || KIND == EVAL_BITS || KIND == EVAL_GEO || QREG) ? 0 : (a.dim + 3) / 4 * 4;
  const uint32_t qwords = (KIND == EVAL_BITS) ? a.bits_pitch : 0;
  const uint32_t table_floats = (KIND == EVAL_ADC_SMEM) ? a.pqM * a.pqK : 0;
  const size_t smem = warp_smem_bytes<VT, FILTER>(qfloats, qwords, a.vt_slots, table_floats);
  static thread_local int cached_dev = -1;
  static thread_local size_t cached_smem = 0;
  static thread_local int ctas_per_sm = 0;
  if (cached_dev != ix->device || cached_smem != smem) {
    if (smem > ix->smem_optin) return fail(SDB_ERR_INTERNAL, "beam search kernel does not fit in shared memory");
    SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    int nb = 0;
    SDB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, 32, smem));
    if (nb <= 0) return fail(SDB_ERR_INTERNAL, "beam search kernel cannot be resident");
    if (MINB > 1 && nb > MINB) nb = MINB;
    ctas_per_sm = nb;
    // The unified L1/shared array is also where in-flight global loads land: ask for no more
    // shared memory than the resident CTAs need so the rest stays L1 (more rows in flight).
    const size_t need_smem = size_t(nb) * (smem + 1024);
    int pct = int((need_smem * 100 + ix->smem_per_sm - 1) / ix->smem_per_sm);
    if (pct > 100) pct = 100;
    SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    if (getenv("SDB_DEBUG_OCC"))
      fprintf(stderr, "[sdb] beam_search variant: smem %zu B/CTA, %d CTAs/SM, carveout %d%% (%zu KB needed)\n", smem, nb, pct,
              need_smem >> 10);
    cached_smem = smem;
    cached_dev = ix->device;
  }
  uint32_t resident = uint32_t(ix->sm_count) * ctas_per_sm;
  uint32_t need = RETRY ? std::min<uint32_t>(uint32_t(ix->sm_count), ix->retry_slots) : a.n_work;
  uint32_t grid = need < resident ? need : resident;
  if (grid == 0) grid = 1;
  kern<<<grid, 32, smem, stream>>>(a, qfloats, qwords);
  ix->launches++;
  SDB_CUDA(cudaGetLastError());
  return SDB_OK;
}

// the start node's overflow edges (after deletes; normally none) get their own instantiation so
// the common case pays nothing for them (the extra loop cost 5 % on C2)
template <int KIND, int METRIC, int TRIPS, int SETS, int MERGE_MIN, class VT, bool FILTER, bool RETRY, int MINB, bool REQ>
int launch_variant_r(sdb_index* ix, const SearchArgs& a, cudaStream_t stream) {
  if (a.n_start_extra != 0)
    return launch_variant_x<KIND, METRIC, TRIPS, SETS, MERGE_MIN, VT, FILTER, RETRY, MINB, true, false, REQ>(ix, a, stream);
  // speculative row prefetch (small-row evaluators, unfiltered first pass)
  // (PQ kernels: +1.6 %; bit rows: -1.6 %, the probes cost more than the L2 hits save — off there)
  constexpr bool PF = !FILTER && !RETRY && (KIND == EVAL_ADC_SMEM || KIND == EVAL_ADC || KIND == EVAL_ADC_FLY);
  return launch_variant_x<KIND, METRIC, TRIPS, SETS, MERGE_MIN, VT, FILTER, RETRY, MINB, false, PF, REQ>(ix, a, stream);
}

// request batches (per-query L / k, a.req) get instantiations of their own, so the kernels every other
// entry launches are compiled exactly as without them
template <int KIND, int METRIC, int TRIPS, int SETS, int MERGE_MIN, class VT, bool FILTER, bool RETRY, int MINB>
int launch_variant(sdb_index* ix, const SearchArgs& a, cudaStream_t stream) {
  if (a.req != nullptr) return launch_variant_r<KIND, METRIC, TRIPS, SETS, MERGE_MIN, VT, FILTER, RETRY, MINB, true>(ix, a, stream);
  return launch_variant_r<KIND, METRIC, TRIPS, SETS, MERGE_MIN, VT, FILTER, RETRY, MINB, false>(ix, a, stream);
}

template <int KIND, int METRIC, int TRIPS, int SETS, int MERGE_MIN, bool FILTER, int MINB>
int launch_with_retry(sdb_index* ix, SearchArgs a, cudaStream_t stream) {
  const bool prof = ix->prof_on && ix->prof_n < sdb_index::PROF_RING;
  if (prof) SDB_CUDA(cudaEventRecord(ix->prof_ev[2 * ix->prof_n], stream));
  int rc = launch_variant<KIND, METRIC, TRIPS, SETS, MERGE_MIN, VisitedCompactN, FILTER, false, MINB>(ix, a, stream);
  if (rc) return rc;
  if (prof) {
    SDB_CUDA(cudaEventRecord(ix->prof_ev[2 * ix->prof_n + 1], stream));
    ix->prof_n++;
  }
  // second pass over queries whose visited set overflowed (normally none): exact visited bitmap
  // over all rows in global memory (VisitedBitmap) — cannot overflow, so every query completes
  a.work_counter = a.work_counter + 2;
  // same evaluator as the first pass (a re-run query walks ~80 hops alone on its SM: the
  // pipelined row gather is what keeps that under a millisecond); the ADC table is read from
  // global memory
  constexpr int RK = (KIND == EVAL_ADC_SMEM) ? EVAL_ADC : KIND;
  constexpr int RT = (KIND == EVAL_BITS || KIND == EVAL_FLOAT_FIXED || KIND == EVAL_ADC_FLY) ? TRIPS : 1;  // rows must still be covered
  constexpr int RS = (KIND == EVAL_BITS || KIND == EVAL_FLOAT_FIXED) ? SETS : 1;
  if (getenv("SDB_DEBUG_RETRY")) {
    uint32_t h[2] = {0, 0};
    cudaStreamSynchronize(stream);
    cudaMemcpy(h, a.work_counter - 2, sizeof(h), cudaMemcpyDeviceToHost);
    fprintf(stderr, "[sdb] beam search: %u of %u queries overflowed the compact visited table -> retry launch\n", h[1], a.B);
  }
  return launch_variant<RK, METRIC, RT, RS, 0, VisitedBitmap, FILTER, true, 1>(ix, a, stream);
}

// PQ search without per-query tables: sub-vectors of 4, 8 or 16 floats whose number is a multiple
// of 4 (C4: 96 x 8). SDB_ADC_TABLE=1 keeps the table kernels (they also serve other shapes), so the
// tests can compare the two.
inline bool adc_on_the_fly(const sdb_index* ix) {
  const bool table = getenv("SDB_ADC_TABLE") != nullptr || getenv("SDB_ADC_GLOBAL") != nullptr;
  return !table && (ix->pqSub == 4 || ix->pqSub == 8 || ix->pqSub == 16) && ix->pqM % 4 == 0 && ix->store_metric != SDB_METRIC_COSINE;
}

// EVAL_ADC_FLY for sub-vectors of SUB floats; METRIC = the store's (euclidean or dot). Instantiated in
// search_pq_fly{4,8,16}.cu.
template <int SUB>
int launch_pq_fly(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream) {
  const bool l2 = ix->store_metric == SDB_METRIC_EUCLIDEAN;
  if (filtered)
    return l2 ? launch_with_retry<EVAL_ADC_FLY, METRIC_EUCLIDEAN, SUB, 1, 0, true, 1>(ix, a, stream)
              : launch_with_retry<EVAL_ADC_FLY, METRIC_DOT, SUB, 1, 0, true, 1>(ix, a, stream);
  return l2 ? launch_with_retry<EVAL_ADC_FLY, METRIC_EUCLIDEAN, SUB, 1, 2, false, 12>(ix, a, stream)
            : launch_with_retry<EVAL_ADC_FLY, METRIC_DOT, SUB, 1, 2, false, 12>(ix, a, stream);
}

template <int METRIC>
int launch_float(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream) {
  if (filtered) return launch_with_retry<EVAL_FLOAT_GENERIC, METRIC, 1, 1, 0, true, 1>(ix, a, stream);
  if (a.dim % 32 == 0) {
    switch (a.dim / 32) {
      case 4: return launch_with_retry<EVAL_FLOAT_FIXED, METRIC, 4, 6, 2, false, 12>(ix, a, stream);
      case 8: return launch_with_retry<EVAL_FLOAT_FIXED, METRIC, 8, 3, 2, false, 12>(ix, a, stream);
      case 12: return launch_with_retry<EVAL_FLOAT_FIXED, METRIC, 12, 2, 2, false, 12>(ix, a, stream);
      case 24: return launch_with_retry<EVAL_FLOAT_FIXED, METRIC, 24, 1, 2, false, 12>(ix, a, stream);
      default: break;
    }
  }
  return launch_with_retry<EVAL_FLOAT_GENERIC, METRIC, 1, 1, 2, false, 12>(ix, a, stream);
}

}  // namespace launch
}  // namespace sdb
