// search_bits.cu — beam-search kernel instantiations for bit-packed rows (hamming / jaccard), see search_launch.cuh.
#include "search_launch.cuh"

namespace sdb {
namespace launch {

int launch_bits(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream) {
    // KIND = bits: METRIC = hamming / jaccard, TRIPS = 128-byte chunks per row, SETS = pipeline depth
    const bool jac = ix->bq_metric == SDB_METRIC_JACCARD;
    const uint32_t nch = (ix->bits_pitch + 15) / 16;
    if (filtered) {
      return jac ? launch_with_retry<EVAL_BITS, METRIC_JACCARD, 4, 2, 0, true, 1>(ix, a, stream)
                 : launch_with_retry<EVAL_BITS, METRIC_HAMMING, 4, 2, 0, true, 1>(ix, a, stream);
    }
    if (jac) {
      if (nch <= 1) return launch_with_retry<EVAL_BITS, METRIC_JACCARD, 1, 8, 2, false, 12>(ix, a, stream);
      return launch_with_retry<EVAL_BITS, METRIC_JACCARD, 4, 2, 2, false, 12>(ix, a, stream);
    }
    if (nch <= 1 && ix->bits_pitch % 4 == 0) {
      // rows of whole 32-byte pieces (1024 bits: the C5b shape): four lanes per row, 256-bit loads
      return launch_with_retry<EVAL_BITS, METRIC_HAMMING, 0, 4, 2, false, 16>(ix, a, stream);
    }
    // 128-byte rows: the search is latency-bound on each warp's dependent chain, not on HBM or on
    // L1 capacity like the f32 kernel, so more resident query-warps pay (16 per SM)
    if (nch <= 1) return launch_with_retry<EVAL_BITS, METRIC_HAMMING, 1, 8, 2, false, 16>(ix, a, stream);
    if (nch <= 2) return launch_with_retry<EVAL_BITS, METRIC_HAMMING, 2, 4, 2, false, 12>(ix, a, stream);
    return launch_with_retry<EVAL_BITS, METRIC_HAMMING, 4, 2, 2, false, 12>(ix, a, stream);
}

}  // namespace launch
}  // namespace sdb
