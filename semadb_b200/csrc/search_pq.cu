// search_pq.cu — beam-search kernel instantiations for PQ codes (on-the-fly entries, table in shared
// memory, table through L1/L2), see search_launch.cuh.
#include "search_launch.cuh"

namespace sdb {
namespace launch {

extern template int launch_pq_fly<4>(sdb_index*, const SearchArgs&, bool, cudaStream_t);
extern template int launch_pq_fly<8>(sdb_index*, const SearchArgs&, bool, cudaStream_t);
extern template int launch_pq_fly<16>(sdb_index*, const SearchArgs&, bool, cudaStream_t);

int launch_pq(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream) {
  if (adc_on_the_fly(ix)) {
    // table entries computed where they are needed from the L2-resident codebook (AdcEvalFly):
    // no per-query table, twelve query-warps per SM. One translation unit per sub-vector length.
    switch (ix->pqSub) {
      case 4: return launch_pq_fly<4>(ix, a, filtered, stream);
      case 8: return launch_pq_fly<8>(ix, a, filtered, stream);
      default: return launch_pq_fly<16>(ix, a, filtered, stream);
    }
  }
  {
    // ADC table in shared memory when at least two query-warps per SM can hold theirs (C4:
    // 96 x 256 x 4 B = 96 KB => exactly two); otherwise the table is read through L1/L2
    const size_t fixed = warp_smem_bytes<VisitedCompactN, false>(0, 0, 0, ix->pqM * ix->pqK) + 1024;
    const size_t room = ix->smem_per_sm / 2 > fixed ? (ix->smem_per_sm / 2 - fixed) / 2 : 0;  // 16-bit visited slots
    if (!filtered && room >= 4096 && !getenv("SDB_ADC_GLOBAL")) {
      SearchArgs t = a;
      if (t.vt_slots > room) t.vt_slots = uint32_t(room) / 8 * 8;
      const uint32_t nch = (ix->pqM + 15) / 16;
      if (nch <= 2) return launch_with_retry<EVAL_ADC_SMEM, 0, 2, 1, 2, false, 12>(ix, t, stream);
      if (nch <= 4) return launch_with_retry<EVAL_ADC_SMEM, 0, 4, 1, 2, false, 12>(ix, t, stream);
      if (nch <= 6) return launch_with_retry<EVAL_ADC_SMEM, 0, 6, 1, 2, false, 12>(ix, t, stream);
      return launch_with_retry<EVAL_ADC_SMEM, 0, 8, 1, 2, false, 12>(ix, t, stream);
    }
    return filtered ? launch_with_retry<EVAL_ADC, 0, 1, 1, 0, true, 1>(ix, a, stream)
                    : launch_with_retry<EVAL_ADC, 0, 1, 1, 2, false, 12>(ix, a, stream);
  }
}

}  // namespace launch
}  // namespace sdb
