// search_geo.cu — beam-search kernel instantiations for dim-2 haversine rows (GeoEval), see search_launch.cuh.
#include "search_launch.cuh"

namespace sdb {
namespace launch {

// Launch bound of the unfiltered geo kernel: 32 CTAs (one query-warp each) per SM, the hardware's
// limit, within 64 registers a thread (no spills). With its 2048-slot visited table (search.cu:
// geo_vt_slots) a query-warp takes 5.3 KB of shared memory. Capping residency at 12, 16 or 24 CTAs/SM
// (a launch-time cap, removed since) measured the same as 32 on a B200 to within 0.5 % at 2048 and 4096 slots
// (profiles/r03_geo.json, 1 M and 10 M points; at 1024 slots 12 CTAs/SM were 7 % slower). Flat
// throughput with more resident queries suggests a per-SM throughput limit; which one is not measured.
constexpr int GEO_MINB = 32;

int launch_geo(sdb_index* ix, const SearchArgs& a, bool filtered, cudaStream_t stream) {
  if (filtered) return launch_with_retry<EVAL_GEO, METRIC_HAVERSINE, 1, 1, 0, true, 1>(ix, a, stream);
  return launch_with_retry<EVAL_GEO, METRIC_HAVERSINE, 1, 1, 2, false, GEO_MINB>(ix, a, stream);
}

}  // namespace launch
}  // namespace sdb
