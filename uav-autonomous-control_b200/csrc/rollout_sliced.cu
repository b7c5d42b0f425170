// rollout_sliced.cu -- instantiations of the time-sliced persistent rollout kernel (metrics-only fp32, the production path).
#include "rollout_impl.cuh"

namespace uavb {

template <bool LAG> static void launch_lag(bool mc, bool table, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch) {
  if (table) {
    if (mc) rollout_sliced_kernel<true, true, false, LAG><<<grid, kRolloutThreads, smem, st>>>(p, sch, g_spec_exact);
    else rollout_sliced_kernel<false, true, false, LAG><<<grid, kRolloutThreads, smem, st>>>(p, sch, g_spec_exact);
  } else {
    if (mc) rollout_sliced_kernel<true, false, false, LAG><<<grid, kRolloutThreads, smem, st>>>(p, sch, g_spec_exact);
    else rollout_sliced_kernel<false, false, false, LAG><<<grid, kRolloutThreads, smem, st>>>(p, sch, g_spec_exact);
  }
}

void launch_rollout_sliced(bool mc, bool table, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch) {
  if (p.a.thrust_frame_lag) launch_lag<true>(mc, table, grid, smem, st, p, sch);
  else launch_lag<false>(mc, table, grid, smem, st, p, sch);
}

cudaError_t spec_counts_sliced(unsigned long long* counts, bool reset) { return spec_counts<0>(counts, reset); }

}  // namespace uavb
