// rollout_tables.cu -- instantiations of the time-sliced fp32 rollout kernel flying caller-supplied trajectory tables, one per
// rollout (uavb_rollout_tables_f32, kTargetPerRollout): metrics only, and metrics plus the viewer's flown-path list.
#include "rollout_impl.cuh"

namespace uavb {

template <bool LAG> static void launch_lag(bool mc, bool traj, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch,
                                           const TableSetDev& ts) {
  if (traj) {
    if (mc) rollout_sliced_tables_traj_kernel<true, LAG><<<grid, kRolloutThreads, smem, st>>>(p, sch, ts);
    else rollout_sliced_tables_traj_kernel<false, LAG><<<grid, kRolloutThreads, smem, st>>>(p, sch, ts);
  } else {
    if (mc) rollout_sliced_tables_kernel<true, false, LAG><<<grid, kRolloutThreads, smem, st>>>(p, sch, ts, g_spec_exact);
    else rollout_sliced_tables_kernel<false, false, LAG><<<grid, kRolloutThreads, smem, st>>>(p, sch, ts, g_spec_exact);
  }
}

void launch_rollout_tables(bool mc, bool traj, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch,
                           const TableSetDev& ts) {
  if (p.a.thrust_frame_lag) launch_lag<true>(mc, traj, grid, smem, st, p, sch, ts);
  else launch_lag<false>(mc, traj, grid, smem, st, p, sch, ts);
}

cudaError_t spec_counts_tables(unsigned long long* counts, bool reset) { return spec_counts<0>(counts, reset); }

}  // namespace uavb
