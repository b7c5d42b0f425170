// rollout_tables_log.cu -- instantiations of the time-sliced fp32 rollout kernel flying caller-supplied trajectory tables, one per
// rollout (uavb_rollout_tables_f32, kTargetPerRollout), with a state log: staged tensor stores or per-thread streaming stores,
// chosen as in rollout_log.cu.
#include "rollout_impl.cuh"

namespace uavb {

template <bool LAG> static void launch_lag(bool mc, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch,
                                           const LogTma* maps, const TableSetDev& ts) {
  if (maps) {
    if (mc) rollout_sliced_tables_tma_kernel<true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, *maps, ts);
    else rollout_sliced_tables_tma_kernel<false, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, *maps, ts);
  } else {
    if (mc) rollout_sliced_tables_kernel<true, true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, ts, 0);
    else rollout_sliced_tables_kernel<false, true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, ts, 0);
  }
}

void launch_rollout_tables_log(bool mc, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch,
                               const LogTma* maps, const TableSetDev& ts) {
  if (p.a.thrust_frame_lag) launch_lag<true>(mc, grid, smem, st, p, sch, maps, ts);
  else launch_lag<false>(mc, grid, smem, st, p, sch, maps, ts);
}

}  // namespace uavb
