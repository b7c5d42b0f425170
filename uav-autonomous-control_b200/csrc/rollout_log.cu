// rollout_log.cu -- instantiations of the time-sliced fp32 rollout kernel with a state log (HBM-bound at full rate): staged tensor
// stores through the TMA unit where the log can be described by a tensor map, per-thread streaming stores otherwise.
#include "rollout_impl.cuh"

namespace uavb {

template <bool LAG> static void launch_tma(bool mc, bool table, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch,
                                           const LogTma& maps) {
  if (table) {
    if (mc) rollout_sliced_tma_kernel<true, true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, maps);
    else rollout_sliced_tma_kernel<false, true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, maps);
  } else {
    if (mc) rollout_sliced_tma_kernel<true, false, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, maps);
    else rollout_sliced_tma_kernel<false, false, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, maps);
  }
}

template <bool LAG> static void launch_lag(bool mc, bool table, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch) {
  if (table) {
    if (mc) rollout_sliced_kernel<true, true, true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, 0);
    else rollout_sliced_kernel<false, true, true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, 0);
  } else {
    if (mc) rollout_sliced_kernel<true, false, true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, 0);
    else rollout_sliced_kernel<false, false, true, LAG><<<grid, kRolloutThreadsLog, smem, st>>>(p, sch, 0);
  }
}

void launch_rollout_sliced_log(bool mc, bool table, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch,
                               const LogTma* maps) {
  if (maps) {
    if (p.a.thrust_frame_lag) launch_tma<true>(mc, table, grid, smem, st, p, sch, *maps);
    else launch_tma<false>(mc, table, grid, smem, st, p, sch, *maps);
    return;
  }
  if (p.a.thrust_frame_lag) launch_lag<true>(mc, table, grid, smem, st, p, sch);
  else launch_lag<false>(mc, table, grid, smem, st, p, sch);
}

}  // namespace uavb
