// rollout_tables_log.cu -- instantiations of the time-sliced fp32 rollout kernel flying caller-supplied trajectory tables, one per
// rollout (uavb_rollout_tables_f32, kTargetPerRollout), with a state log: staged tensor stores or per-thread streaming stores,
// chosen as in rollout_log.cu.
#include "rollout_impl.cuh"

namespace uavb {

UAVB_LAUNCH_PAIR(kTargetPerRollout, 1);
UAVB_LAUNCH_PAIR(kTargetPerRollout, 2);

}  // namespace uavb
