// rollout_tables.cu -- instantiations of the time-sliced fp32 rollout kernel flying caller-supplied trajectory tables, one per
// rollout (uavb_rollout_tables_f32, kTargetPerRollout): metrics only, and metrics plus the viewer's flown-path list.
#include "rollout_impl.cuh"

namespace uavb {

UAVB_LAUNCH_PAIR(kTargetPerRollout, 0);
UAVB_LAUNCH_PAIR(kTargetPerRollout, 3);

}  // namespace uavb
