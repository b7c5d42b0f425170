// rollout_log.cu -- instantiations of the time-sliced fp32 rollout kernel with a state log (HBM-bound at full rate): staged tensor
// stores through the TMA unit where the log can be described by a tensor map, per-thread streaming stores otherwise.
#include "rollout_impl.cuh"

namespace uavb {

UAVB_LAUNCH_PAIR(kTargetFly, 1);
UAVB_LAUNCH_PAIR(kTargetShared, 1);
UAVB_LAUNCH_PAIR(kTargetFly, 2);
UAVB_LAUNCH_PAIR(kTargetShared, 2);

}  // namespace uavb
