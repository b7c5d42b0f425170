// rollout_sliced.cu -- instantiations of the time-sliced persistent rollout kernel (metrics-only fp32, the production path).
#include "rollout_impl.cuh"

namespace uavb {

UAVB_LAUNCH_PAIR(kTargetFly, 0);
UAVB_LAUNCH_PAIR(kTargetShared, 0);

}  // namespace uavb
