// rollout_traj.cu -- instantiations of the time-sliced fp32 rollout kernel that also records the viewer's flown-path list
// (MujocoSimulation._record_actual_trajectory, mujoco_sim.py:201-218): metrics-only numerics plus a gated 20 Hz position sample.
#include "rollout_impl.cuh"

namespace uavb {

UAVB_LAUNCH_PAIR(kTargetFly, 3);
UAVB_LAUNCH_PAIR(kTargetShared, 3);

}  // namespace uavb
