// until_m7.cu — instantiates the parking rollout kernel (rollout_until_kernel, cavgym_rollout_until) for M = 7 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m7.cu.
#include "kernels_until.cuh"

namespace cav {
extern const RolloutUntilLauncher<double> kUntilF64M7;
extern const RolloutUntilLauncher<float> kUntilF32M7;
#ifdef CAV_STUB
const RolloutUntilLauncher<double> kUntilF64M7 = nullptr;
const RolloutUntilLauncher<float> kUntilF32M7 = nullptr;
#else
const RolloutUntilLauncher<double> kUntilF64M7 = &launch_rollout_until<double, 7>;
const RolloutUntilLauncher<float> kUntilF32M7 = &launch_rollout_until<float, 7>;
#endif
}  // namespace cav
