// until_m4.cu — instantiates the parking rollout kernel (rollout_until_kernel, cavgym_rollout_until) for M = 4 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m4.cu.
#include "kernels_until.cuh"

namespace cav {
extern const RolloutUntilLauncher<double> kUntilF64M4;
extern const RolloutUntilLauncher<float> kUntilF32M4;
#ifdef CAV_STUB
const RolloutUntilLauncher<double> kUntilF64M4 = nullptr;
const RolloutUntilLauncher<float> kUntilF32M4 = nullptr;
#else
const RolloutUntilLauncher<double> kUntilF64M4 = &launch_rollout_until<double, 4>;
const RolloutUntilLauncher<float> kUntilF32M4 = &launch_rollout_until<float, 4>;
#endif
}  // namespace cav
