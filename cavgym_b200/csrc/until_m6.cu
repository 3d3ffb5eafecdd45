// until_m6.cu — instantiates the parking rollout kernel (rollout_until_kernel, cavgym_rollout_until) for M = 6 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m6.cu.
#include "kernels_until.cuh"

namespace cav {
extern const RolloutUntilLauncher<double> kUntilF64M6;
extern const RolloutUntilLauncher<float> kUntilF32M6;
#ifdef CAV_STUB
const RolloutUntilLauncher<double> kUntilF64M6 = nullptr;
const RolloutUntilLauncher<float> kUntilF32M6 = nullptr;
#else
const RolloutUntilLauncher<double> kUntilF64M6 = &launch_rollout_until<double, 6>;
const RolloutUntilLauncher<float> kUntilF32M6 = &launch_rollout_until<float, 6>;
#endif
}  // namespace cav
