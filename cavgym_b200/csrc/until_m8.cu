// until_m8.cu — instantiates the parking rollout kernel (rollout_until_kernel, cavgym_rollout_until) for M = 8 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m8.cu.
#include "kernels_until.cuh"

namespace cav {
extern const RolloutUntilLauncher<double> kUntilF64M8;
extern const RolloutUntilLauncher<float> kUntilF32M8;
#ifdef CAV_STUB
const RolloutUntilLauncher<double> kUntilF64M8 = nullptr;
const RolloutUntilLauncher<float> kUntilF32M8 = nullptr;
#else
const RolloutUntilLauncher<double> kUntilF64M8 = &launch_rollout_until<double, 8>;
const RolloutUntilLauncher<float> kUntilF32M8 = &launch_rollout_until<float, 8>;
#endif
}  // namespace cav
