// until_m5.cu — instantiates the parking rollout kernel (rollout_until_kernel, cavgym_rollout_until) for M = 5 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m5.cu.
#include "kernels_until.cuh"

namespace cav {
extern const RolloutUntilLauncher<double> kUntilF64M5;
extern const RolloutUntilLauncher<float> kUntilF32M5;
#ifdef CAV_STUB
const RolloutUntilLauncher<double> kUntilF64M5 = nullptr;
const RolloutUntilLauncher<float> kUntilF32M5 = nullptr;
#else
const RolloutUntilLauncher<double> kUntilF64M5 = &launch_rollout_until<double, 5>;
const RolloutUntilLauncher<float> kUntilF32M5 = &launch_rollout_until<float, 5>;
#endif
}  // namespace cav
