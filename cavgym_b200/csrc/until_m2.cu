// until_m2.cu — instantiates the parking rollout kernel (rollout_until_kernel, cavgym_rollout_until) for M = 2 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m2.cu.
#include "kernels_until.cuh"

namespace cav {
extern const RolloutUntilLauncher<double> kUntilF64M2;
extern const RolloutUntilLauncher<float> kUntilF32M2;
#ifdef CAV_STUB
const RolloutUntilLauncher<double> kUntilF64M2 = nullptr;
const RolloutUntilLauncher<float> kUntilF32M2 = nullptr;
#else
const RolloutUntilLauncher<double> kUntilF64M2 = &launch_rollout_until<double, 2>;
const RolloutUntilLauncher<float> kUntilF32M2 = &launch_rollout_until<float, 2>;
#endif
}  // namespace cav
