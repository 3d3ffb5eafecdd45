// until_m1.cu — instantiates the parking rollout kernel (rollout_until_kernel, cavgym_rollout_until) for M = 1 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m1.cu.
#include "kernels_until.cuh"

namespace cav {
extern const RolloutUntilLauncher<double> kUntilF64M1;
extern const RolloutUntilLauncher<float> kUntilF32M1;
#ifdef CAV_STUB
const RolloutUntilLauncher<double> kUntilF64M1 = nullptr;
const RolloutUntilLauncher<float> kUntilF32M1 = nullptr;
#else
const RolloutUntilLauncher<double> kUntilF64M1 = &launch_rollout_until<double, 1>;
const RolloutUntilLauncher<float> kUntilF32M1 = &launch_rollout_until<float, 1>;
#endif
}  // namespace cav
