// until_m3.cu — instantiates the parking rollout kernel (rollout_until_kernel, cavgym_rollout_until) for M = 3 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m3.cu.
#include "kernels_until.cuh"

namespace cav {
extern const RolloutUntilLauncher<double> kUntilF64M3;
extern const RolloutUntilLauncher<float> kUntilF32M3;
#ifdef CAV_STUB
const RolloutUntilLauncher<double> kUntilF64M3 = nullptr;
const RolloutUntilLauncher<float> kUntilF32M3 = nullptr;
#else
const RolloutUntilLauncher<double> kUntilF64M3 = &launch_rollout_until<double, 3>;
const RolloutUntilLauncher<float> kUntilF32M3 = &launch_rollout_until<float, 3>;
#endif
}  // namespace cav
