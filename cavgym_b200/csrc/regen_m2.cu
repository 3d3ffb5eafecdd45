// regen_m2.cu — instantiates the regeneration kernel (kernels_regen.cuh, cavgym_regenerate_episodes) for M = 2 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m2.cu.
#include "kernels_regen.cuh"

namespace cav {
extern const RegenerateLauncher<double> kRegenF64M2;
extern const RegenerateLauncher<float> kRegenF32M2;
#ifdef CAV_STUB
const RegenerateLauncher<double> kRegenF64M2 = nullptr;
const RegenerateLauncher<float> kRegenF32M2 = nullptr;
#else
const RegenerateLauncher<double> kRegenF64M2 = &launch_regenerate<double, 2>;
const RegenerateLauncher<float> kRegenF32M2 = &launch_regenerate<float, 2>;
#endif
}  // namespace cav
