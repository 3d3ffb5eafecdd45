// regen_m6.cu — instantiates the regeneration kernel (kernels_regen.cuh, cavgym_regenerate_episodes) for M = 6 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m6.cu.
#include "kernels_regen.cuh"

namespace cav {
extern const RegenerateLauncher<double> kRegenF64M6;
extern const RegenerateLauncher<float> kRegenF32M6;
#ifdef CAV_STUB
const RegenerateLauncher<double> kRegenF64M6 = nullptr;
const RegenerateLauncher<float> kRegenF32M6 = nullptr;
#else
const RegenerateLauncher<double> kRegenF64M6 = &launch_regenerate<double, 6>;
const RegenerateLauncher<float> kRegenF32M6 = &launch_regenerate<float, 6>;
#endif
}  // namespace cav
