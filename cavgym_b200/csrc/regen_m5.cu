// regen_m5.cu — instantiates the regeneration kernel (kernels_regen.cuh, cavgym_regenerate_episodes) for M = 5 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m5.cu.
#include "kernels_regen.cuh"

namespace cav {
extern const RegenerateLauncher<double> kRegenF64M5;
extern const RegenerateLauncher<float> kRegenF32M5;
#ifdef CAV_STUB
const RegenerateLauncher<double> kRegenF64M5 = nullptr;
const RegenerateLauncher<float> kRegenF32M5 = nullptr;
#else
const RegenerateLauncher<double> kRegenF64M5 = &launch_regenerate<double, 5>;
const RegenerateLauncher<float> kRegenF32M5 = &launch_regenerate<float, 5>;
#endif
}  // namespace cav
