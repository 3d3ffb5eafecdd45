// regen_m8.cu — instantiates the regeneration kernel (kernels_regen.cuh, cavgym_regenerate_episodes) for M = 8 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m8.cu.
#include "kernels_regen.cuh"

namespace cav {
extern const RegenerateLauncher<double> kRegenF64M8;
extern const RegenerateLauncher<float> kRegenF32M8;
#ifdef CAV_STUB
const RegenerateLauncher<double> kRegenF64M8 = nullptr;
const RegenerateLauncher<float> kRegenF32M8 = nullptr;
#else
const RegenerateLauncher<double> kRegenF64M8 = &launch_regenerate<double, 8>;
const RegenerateLauncher<float> kRegenF32M8 = &launch_regenerate<float, 8>;
#endif
}  // namespace cav
