// regen_m4.cu — instantiates the regeneration kernel (kernels_regen.cuh, cavgym_regenerate_episodes) for M = 4 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m4.cu.
#include "kernels_regen.cuh"

namespace cav {
extern const RegenerateLauncher<double> kRegenF64M4;
extern const RegenerateLauncher<float> kRegenF32M4;
#ifdef CAV_STUB
const RegenerateLauncher<double> kRegenF64M4 = nullptr;
const RegenerateLauncher<float> kRegenF32M4 = nullptr;
#else
const RegenerateLauncher<double> kRegenF64M4 = &launch_regenerate<double, 4>;
const RegenerateLauncher<float> kRegenF32M4 = &launch_regenerate<float, 4>;
#endif
}  // namespace cav
