// regen_m7.cu — instantiates the regeneration kernel (kernels_regen.cuh, cavgym_regenerate_episodes) for M = 7 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m7.cu.
#include "kernels_regen.cuh"

namespace cav {
extern const RegenerateLauncher<double> kRegenF64M7;
extern const RegenerateLauncher<float> kRegenF32M7;
#ifdef CAV_STUB
const RegenerateLauncher<double> kRegenF64M7 = nullptr;
const RegenerateLauncher<float> kRegenF32M7 = nullptr;
#else
const RegenerateLauncher<double> kRegenF64M7 = &launch_regenerate<double, 7>;
const RegenerateLauncher<float> kRegenF32M7 = &launch_regenerate<float, 7>;
#endif
}  // namespace cav
