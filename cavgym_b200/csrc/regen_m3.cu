// regen_m3.cu — instantiates the regeneration kernel (kernels_regen.cuh, cavgym_regenerate_episodes) for M = 3 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m3.cu.
#include "kernels_regen.cuh"

namespace cav {
extern const RegenerateLauncher<double> kRegenF64M3;
extern const RegenerateLauncher<float> kRegenF32M3;
#ifdef CAV_STUB
const RegenerateLauncher<double> kRegenF64M3 = nullptr;
const RegenerateLauncher<float> kRegenF32M3 = nullptr;
#else
const RegenerateLauncher<double> kRegenF64M3 = &launch_regenerate<double, 3>;
const RegenerateLauncher<float> kRegenF32M3 = &launch_regenerate<float, 3>;
#endif
}  // namespace cav
