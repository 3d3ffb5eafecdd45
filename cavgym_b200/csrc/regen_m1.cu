// regen_m1.cu — instantiates the regeneration kernel (kernels_regen.cuh, cavgym_regenerate_episodes) for M = 1 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m1.cu.
#include "kernels_regen.cuh"

namespace cav {
extern const RegenerateLauncher<double> kRegenF64M1;
extern const RegenerateLauncher<float> kRegenF32M1;
#ifdef CAV_STUB
const RegenerateLauncher<double> kRegenF64M1 = nullptr;
const RegenerateLauncher<float> kRegenF32M1 = nullptr;
#else
const RegenerateLauncher<double> kRegenF64M1 = &launch_regenerate<double, 1>;
const RegenerateLauncher<float> kRegenF32M1 = &launch_regenerate<float, 1>;
#endif
}  // namespace cav
