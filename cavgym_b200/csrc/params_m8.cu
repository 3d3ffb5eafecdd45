// params_m8.cu — instantiates the kernels with per-env tester parameters (kernels_params.cuh, cavgym_set_agent_params) for
// M = 8 bodies.  CAV_STUB (development builds, CAVGYM_ONLY_M) leaves them out, as in small_m8.cu.
#include "kernels_params.cuh"

namespace cav {
extern const ParamsLaunchers<double> kParamsF64M8;
extern const ParamsLaunchers<float> kParamsF32M8;
#ifdef CAV_STUB
const ParamsLaunchers<double> kParamsF64M8 = {nullptr, nullptr, nullptr};
const ParamsLaunchers<float> kParamsF32M8 = {nullptr, nullptr, nullptr};
#else
const ParamsLaunchers<double> kParamsF64M8 = make_params_launchers<double, 8>();
const ParamsLaunchers<float> kParamsF32M8 = make_params_launchers<float, 8>();
#endif
}  // namespace cav
