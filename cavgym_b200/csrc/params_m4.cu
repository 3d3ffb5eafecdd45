// params_m4.cu — instantiates the kernels with per-env tester parameters (kernels_params.cuh, cavgym_set_agent_params) for
// M = 4 bodies.  CAV_STUB (development builds, CAVGYM_ONLY_M) leaves them out, as in small_m4.cu.
#include "kernels_params.cuh"

namespace cav {
extern const ParamsLaunchers<double> kParamsF64M4;
extern const ParamsLaunchers<float> kParamsF32M4;
#ifdef CAV_STUB
const ParamsLaunchers<double> kParamsF64M4 = {nullptr, nullptr, nullptr};
const ParamsLaunchers<float> kParamsF32M4 = {nullptr, nullptr, nullptr};
#else
const ParamsLaunchers<double> kParamsF64M4 = make_params_launchers<double, 4>();
const ParamsLaunchers<float> kParamsF32M4 = make_params_launchers<float, 4>();
#endif
}  // namespace cav
