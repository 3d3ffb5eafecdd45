// params_m7.cu — instantiates the kernels with per-env tester parameters (kernels_params.cuh, cavgym_set_agent_params) for
// M = 7 bodies.  CAV_STUB (development builds, CAVGYM_ONLY_M) leaves them out, as in small_m7.cu.
#include "kernels_params.cuh"

namespace cav {
extern const ParamsLaunchers<double> kParamsF64M7;
extern const ParamsLaunchers<float> kParamsF32M7;
#ifdef CAV_STUB
const ParamsLaunchers<double> kParamsF64M7 = {nullptr, nullptr, nullptr};
const ParamsLaunchers<float> kParamsF32M7 = {nullptr, nullptr, nullptr};
#else
const ParamsLaunchers<double> kParamsF64M7 = make_params_launchers<double, 7>();
const ParamsLaunchers<float> kParamsF32M7 = make_params_launchers<float, 7>();
#endif
}  // namespace cav
