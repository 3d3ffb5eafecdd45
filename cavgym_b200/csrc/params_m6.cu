// params_m6.cu — instantiates the kernels with per-env tester parameters (kernels_params.cuh, cavgym_set_agent_params) for
// M = 6 bodies.  CAV_STUB (development builds, CAVGYM_ONLY_M) leaves them out, as in small_m6.cu.
#include "kernels_params.cuh"

namespace cav {
extern const ParamsLaunchers<double> kParamsF64M6;
extern const ParamsLaunchers<float> kParamsF32M6;
#ifdef CAV_STUB
const ParamsLaunchers<double> kParamsF64M6 = {nullptr, nullptr, nullptr};
const ParamsLaunchers<float> kParamsF32M6 = {nullptr, nullptr, nullptr};
#else
const ParamsLaunchers<double> kParamsF64M6 = make_params_launchers<double, 6>();
const ParamsLaunchers<float> kParamsF32M6 = make_params_launchers<float, 6>();
#endif
}  // namespace cav
