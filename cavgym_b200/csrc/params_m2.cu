// params_m2.cu — instantiates the kernels with per-env tester parameters (kernels_params.cuh, cavgym_set_agent_params) for
// M = 2 bodies.  CAV_STUB (development builds, CAVGYM_ONLY_M) leaves them out, as in small_m2.cu.
#include "kernels_params.cuh"

namespace cav {
extern const ParamsLaunchers<double> kParamsF64M2;
extern const ParamsLaunchers<float> kParamsF32M2;
#ifdef CAV_STUB
const ParamsLaunchers<double> kParamsF64M2 = {nullptr, nullptr, nullptr};
const ParamsLaunchers<float> kParamsF32M2 = {nullptr, nullptr, nullptr};
#else
const ParamsLaunchers<double> kParamsF64M2 = make_params_launchers<double, 2>();
const ParamsLaunchers<float> kParamsF32M2 = make_params_launchers<float, 2>();
#endif
}  // namespace cav
