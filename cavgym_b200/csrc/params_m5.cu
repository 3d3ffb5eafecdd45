// params_m5.cu — instantiates the kernels with per-env tester parameters (kernels_params.cuh, cavgym_set_agent_params) for
// M = 5 bodies.  CAV_STUB (development builds, CAVGYM_ONLY_M) leaves them out, as in small_m5.cu.
#include "kernels_params.cuh"

namespace cav {
extern const ParamsLaunchers<double> kParamsF64M5;
extern const ParamsLaunchers<float> kParamsF32M5;
#ifdef CAV_STUB
const ParamsLaunchers<double> kParamsF64M5 = {nullptr, nullptr, nullptr};
const ParamsLaunchers<float> kParamsF32M5 = {nullptr, nullptr, nullptr};
#else
const ParamsLaunchers<double> kParamsF64M5 = make_params_launchers<double, 5>();
const ParamsLaunchers<float> kParamsF32M5 = make_params_launchers<float, 5>();
#endif
}  // namespace cav
