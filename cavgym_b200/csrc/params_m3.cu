// params_m3.cu — instantiates the kernels with per-env tester parameters (kernels_params.cuh, cavgym_set_agent_params) for
// M = 3 bodies.  CAV_STUB (development builds, CAVGYM_ONLY_M) leaves them out, as in small_m3.cu.
#include "kernels_params.cuh"

namespace cav {
extern const ParamsLaunchers<double> kParamsF64M3;
extern const ParamsLaunchers<float> kParamsF32M3;
#ifdef CAV_STUB
const ParamsLaunchers<double> kParamsF64M3 = {nullptr, nullptr, nullptr};
const ParamsLaunchers<float> kParamsF32M3 = {nullptr, nullptr, nullptr};
#else
const ParamsLaunchers<double> kParamsF64M3 = make_params_launchers<double, 3>();
const ParamsLaunchers<float> kParamsF32M3 = make_params_launchers<float, 3>();
#endif
}  // namespace cav
