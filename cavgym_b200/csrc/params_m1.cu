// params_m1.cu — instantiates the kernels with per-env tester parameters (kernels_params.cuh, cavgym_set_agent_params) for
// M = 1 bodies.  CAV_STUB (development builds, CAVGYM_ONLY_M) leaves them out, as in small_m1.cu.
#include "kernels_params.cuh"

namespace cav {
extern const ParamsLaunchers<double> kParamsF64M1;
extern const ParamsLaunchers<float> kParamsF32M1;
#ifdef CAV_STUB
const ParamsLaunchers<double> kParamsF64M1 = {nullptr, nullptr, nullptr};
const ParamsLaunchers<float> kParamsF32M1 = {nullptr, nullptr, nullptr};
#else
const ParamsLaunchers<double> kParamsF64M1 = make_params_launchers<double, 1>();
const ParamsLaunchers<float> kParamsF32M1 = make_params_launchers<float, 1>();
#endif
}  // namespace cav
