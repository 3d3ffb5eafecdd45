// record_m4.cu — instantiates the recording rollout kernel (rollout_record_kernel, cavgym_rollout_record) for M = 4 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m4.cu.
#include "kernels_small.cuh"

namespace cav {
extern const RolloutRecordLauncher<double> kRecordF64M4;
extern const RolloutRecordLauncher<float> kRecordF32M4;
#ifdef CAV_STUB
const RolloutRecordLauncher<double> kRecordF64M4 = nullptr;
const RolloutRecordLauncher<float> kRecordF32M4 = nullptr;
#else
const RolloutRecordLauncher<double> kRecordF64M4 = &launch_rollout_record<double, 4>;
const RolloutRecordLauncher<float> kRecordF32M4 = &launch_rollout_record<float, 4>;
#endif
}  // namespace cav
