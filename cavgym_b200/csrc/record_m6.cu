// record_m6.cu — instantiates the recording rollout kernel (rollout_record_kernel, cavgym_rollout_record) for M = 6 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m6.cu.
#include "kernels_small.cuh"

namespace cav {
extern const RolloutRecordLauncher<double> kRecordF64M6;
extern const RolloutRecordLauncher<float> kRecordF32M6;
#ifdef CAV_STUB
const RolloutRecordLauncher<double> kRecordF64M6 = nullptr;
const RolloutRecordLauncher<float> kRecordF32M6 = nullptr;
#else
const RolloutRecordLauncher<double> kRecordF64M6 = &launch_rollout_record<double, 6>;
const RolloutRecordLauncher<float> kRecordF32M6 = &launch_rollout_record<float, 6>;
#endif
}  // namespace cav
