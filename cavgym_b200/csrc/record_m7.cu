// record_m7.cu — instantiates the recording rollout kernel (rollout_record_kernel, cavgym_rollout_record) for M = 7 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m7.cu.
#include "kernels_small.cuh"

namespace cav {
extern const RolloutRecordLauncher<double> kRecordF64M7;
extern const RolloutRecordLauncher<float> kRecordF32M7;
#ifdef CAV_STUB
const RolloutRecordLauncher<double> kRecordF64M7 = nullptr;
const RolloutRecordLauncher<float> kRecordF32M7 = nullptr;
#else
const RolloutRecordLauncher<double> kRecordF64M7 = &launch_rollout_record<double, 7>;
const RolloutRecordLauncher<float> kRecordF32M7 = &launch_rollout_record<float, 7>;
#endif
}  // namespace cav
