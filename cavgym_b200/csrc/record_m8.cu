// record_m8.cu — instantiates the recording rollout kernel (rollout_record_kernel, cavgym_rollout_record) for M = 8 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m8.cu.
#include "kernels_small.cuh"

namespace cav {
extern const RolloutRecordLauncher<double> kRecordF64M8;
extern const RolloutRecordLauncher<float> kRecordF32M8;
#ifdef CAV_STUB
const RolloutRecordLauncher<double> kRecordF64M8 = nullptr;
const RolloutRecordLauncher<float> kRecordF32M8 = nullptr;
#else
const RolloutRecordLauncher<double> kRecordF64M8 = &launch_rollout_record<double, 8>;
const RolloutRecordLauncher<float> kRecordF32M8 = &launch_rollout_record<float, 8>;
#endif
}  // namespace cav
