// record_m5.cu — instantiates the recording rollout kernel (rollout_record_kernel, cavgym_rollout_record) for M = 5 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m5.cu.
#include "kernels_small.cuh"

namespace cav {
extern const RolloutRecordLauncher<double> kRecordF64M5;
extern const RolloutRecordLauncher<float> kRecordF32M5;
#ifdef CAV_STUB
const RolloutRecordLauncher<double> kRecordF64M5 = nullptr;
const RolloutRecordLauncher<float> kRecordF32M5 = nullptr;
#else
const RolloutRecordLauncher<double> kRecordF64M5 = &launch_rollout_record<double, 5>;
const RolloutRecordLauncher<float> kRecordF32M5 = &launch_rollout_record<float, 5>;
#endif
}  // namespace cav
