// record_m2.cu — instantiates the recording rollout kernel (rollout_record_kernel, cavgym_rollout_record) for M = 2 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m2.cu.
#include "kernels_small.cuh"

namespace cav {
extern const RolloutRecordLauncher<double> kRecordF64M2;
extern const RolloutRecordLauncher<float> kRecordF32M2;
#ifdef CAV_STUB
const RolloutRecordLauncher<double> kRecordF64M2 = nullptr;
const RolloutRecordLauncher<float> kRecordF32M2 = nullptr;
#else
const RolloutRecordLauncher<double> kRecordF64M2 = &launch_rollout_record<double, 2>;
const RolloutRecordLauncher<float> kRecordF32M2 = &launch_rollout_record<float, 2>;
#endif
}  // namespace cav
