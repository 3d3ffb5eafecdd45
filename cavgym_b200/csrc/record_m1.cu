// record_m1.cu — instantiates the recording rollout kernel (rollout_record_kernel, cavgym_rollout_record) for M = 1 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m1.cu.
#include "kernels_small.cuh"

namespace cav {
extern const RolloutRecordLauncher<double> kRecordF64M1;
extern const RolloutRecordLauncher<float> kRecordF32M1;
#ifdef CAV_STUB
const RolloutRecordLauncher<double> kRecordF64M1 = nullptr;
const RolloutRecordLauncher<float> kRecordF32M1 = nullptr;
#else
const RolloutRecordLauncher<double> kRecordF64M1 = &launch_rollout_record<double, 1>;
const RolloutRecordLauncher<float> kRecordF32M1 = &launch_rollout_record<float, 1>;
#endif
}  // namespace cav
