// record_m3.cu — instantiates the recording rollout kernel (rollout_record_kernel, cavgym_rollout_record) for M = 3 bodies.
// CAV_STUB (development builds, CAVGYM_ONLY_M) leaves it out, as in small_m3.cu.
#include "kernels_small.cuh"

namespace cav {
extern const RolloutRecordLauncher<double> kRecordF64M3;
extern const RolloutRecordLauncher<float> kRecordF32M3;
#ifdef CAV_STUB
const RolloutRecordLauncher<double> kRecordF64M3 = nullptr;
const RolloutRecordLauncher<float> kRecordF32M3 = nullptr;
#else
const RolloutRecordLauncher<double> kRecordF64M3 = &launch_rollout_record<double, 3>;
const RolloutRecordLauncher<float> kRecordF32M3 = &launch_rollout_record<float, 3>;
#endif
}  // namespace cav
