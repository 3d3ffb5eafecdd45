// dense.cu — instantiates the warp-per-environment kernels (kernels_dense.cuh) for fp64 and fp32.
#include "kernels_dense.cuh"

namespace cav {
static const DenseLaunchers<double> kDenseF64 = {launch_dense<double>, launch_dense_reset<double>, launch_dense_record<double>};
static const DenseLaunchers<float> kDenseF32 = {launch_dense<float>, launch_dense_reset<float>, launch_dense_record<float>};
template <> const DenseLaunchers<double>* dense_launchers<double>() { return &kDenseF64; }
template <> const DenseLaunchers<float>* dense_launchers<float>() { return &kDenseF32; }
}  // namespace cav
