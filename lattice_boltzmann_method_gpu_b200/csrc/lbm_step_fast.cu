// FAST arithmetic instantiation of the fused step.  This is the measured path.  Built with -fmad=false
// like the STRICT unit: the FAST collision fuses by explicit fma() calls (lattice.cuh), so its results do
// not depend on which kernel variant ptxas happened to contract how.
#include "step_launch.cuh"

namespace lbm {
template cudaError_t launch_step<float, false>(const SparseParams<float> &, int, bool, bool, cudaStream_t);
template cudaError_t launch_step<double, false>(const SparseParams<double> &, int, bool, bool, cudaStream_t);
template cudaError_t launch_persist<float, false>(const SparseParams<float> &, int, int, int, double *, const float *, unsigned *,
                                                  int, cudaStream_t);
template cudaError_t launch_persist<double, false>(const SparseParams<double> &, int, int, int, double *, const double *,
                                                   unsigned *, int, cudaStream_t);
template cudaError_t preload_step_kernels<float, false>(int, int, bool, bool, bool);
template cudaError_t preload_step_kernels<double, false>(int, int, bool, bool, bool);
}  // namespace lbm
