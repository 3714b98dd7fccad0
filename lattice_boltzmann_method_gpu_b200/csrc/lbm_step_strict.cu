// STRICT arithmetic instantiation of the fused step.  This file is compiled with
// -fmad=false so that every expression keeps the reference's evaluation order
// with IEEE rounding after each operation -- the results are bit-identical to
// the CPU oracle (gcc -ffp-contract=off).  Used by the parity tests to separate
// "indexing / boundary logic" (must be exact) from "arithmetic reformulation"
// (FAST vs STRICT, tolerance).
#include "step_launch.cuh"

namespace lbm {
template cudaError_t launch_step<float, true>(const SparseParams<float> &, int, bool, bool, cudaStream_t);
template cudaError_t launch_step<double, true>(const SparseParams<double> &, int, bool, bool, cudaStream_t);
template cudaError_t launch_persist<float, true>(const SparseParams<float> &, int, int, int, double *, const float *, unsigned *,
                                                 int, cudaStream_t);
template cudaError_t launch_persist<double, true>(const SparseParams<double> &, int, int, int, double *, const double *,
                                                  unsigned *, int, cudaStream_t);
template cudaError_t preload_step_kernels<float, true>(int, int, bool, bool, bool);
template cudaError_t preload_step_kernels<double, true>(int, int, bool, bool, bool);
}  // namespace lbm
