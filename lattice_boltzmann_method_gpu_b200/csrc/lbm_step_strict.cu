// STRICT arithmetic instantiation of the fused step.  This file is compiled with
// -fmad=false so that every expression keeps the reference's evaluation order
// with IEEE rounding after each operation -- the results are bit-identical to
// the CPU oracle (gcc -ffp-contract=off).  Used by the parity tests to separate
// "indexing / boundary logic" (must be exact) from "arithmetic reformulation"
// (FAST vs STRICT, tolerance).
#include "step_dense.cuh"

namespace lbm {
template <typename T>
cudaError_t launch_step_dense_strict(const StepParams<T> &p, bool moments, bool resid, int storage, cudaStream_t s) {
    return launch_step_dense_impl<T, true>(p, moments, resid, storage, s);
}
template cudaError_t launch_step_dense_strict<float>(const StepParams<float> &, bool, bool, int, cudaStream_t);
template cudaError_t launch_step_dense_strict<double>(const StepParams<double> &, bool, bool, int, cudaStream_t);
}  // namespace lbm

#include "step_sparse.cuh"
namespace lbm {
template <typename T>
cudaError_t launch_step_sparse_strict(const SparseParams<T> &p, bool moments, bool resid, cudaStream_t s) {
    return launch_step_sparse_impl<T, true>(p, moments, resid, s);
}
template cudaError_t launch_step_sparse_strict<float>(const SparseParams<float> &, bool, bool, cudaStream_t);
template cudaError_t launch_step_sparse_strict<double>(const SparseParams<double> &, bool, bool, cudaStream_t);
}  // namespace lbm

#include "step_sparse_aa.cuh"
namespace lbm {
template <typename T>
cudaError_t launch_step_sparse_aa_strict(const SparseParams<T> &p, bool moments, bool resid, cudaStream_t s) {
    return launch_step_sparse_aa_impl<T, true>(p, moments, resid, s);
}
template cudaError_t launch_step_sparse_aa_strict<float>(const SparseParams<float> &, bool, bool, cudaStream_t);
template cudaError_t launch_step_sparse_aa_strict<double>(const SparseParams<double> &, bool, bool, cudaStream_t);
template <typename T>
cudaError_t launch_sparse_aa_persist_strict(const SparseParams<T> &p, int nsteps, int parity0, int moments_last, double *S,
                                             const T *pulse, unsigned *barrier, int sm_count, cudaStream_t s) {
    PersistArgs<T> a{nsteps, parity0, moments_last, S ? 1 : 0, S, pulse, barrier};
    return launch_sparse_aa_persist_impl<T, true>(p, a, sm_count, s);
}
template cudaError_t launch_sparse_aa_persist_strict<float>(const SparseParams<float> &, int, int, int, double *, const float *,
                                                             unsigned *, int, cudaStream_t);
template cudaError_t launch_sparse_aa_persist_strict<double>(const SparseParams<double> &, int, int, int, double *, const double *,
                                                              unsigned *, int, cudaStream_t);
}  // namespace lbm

namespace lbm {
// loads the step kernels a run loop of this storage is about to launch (step_dense.cuh preload_kernel);
// resid: the variants that sum |u| (lbm_run_converge) or those that do not (lbm_run_fixed)
template <typename T>
cudaError_t preload_step_kernels_strict(int storage, bool speculative, bool peers, bool resid) {
    if (storage == LBM_STORE_SPARSE_AA) return preload_step_sparse_aa_impl<T, true, LBM_COLL_BGK>(peers, resid);
    if (storage == LBM_STORE_SPARSE_AB) return preload_step_sparse_impl<T, true, LBM_COLL_BGK>(resid);
    return preload_step_dense_impl<T, true, LBM_COLL_BGK>(storage, speculative, resid);
}
template cudaError_t preload_step_kernels_strict<float>(int, bool, bool, bool);
template cudaError_t preload_step_kernels_strict<double>(int, bool, bool, bool);
}  // namespace lbm
