// FAST arithmetic instantiation of the fused step.  This is the measured path.  Built with -fmad=false
// like the STRICT unit: the FAST collision fuses by explicit fma() calls (lattice.cuh), so its results do
// not depend on which kernel variant ptxas happened to contract how.
#include "step_dense.cuh"

namespace lbm {
template <typename T>
cudaError_t launch_step_dense_fast(const StepParams<T> &p, bool moments, bool resid, int storage, cudaStream_t s) {
    return launch_step_dense_impl<T, false>(p, moments, resid, storage, s);
}
template cudaError_t launch_step_dense_fast<float>(const StepParams<float> &, bool, bool, int, cudaStream_t);
template cudaError_t launch_step_dense_fast<double>(const StepParams<double> &, bool, bool, int, cudaStream_t);
}  // namespace lbm

#include "step_sparse.cuh"
namespace lbm {
template <typename T>
cudaError_t launch_step_sparse_fast(const SparseParams<T> &p, bool moments, bool resid, cudaStream_t s) {
    return launch_step_sparse_impl<T, false>(p, moments, resid, s);
}
template cudaError_t launch_step_sparse_fast<float>(const SparseParams<float> &, bool, bool, cudaStream_t);
template cudaError_t launch_step_sparse_fast<double>(const SparseParams<double> &, bool, bool, cudaStream_t);
}  // namespace lbm

#include "step_sparse_aa.cuh"
namespace lbm {
template <typename T>
cudaError_t launch_step_sparse_aa_fast(const SparseParams<T> &p, bool moments, bool resid, cudaStream_t s) {
    return launch_step_sparse_aa_impl<T, false>(p, moments, resid, s);
}
template cudaError_t launch_step_sparse_aa_fast<float>(const SparseParams<float> &, bool, bool, cudaStream_t);
template cudaError_t launch_step_sparse_aa_fast<double>(const SparseParams<double> &, bool, bool, cudaStream_t);
template <typename T>
cudaError_t launch_sparse_aa_persist_fast(const SparseParams<T> &p, int nsteps, int parity0, int moments_last, double *S,
                                             const T *pulse, unsigned *barrier, int sm_count, cudaStream_t s) {
    PersistArgs<T> a{nsteps, parity0, moments_last, S ? 1 : 0, S, pulse, barrier};
    return launch_sparse_aa_persist_impl<T, false>(p, a, sm_count, s);
}
template cudaError_t launch_sparse_aa_persist_fast<float>(const SparseParams<float> &, int, int, int, double *, const float *,
                                                             unsigned *, int, cudaStream_t);
template cudaError_t launch_sparse_aa_persist_fast<double>(const SparseParams<double> &, int, int, int, double *, const double *,
                                                              unsigned *, int, cudaStream_t);
}  // namespace lbm

namespace lbm {
// loads the step kernels a run loop of this storage is about to launch (step_dense.cuh preload_kernel);
// resid: the variants that sum |u| (lbm_run_converge) or those that do not (lbm_run_fixed); collision: those of
// this lbm_collision
template <typename T, int COLL>
cudaError_t preload_step_kernels_coll(int storage, bool speculative, bool peers, bool resid) {
    if (storage == LBM_STORE_SPARSE_AA) return preload_step_sparse_aa_impl<T, false, COLL>(peers, resid);
    if (storage == LBM_STORE_SPARSE_AB) return preload_step_sparse_impl<T, false, COLL>(resid);
    return preload_step_dense_impl<T, false, COLL>(storage, speculative, resid);
}
template <typename T>
cudaError_t preload_step_kernels_fast(int storage, bool speculative, bool peers, bool resid, int collision) {
    if (collision == LBM_COLL_TRT) return preload_step_kernels_coll<T, LBM_COLL_TRT>(storage, speculative, peers, resid);
    return preload_step_kernels_coll<T, LBM_COLL_BGK>(storage, speculative, peers, resid);
}
template cudaError_t preload_step_kernels_fast<float>(int, bool, bool, bool, int);
template cudaError_t preload_step_kernels_fast<double>(int, bool, bool, bool, int);
}  // namespace lbm
