// Host side of the fused step: which instantiation of a step kernel a launch runs, the launches, and the preload
// of the run loops.  One selector per kernel family turns the per-launch switches into the instantiation; launch
// and preload both ask it, so a run loop loads exactly the kernels it is about to launch.
// Instantiated for STRICT = false in lbm_step_fast.cu and for STRICT = true in lbm_step_strict.cu.
#pragma once
#include <algorithm>
#include <type_traits>
#include "step_sparse_aa.cuh"

namespace lbm {

// f(std::bool_constant<b>...): run-time switches as template arguments
template <typename F>
auto with_bools(F f) {
    return f();
}
template <typename F, typename... B>
auto with_bools(F f, bool b, B... rest) {
    if (b) return with_bools([&](auto... c) { return f(std::true_type{}, c...); }, rest...);
    return with_bools([&](auto... c) { return f(std::false_type{}, c...); }, rest...);
}
// The kernel f(COLL, b...) names, every argument a compile-time constant.  The collision is a template parameter of
// every step kernel; TRT kernels exist in FAST arithmetic only, so TRT in STRICT arithmetic (or an unknown model)
// selects no kernel: null.
template <bool STRICT, typename F, typename... B>
auto select_kernel(int collision, F f, B... b) {
    auto with = [&](auto coll) { return with_bools([&](auto... c) { return f(coll, c...); }, b...); };
    using K = decltype(with(std::integral_constant<int, LBM_COLL_BGK>{}));
    if (collision == LBM_COLL_BGK) return with(std::integral_constant<int, LBM_COLL_BGK>{});
    if constexpr (!STRICT) {
        if (collision == LBM_COLL_TRT) return with(std::integral_constant<int, LBM_COLL_TRT>{});
    }
    return K(nullptr);
}

template <typename T>
using DenseKernel = void (*)(StepParams<T>);
template <typename T>
using SparseKernel = void (*)(SparseParams<T>);

template <typename T, bool STRICT>
DenseKernel<T> dense_kernel(int collision, bool moments, bool resid, bool spec, int mode) {
    return select_kernel<STRICT>(collision, [&](auto C, auto M, auto R, auto S) -> DenseKernel<T> {
        if (mode == MODE_AA_EVEN) return k_step_dense<T, STRICT, C, M, R, S, MODE_AA_EVEN>;
        if (mode == MODE_AA_ODD) return k_step_dense<T, STRICT, C, M, R, S, MODE_AA_ODD>;
        return k_step_dense<T, STRICT, C, M, R, S, MODE_AB>;
    }, moments, resid, spec);
}
template <typename T, bool STRICT>
SparseKernel<T> sparse_kernel(int collision, bool moments, bool resid) {
    return select_kernel<STRICT>(collision, [](auto C, auto M, auto R) -> SparseKernel<T> {
        return k_step_sparse<T, STRICT, C, M, R>;
    }, moments, resid);
}
template <typename T, bool STRICT>
SparseKernel<T> sparse_aa_kernel(int collision, bool moments, bool resid, bool peers, int parity) {
    return select_kernel<STRICT>(collision, [&](auto C, auto M, auto R, auto P) -> SparseKernel<T> {
        if (parity == 0) return k_sparse_aa_even<T, STRICT, C, M, R, P>;
        return k_sparse_aa_odd<T, STRICT, C, M, R, P>;
    }, moments, resid, peers);
}
template <typename T, bool STRICT>
auto persist_kernel(int collision) {
    return select_kernel<STRICT>(collision, [](auto C) { return k_sparse_aa_persist<T, STRICT, C>; });
}

inline int dense_mode(int storage, int parity) {
    if (storage != LBM_STORE_DENSE_AA) return MODE_AB;
    return parity == 0 ? MODE_AA_EVEN : MODE_AA_ODD;
}
// host: the per-direction base pointers of the compact arrays, and dk[] of the in-place storage
template <typename T>
void set_bases(SparseParams<T> &sp) {
    StepParams<T> &p = sp.base;
    for (int q = 0; q < Q; q++) {
        p.pull_base[q] = p.src + (long long)q * p.qstride;
        p.store_base[q] = p.dst + (long long)q * p.qstride;
        sp.dk[q] = (int)((long long)(q - oppq(q)) * p.qstride);  // |q - opp q| <= 3, qstride < 2^31 / 3 (checked by the host)
    }
}

template <typename T, bool STRICT>
cudaError_t launch_step(const SparseParams<T> &sp_in, int storage, bool moments, bool resid, cudaStream_t s) {
    SparseParams<T> sp = sp_in;
    StepParams<T> &p = sp.base;
    cudaLaunchAttribute pdl[1];
    pdl[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.stream = s, cfg.attrs = pdl;
    if (storage == LBM_STORE_SPARSE_AB || storage == LBM_STORE_SPARSE_AA) {
        const bool aa = storage == LBM_STORE_SPARSE_AA, peers = p.peer_up || p.peer_dn;
        const SparseKernel<T> k = aa ? sparse_aa_kernel<T, STRICT>(p.collision, moments, resid, peers, p.parity)
                                     : sparse_kernel<T, STRICT>(p.collision, moments, resid);
        if (!k) return cudaErrorInvalidValue;
        set_bases(sp);
        // threads: one warp per spw records (two-buffer), one per id (in-place, even step), one warp per record (odd step)
        const long long n = !aa ? (sp.seg_end - sp.seg_begin + sp.spw - 1) / sp.spw * 32
                                : p.parity == 0 ? sp.id_end - sp.id_begin : (sp.seg_end - sp.seg_begin) * 32;
        cfg.gridDim = dim3((unsigned)((n + SPARSE_BLOCK - 1) / SPARSE_BLOCK)), cfg.blockDim = dim3(SPARSE_BLOCK);
        cfg.numAttrs = (aa && !peers && p.pdl) ? 1 : 0;
        return cudaLaunchKernelEx(&cfg, k, sp);
    }
    const int mode = dense_mode(storage, p.parity);
    const DenseKernel<T> k = dense_kernel<T, STRICT>(p.collision, moments, resid, p.speculative, mode);
    if (!k) return cudaErrorInvalidValue;
    if (mode == MODE_AA_EVEN) set_bases<T, MODE_AA_EVEN>(p);
    else if (mode == MODE_AA_ODD) set_bases<T, MODE_AA_ODD>(p);
    else set_bases<T, MODE_AB>(p);
    cfg.gridDim = dim3((unsigned)((p.c_end - p.c_begin + DENSE_BLOCK - 1) / DENSE_BLOCK)), cfg.blockDim = dim3(DENSE_BLOCK);
    cfg.numAttrs = (mode != MODE_AB && p.pdl) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, k, p);
}

template <typename T, bool STRICT>
cudaError_t launch_persist(const SparseParams<T> &sp_in, int nsteps, int parity0, int moments_last, double *S, const T *pulse,
                           unsigned *barrier, int sm_count, cudaStream_t s) {
    const auto k = persist_kernel<T, STRICT>(sp_in.base.collision);
    if (!k) return cudaErrorInvalidValue;
    SparseParams<T> sp = sp_in;
    set_bases(sp);
    PersistArgs<T> pa{nsteps, parity0, moments_last, S ? 1 : 0, S, pulse, barrier};
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, PERSIST_BLOCK, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    per_sm = std::min(per_sm, sizeof(T) == 8 ? 1 : 2);
    const long long work = std::max((sp.id_end - sp.id_begin + 31) / 32 + 1, sp.seg_end - sp.seg_begin);
    // as many warps as give every warp the same number of rounds (an uneven last round makes everybody wait)
    const long long wpb = PERSIST_BLOCK / 32, max_blocks = std::min<long long>((long long)sm_count * per_sm, (long long)BAR_GROUP * 64);
    const long long rounds = std::max<long long>(1, (work + max_blocks * wpb - 1) / (max_blocks * wpb));
    const long long warps = (work + rounds - 1) / rounds;
    long long blocks = std::max<long long>(1, std::min(max_blocks, (warps + wpb - 1) / wpb));
    void *args[2] = {(void *)&sp, (void *)&pa};
    return cudaLaunchCooperativeKernel((const void *)k, dim3((unsigned)blocks), dim3(PERSIST_BLOCK), args, 0, s);
}

// With lazy module loading (the CUDA default) a kernel is loaded the first time it is launched -- 5 to 10 ms
// each for functions of this size, 18 ms of a 65 ms drivers/ldc run.  The run loops (lbm_run_fixed,
// lbm_run_converge) load the step kernels they are about to launch before they start their clock, by asking for
// their attributes; lbm_step keeps the lazy behaviour (it would load variants it may never use).  A run loop
// launches single-domain steps, with and without moments, summing |u| (resid) or not, both parities of an
// in-place storage -- or, persistent, only k_sparse_aa_persist.
template <typename T, bool STRICT>
cudaError_t preload_step_kernels(int storage, int collision, bool speculative, bool resid, bool persist) {
    cudaFuncAttributes a;
    auto load = [&](auto k) { return k ? cudaFuncGetAttributes(&a, k) : cudaErrorInvalidValue; };
    if (persist) return load(persist_kernel<T, STRICT>(collision));
    const int parities = storage == LBM_STORE_DENSE_AA || storage == LBM_STORE_SPARSE_AA ? 2 : 1;
    for (int parity = 0; parity < parities; parity++)
        for (bool moments : {false, true}) {
            cudaError_t e;
            if (storage == LBM_STORE_SPARSE_AB) e = load(sparse_kernel<T, STRICT>(collision, moments, resid));
            else if (storage == LBM_STORE_SPARSE_AA) e = load(sparse_aa_kernel<T, STRICT>(collision, moments, resid, false, parity));
            else e = load(dense_kernel<T, STRICT>(collision, moments, resid, speculative, dense_mode(storage, parity)));
            if (e != cudaSuccess) return e;
        }
    return cudaSuccess;
}

}  // namespace lbm
