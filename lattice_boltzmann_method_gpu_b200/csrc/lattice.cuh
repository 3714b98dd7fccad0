// D3Q19 lattice constants and the per-node collision arithmetic (BGK, TRT), device side.
//
// Lattice numbering, weights and opposite pairs follow the reference's pull
// offsets and swap list (ldc.cu:184-201, 207-313, 320-322; SURVEY A.1).
//
// Two arithmetic policies (lbm_math in include/lbm_b200.h):
//   STRICT : the reference's expression order (bif.cu:574-634), compiled in a
//            translation unit built with -fmad=false, so results are
//            bit-identical to the CPU oracle (gcc -ffp-contract=off).
//   FAST   : algebraically equal, reciprocal-multiply form with EXPLICIT fma()s (its translation
//            unit is built with -fmad=false as well) -- the measured path.  Agreement with
//            STRICT is tolerance-tested; every kernel variant agrees with every other bit for bit.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "lbm_internal.h"

namespace lbm {



__host__ __device__ constexpr int cxq(int q) {
    constexpr int a[Q] = {0, 1, -1, 0, 0, 0, 0, 1, 1, -1, -1, 1, 1, -1, -1, 0, 0, 0, 0};
    return a[q];
}
__host__ __device__ constexpr int cyq(int q) {
    constexpr int a[Q] = {0, 0, 0, 1, -1, 0, 0, 1, -1, 1, -1, 0, 0, 0, 0, 1, -1, 1, -1};
    return a[q];
}
__host__ __device__ constexpr int czq(int q) {
    constexpr int a[Q] = {0, 0, 0, 0, 0, 1, -1, 0, 0, 0, 0, 1, -1, 1, -1, 1, 1, -1, -1};
    return a[q];
}
__host__ __device__ constexpr int oppq(int q) {
    constexpr int a[Q] = {0, 2, 1, 4, 3, 6, 5, 10, 9, 8, 7, 14, 13, 12, 11, 18, 17, 16, 15};
    return a[q];
}
// the 5 directions with c_z = +1 (and, same order, their counterparts with c_z = -1) numbered 0..4: slot of a
// crossing population in a slab's mailbox
__host__ __device__ constexpr int kslot(int q) {
    constexpr int a[Q] = {-1, -1, -1, -1, -1, 0, 0, -1, -1, -1, -1, 1, 1, 2, 2, 3, 4, 3, 4};
    return a[q];
}
__host__ __device__ constexpr int caxis(int q, int axis) { return axis == 0 ? cxq(q) : (axis == 1 ? cyq(q) : czq(q)); }

// ---------------------------------------------------------------------------
// literal ("strict") equilibrium forms, one per direction family
// ---------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T feq_rest_lit(T rw, T ux, T uy, T uz) {
    return rw * (T(1.0) - T(1.5) * ux * ux - T(1.5) * uy * uy - T(1.5) * uz * uz);
}
template <typename T>
__device__ __forceinline__ T feq_axis_lit(T rw, int sgn, T ua, T ub, T uc) {
    T t = sgn > 0 ? T(1.0) + T(3.0) * ua : T(1.0) - T(3.0) * ua;
    return rw * (t + T(3.0) * ua * ua - T(1.5) * ub * ub - T(1.5) * uc * uc);
}
// form 0: +3(ua+ub), +9uaub   1: +3(ua-ub), -9uaub   2: +3(ub-ua), -9uaub   3: -3(ua+ub), +9uaub
template <typename T>
__device__ __forceinline__ T feq_diag_lit(T rw, int form, T ua, T ub, T uc) {
    T t;
    if (form == 0) t = T(1.0) + T(3.0) * (ua + ub);
    else if (form == 1) t = T(1.0) + T(3.0) * (ua - ub);
    else if (form == 2) t = T(1.0) + T(3.0) * (ub - ua);
    else t = T(1.0) - T(3.0) * (ua + ub);
    t = t + T(3.0) * ua * ua + T(3.0) * ub * ub;
    if (form == 0 || form == 3) t = t + T(9.0) * ua * ub;
    else t = t - T(9.0) * ua * ub;
    return rw * (t - T(1.5) * uc * uc);
}
// Direction 14 is evaluated partly in double in every copy of the reference
// (a `3.0` literal without the f suffix: ldc.cu:344, pos:557, bif:625, cor:540).
template <typename T>
__device__ __forceinline__ T feq_14_lit(T rw, T ux, T uy, T uz) {
    T head = T(1.0) - T(3.0) * (ux + uz) + T(3.0) * ux * ux;
    double t = (double)head + 3.0 * (double)uz * (double)uz;
    t = t + (double)(T(9.0) * ux * uz);
    t = t - (double)(T(1.5) * uy * uy);
    return (T)((double)rw * t);
}
// q may be a runtime value (boundary path) or a literal (unrolled fluid path)
template <typename T>
__device__ __forceinline__ T feq_lit(int q, T r3, T r18, T r36, T ux, T uy, T uz) {
    switch (q) {
    case 0: return feq_rest_lit(r3, ux, uy, uz);
    case 1: return feq_axis_lit(r18, +1, ux, uy, uz);
    case 2: return feq_axis_lit(r18, -1, ux, uy, uz);
    case 3: return feq_axis_lit(r18, +1, uy, ux, uz);
    case 4: return feq_axis_lit(r18, -1, uy, ux, uz);
    case 5: return feq_axis_lit(r18, +1, uz, ux, uy);
    case 6: return feq_axis_lit(r18, -1, uz, ux, uy);
    case 7: return feq_diag_lit(r36, 0, ux, uy, uz);
    case 8: return feq_diag_lit(r36, 1, ux, uy, uz);
    case 9: return feq_diag_lit(r36, 2, ux, uy, uz);
    case 10: return feq_diag_lit(r36, 3, ux, uy, uz);
    case 11: return feq_diag_lit(r36, 0, ux, uz, uy);
    case 12: return feq_diag_lit(r36, 1, ux, uz, uy);
    case 13: return feq_diag_lit(r36, 2, ux, uz, uy);
    case 14: return feq_14_lit(r36, ux, uy, uz);
    case 15: return feq_diag_lit(r36, 0, uy, uz, ux);
    case 16: return feq_diag_lit(r36, 2, uy, uz, ux);
    case 17: return feq_diag_lit(r36, 1, uy, uz, ux);
    default: return feq_diag_lit(r36, 3, uy, uz, ux);
    }
}

// factored form used only by the LDC initial state (ldc.cu:542-571)
template <typename T>
__device__ __forceinline__ void feq_all_ldc_init(T rho, T ux, T uy, T uz, T *feq) {
    const T w0 = T(1.0) / T(3.0), w1 = T(1.0) / T(18.0), w2 = T(1.0) / T(36.0);
    T ux2 = ux * ux, uy2 = uy * uy, uz2 = uz * uz;
    T u2 = ux2 + uy2 + uz2, xy2 = ux2 + uy2, xz2 = ux2 + uz2, yz2 = uy2 + uz2;
    T xy = T(2.0) * ux * uy, xz = T(2.0) * ux * uz, yz = T(2.0) * uy * uz;
    feq[0] = rho * w0 * (T(1.0) - T(1.5) * u2);
    feq[1] = rho * w1 * (T(1.0) + T(3.0) * ux + T(4.5) * ux2 - T(1.5) * u2);
    feq[2] = rho * w1 * (T(1.0) - T(3.0) * ux + T(4.5) * ux2 - T(1.5) * u2);
    feq[3] = rho * w1 * (T(1.0) + T(3.0) * uy + T(4.5) * uy2 - T(1.5) * u2);
    feq[4] = rho * w1 * (T(1.0) - T(3.0) * uy + T(4.5) * uy2 - T(1.5) * u2);
    feq[5] = rho * w1 * (T(1.0) + T(3.0) * uz + T(4.5) * uz2 - T(1.5) * u2);
    feq[6] = rho * w1 * (T(1.0) - T(3.0) * uz + T(4.5) * uz2 - T(1.5) * u2);
    feq[7] = rho * w2 * (T(1.0) + T(3.0) * (ux + uy) + T(4.5) * (xy2 + xy) - T(1.5) * u2);
    feq[8] = rho * w2 * (T(1.0) + T(3.0) * (ux - uy) + T(4.5) * (xy2 - xy) - T(1.5) * u2);
    feq[9] = rho * w2 * (T(1.0) + T(3.0) * (uy - ux) + T(4.5) * (xy2 - xy) - T(1.5) * u2);
    feq[10] = rho * w2 * (T(1.0) - T(3.0) * (ux + uy) + T(4.5) * (xy2 + xy) - T(1.5) * u2);
    feq[11] = rho * w2 * (T(1.0) + T(3.0) * (ux + uz) + T(4.5) * (xz2 + xz) - T(1.5) * u2);
    feq[12] = rho * w2 * (T(1.0) + T(3.0) * (ux - uz) + T(4.5) * (xz2 - xz) - T(1.5) * u2);
    feq[13] = rho * w2 * (T(1.0) + T(3.0) * (uz - ux) + T(4.5) * (xz2 - xz) - T(1.5) * u2);
    feq[14] = rho * w2 * (T(1.0) - T(3.0) * (ux + uz) + T(4.5) * (xz2 + xz) - T(1.5) * u2);
    feq[15] = rho * w2 * (T(1.0) + T(3.0) * (uy + uz) + T(4.5) * (yz2 + yz) - T(1.5) * u2);
    feq[16] = rho * w2 * (T(1.0) + T(3.0) * (uz - uy) + T(4.5) * (yz2 - yz) - T(1.5) * u2);
    feq[17] = rho * w2 * (T(1.0) + T(3.0) * (uy - uz) + T(4.5) * (yz2 - yz) - T(1.5) * u2);
    feq[18] = rho * w2 * (T(1.0) - T(3.0) * (uy + uz) + T(4.5) * (yz2 + yz) - T(1.5) * u2);
}

// r / d for d in {3, 18} without a division: with hi + lo = 1/d to twice the working precision,
//   p = r*hi,  e = fma(r, hi, -p) (the exact rounding error of p),  result = p + (e + r*lo)
// is r/d rounded once (up to rare ties) -- 4 dependent instructions instead of ~10 / ~25.
// (Adding r*lo to the ROUNDED p alone changes nothing: lo is below half an ulp of hi.)
template <typename T>
__device__ __forceinline__ T div_by_const(T r, T hi, T lo) {
    const T p = r * hi;
    return p + fma(r, lo, fma(r, hi, -p));
}
template <typename T>
__device__ __forceinline__ T rho_over(T r, int d);
template <>
__device__ __forceinline__ float rho_over<float>(float r, int d) {
    constexpr float h3 = (float)(1.0 / 3.0), l3 = (float)(1.0 / 3.0 - (double)h3);
    constexpr float h18 = (float)(1.0 / 18.0), l18 = (float)(1.0 / 18.0 - (double)h18);
    return d == 3 ? div_by_const<float>(r, h3, l3) : div_by_const<float>(r, h18, l18);
}
template <>
__device__ __forceinline__ double rho_over<double>(double r, int d) {
    // 1/3 - fl(1/3) and 1/18 - fl(1/18), exact to double precision
    constexpr double h3 = 0x1.5555555555555p-2, l3 = 0x1.5555555555555p-56;
    constexpr double h18 = 0x1.c71c71c71c71cp-5, l18 = 0x1.c71c71c71c71cp-59;
    return d == 3 ? div_by_const<double>(r, h3, l3) : div_by_const<double>(r, h18, l18);
}

// ---------------------------------------------------------------------------
// moments of one node in FAST arithmetic, shared by both FAST collisions (collide_bgk, collide_trt).
// ---------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void moments_fast(const T (&f)[Q], T &rho, T &ux, T &uy, T &uz) {
    // pairwise sums shorten the dependency chains; order is free in FAST mode.
    // Every multiply-add below is an EXPLICIT fma and the translation unit is compiled with -fmad=false
    // like the STRICT one: which operations fuse is then decided here, not by ptxas per kernel
    // instantiation, so all storages, the persistent kernel, the two-segment kernel and the slab (peer
    // store) variants produce the same bits from the same inputs -- "N slabs == 1 domain" and
    // "in-place == two buffers" hold bit for bit in FAST arithmetic too.
    T a0 = f[1] + f[2], a1 = f[3] + f[4], a2 = f[5] + f[6];
    T d0 = f[7] + f[10], d1 = f[8] + f[9], d2 = f[11] + f[14], d3 = f[12] + f[13], d4 = f[15] + f[18],
      d5 = f[16] + f[17];
    T r = ((f[0] + a0) + (a1 + a2)) + ((d0 + d1) + (d2 + d3)) + (d4 + d5);
    T inv = T(1.0) / r;
    T mx = ((f[1] - f[2]) + (f[7] - f[10])) + ((f[8] - f[9]) + (f[11] - f[14])) + (f[12] - f[13]);
    T my = ((f[3] - f[4]) + (f[7] - f[10])) + ((f[9] - f[8]) + (f[15] - f[18])) + (f[17] - f[16]);
    T mz = ((f[5] - f[6]) + (f[11] - f[14])) + ((f[13] - f[12]) + (f[15] - f[18])) + (f[16] - f[17]);
    rho = r;
    ux = mx * inv, uy = my * inv, uz = mz * inv;
}

// ---------------------------------------------------------------------------
// moments + BGK collision of one node.  f[] in: post-streaming populations,
// out: post-collision.  Moments returned are the pre-collision ones the
// reference stores (bif.cu:574-595).
// ---------------------------------------------------------------------------
template <typename T, bool STRICT>
__device__ __forceinline__ void collide_bgk(T (&f)[Q], T tau, T inv_tau, T &rho, T &ux, T &uy, T &uz) {
    if constexpr (STRICT) {
        T r = T(0.0);
#pragma unroll
        for (int q = 0; q < Q; q++) r = r + f[q];
        rho = r;
        ux = (f[1] - f[2] + f[7] + f[8] - f[9] - f[10] + f[11] + f[12] - f[13] - f[14]) / r;
        uy = (f[3] - f[4] + f[7] - f[8] + f[9] - f[10] + f[15] - f[16] + f[17] - f[18]) / r;
        uz = (f[5] - f[6] + f[11] - f[12] + f[13] - f[14] + f[15] + f[16] - f[17] - f[18]) / r;
        const T r3 = r / T(3.0), r18 = r / T(18.0), r36 = r / T(36.0);
#pragma unroll
        for (int q = 0; q < Q; q++) {
            T feq = feq_lit<T>(q, r3, r18, r36, ux, uy, uz);
            f[q] = f[q] - (f[q] - feq) / tau;
        }
    } else {
        moments_fast<T>(f, rho, ux, uy, uz);
        const T r = rho;
        // f* = f + om (feq - f): the difference is formed first, like the reference's
        // f - (f - feq)/tau, so the rounding error scales with the (small) non-equilibrium
        // part.  The algebraically equal (1-om) f + om feq cancels two O(f) terms when
        // tau < 1 and is 3-10x less accurate in fp32 (measured, profiles/r01_notes.md).
        const T om = inv_tau;
        // feq_q = rho w_q (1 + 3cu + 4.5cu^2 - 1.5u^2)
        const T base = fma(T(-1.5), fma(ux, ux, fma(uy, uy, uz * uz)), T(1.0));
        // rho w_q must not carry a systematic error: multiplying by a rounded 1/18 gives every cell
        // the same signed error in sum_q feq_q, i.e. a coherent mass drift of ~2 ulp per step
        // (visible in fp32 after 1000 steps; the reference divides, rho/18).  A division costs
        // ~10 (fp32) / ~25 (fp64) dependent instructions on a latency-bound kernel, so the weight is
        // applied as an error-free two-term product instead (rho_over).
        const T k0 = rho_over<T>(r, 3), k1 = rho_over<T>(r, 18), k2 = T(0.5) * k1;
        f[0] = fma(om, fma(k0, base, -f[0]), f[0]);
#define LBM_PAIR(qp, qm, cu, kw)                                    \
    {                                                               \
        T cu_ = (cu);                                               \
        T even = fma(T(4.5) * cu_, cu_, base);                      \
        T odd = T(3.0) * cu_;                                       \
        f[qp] = fma(om, fma((kw), even + odd, -f[qp]), f[qp]);      \
        f[qm] = fma(om, fma((kw), even - odd, -f[qm]), f[qm]);      \
    }
        LBM_PAIR(1, 2, ux, k1)
        LBM_PAIR(3, 4, uy, k1)
        LBM_PAIR(5, 6, uz, k1)
        LBM_PAIR(7, 10, ux + uy, k2)
        LBM_PAIR(8, 9, ux - uy, k2)
        LBM_PAIR(11, 14, ux + uz, k2)
        LBM_PAIR(12, 13, ux - uz, k2)
        LBM_PAIR(15, 18, uy + uz, k2)
        LBM_PAIR(17, 16, uy - uz, k2)
#undef LBM_PAIR
    }
}

// ---------------------------------------------------------------------------
// moments + two-relaxation-time (TRT) collision of one node, FAST arithmetic only (Ginzburg, Verhaeghe &
// d'Humieres, Commun. Comput. Phys. 3, 2008).  For an opposite pair (q, qbar) the non-equilibrium splits
// into an even and an odd part,
//     n+ = (f_q + f_qbar)/2 - kw even      n- = (f_q - f_qbar)/2 - kw odd
//     f_q <- f_q - om_p n+ - om_m n-       f_qbar <- f_qbar - om_p n+ + om_m n-
// with the equilibrium parts even / odd of collide_bgk's LBM_PAIR.  om_p = 1/tau keeps the viscosity;
// om_m is set by the host from the magic parameter Lambda = (1/om_p - 1/2)(1/om_m - 1/2).  Moments returned
// are the pre-collision ones, as for collide_bgk.
// ---------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void collide_trt(T (&f)[Q], T om_p, T om_m, T &rho, T &ux, T &uy, T &uz) {
    moments_fast<T>(f, rho, ux, uy, uz);
    const T r = rho;
    const T base = fma(T(-1.5), fma(ux, ux, fma(uy, uy, uz * uz)), T(1.0));
    const T k0 = rho_over<T>(r, 3), k1 = rho_over<T>(r, 18), k2 = T(0.5) * k1;
    f[0] = fma(om_p, fma(k0, base, -f[0]), f[0]);
#define LBM_PAIR_TRT(qp, qm, cu, kw)                                  \
    {                                                                 \
        T cu_ = (cu);                                                 \
        T even = fma(T(4.5) * cu_, cu_, base);                        \
        T odd = T(3.0) * cu_;                                         \
        T np = fma(-(kw), even, T(0.5) * (f[qp] + f[qm]));            \
        T nm = fma(-(kw), odd, T(0.5) * (f[qp] - f[qm]));             \
        T rp = om_p * np;                                             \
        f[qp] = fma(-om_m, nm, f[qp] - rp);                           \
        f[qm] = fma(om_m, nm, f[qm] - rp);                            \
    }
    LBM_PAIR_TRT(1, 2, ux, k1)
    LBM_PAIR_TRT(3, 4, uy, k1)
    LBM_PAIR_TRT(5, 6, uz, k1)
    LBM_PAIR_TRT(7, 10, ux + uy, k2)
    LBM_PAIR_TRT(8, 9, ux - uy, k2)
    LBM_PAIR_TRT(11, 14, ux + uz, k2)
    LBM_PAIR_TRT(12, 13, ux - uz, k2)
    LBM_PAIR_TRT(15, 18, uy + uz, k2)
    LBM_PAIR_TRT(17, 16, uy - uz, k2)
#undef LBM_PAIR_TRT
}

// one collision of the fused step kernels, chosen at compile time: COLL is an lbm_collision value
template <typename T, bool STRICT, int COLL>
__device__ __forceinline__ void collide(T (&f)[Q], const StepParams<T> &p, T &rho, T &ux, T &uy, T &uz) {
    static_assert(COLL == LBM_COLL_BGK || !STRICT, "TRT exists in FAST arithmetic only");
    if constexpr (COLL == LBM_COLL_TRT) collide_trt<T>(f, p.inv_tau, p.om_m, rho, ux, uy, uz);
    else collide_bgk<T, STRICT>(f, p.tau, p.inv_tau, rho, ux, uy, uz);
}

}  // namespace lbm
