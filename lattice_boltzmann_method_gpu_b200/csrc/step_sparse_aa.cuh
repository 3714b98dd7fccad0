// Fused step on the SPARSE IN-PLACE storage (LBM_STORE_SPARSE_AA): ONE population buffer in the
// reference's compact order (index_transform numbering, bifurcation.cu:241-252), AA-pattern streaming
// (Bailey et al. 2009), and every boundary link kept in the FLUID node's own slot.
//
//   even step (purely local):  f_k(x) = a[k][x]                      g_opp(k)(x) -> a[k][x]
//   odd step:                  f_k(x) = a[opp k][x - c_k]            g_opp(k)(x) -> a[opp k][x - c_k]
// i.e. each step reads and writes the SAME 19 addresses.  For a link k whose source x - c_k is not a
// fluid node the odd step uses the even step's address a[k][x] as well -- the node's own slot:
//   wall        : g_opp(k)(x) written there IS the half-way bounce-back value f_k(x) of the next step
//                 (bif:655-798), so a wall link costs one address select and no extra store;
//   inlet/outlet: the non-equilibrium extrapolation value (bif:877-1021) goes there instead of g_opp(k);
//   static      : the slot is simply never written -- it keeps the initial equilibrium of its source.
// Solid nodes are never read or written by a step (they only keep their place in the numbering), the
// scattered partial-sector stores into wall slots of the two-buffer sparse kernel are gone, and the even
// step needs no neighbour information at all: it is a straight pass over the compact arrays.
//
// The odd step takes neighbour ids from the same run-segment records as step_sparse.cuh, but only
// EIGHT of the 19 base ids: in the compact order the sources of the three directions that share a
// neighbouring row (same c_y, c_z) are consecutive ids, so one id per row -- that of the c_x = 0
// direction -- gives all three.
//
// Across z-slabs (fused peer stores): the even step copies the crossing populations of a face-plane node
// into the neighbour's halo replica of that node (slot opp q, what the neighbour's odd step pulls); the
// odd step stores g for a target in the halo plane straight into the neighbour's owned plane instead.
#pragma once
#include "step_sparse.cuh"

namespace lbm {

// resident CTAs per SM (128 threads each) of the local (even) and of the neighbour (odd) step; the odd one
// keeps 18 element indices next to the populations.  Measured choices: profiles/r02_notes.md
#ifndef LBM_SPAA64_MINB
#define LBM_SPAA64_MINB 6
#endif
#ifndef LBM_SPAA32_MINB
#define LBM_SPAA32_MINB 10
#endif
#ifndef LBM_SPAA64_ODD_MINB
#define LBM_SPAA64_ODD_MINB 5  // 96 registers, no spills: +1.2 % over 6 x 80 with 22 spilled words
#endif
#ifndef LBM_SPAA32_ODD_MINB
#define LBM_SPAA32_ODD_MINB 8  // 64 registers: +12 % over 10 x 48 with 43 spilled words
#endif

// neighbouring rows (c_y, c_z) != (0,0) of D3Q19 and the direction with c_x = 0 in each
__host__ __device__ constexpr int row_rep(int r) {
    constexpr int a[8] = {3, 4, 5, 6, 15, 16, 17, 18};
    return a[r];
}
__host__ __device__ constexpr int row_of(int k) {
    constexpr int a[Q] = {-1, -1, -1, 0, 1, 2, 3, 0, 1, 0, 1, 2, 3, 2, 3, 4, 5, 6, 7};
    return a[k];
}

// population load: plain, or (persistent kernel, where other SMs rewrote the element since this SM last
// read it and no kernel boundary has invalidated L1 in between) served by L2
template <bool CG, typename T>
__device__ __forceinline__ T ld_pop(const T *a) {
    return CG ? __ldcg(a) : *a;
}

// inlet / outlet links of a node, after its collision: the non-equilibrium extrapolation value
//     feq_q(rho_bc, u_bc(s)) + (g_q(x) - feq_q(rho_x, u_x)) (1 - 1/tau)          (bif:877-1021, step_dense.cuh)
// (under TRT the extrapolated part relaxes with both rates, as in step_dense.cuh boundary_node)
// goes into the node's own slot.  Which links, of which kind, with which prescribed speed was worked out once
// by k_bc_links (lbm_geo.cu); here the 18 directions are unrolled with compile-time q, so a boundary node costs
// a few dozen instructions per link instead of the ~3600-instruction generic path -- on a 64^3 grid the nodes
// under the lid / at the inlet otherwise set the duration of every step.
template <typename T, int COLL>
__device__ __forceinline__ void own_slot_bc(const SparseParams<T> &sp, long long i, T rho, T ux, T uy, T uz,
                                            const T (&f)[Q], T pulse) {
    const StepParams<T> &p = sp.base;
    const BcLink<T> *L = sp.bclinks + sp.bcslot[i];
    const uint32_t bcm = L[0].meta;
    const T r3 = rho / T(3.0), r18 = rho / T(18.0), r36 = rho / T(36.0);
    const T one = T(1.0);
    int e = 1;
#pragma unroll
    for (int q = 1; q < Q; q++) {
        if (!(bcm & (1u << q))) continue;
        const BcLink<T> l = L[e++];
        const int kind = (int)(l.meta & 3u), cs = (int)((l.meta >> 2) & 3u) - 1;
        T u = l.ubc;
        if (l.meta & 16u) u = u * pulse;
        const T feq = feq_lit<T>(q, r3, r18, r36, ux, uy, uz);
        T tmp;
        if (kind == LBM_BC_P) {
            tmp = feq_lit<T>(q, one / T(3.0), one / T(18.0), one / T(36.0), ux, uy, uz);
        } else {
            const T rw = kind == LBM_BC_V ? (q < 7 ? r18 : r36) : (q < 7 ? one / T(18.0) : one / T(36.0));
            tmp = feq_bc_axis<T>(rw, cs, u);
        }
        LBM_CHK(p, p.store_base[q] + i);
        if constexpr (COLL == LBM_COLL_TRT) {  // the rule of step_dense.cuh boundary_node
            const T nq = f[q] - feq, nb = f[oppq(q)] - feq_lit<T>(oppq(q), r3, r18, r36, ux, uy, uz);
            p.store_base[q][i] = tmp + (p.om1 * (T(0.5) * (nq + nb)) + p.om1_m * (T(0.5) * (nq - nb)));
        } else {
            p.store_base[q][i] = tmp + (f[q] - feq) * p.om1;
        }
    }
}

// per-step switches that are template parameters of the one-step kernels and run-time values of the
// persistent one
struct AaStep {
    bool moments, resid;
};

// the local (even) step of one node i in [sp.id_begin, sp.id_end)
template <typename T, bool STRICT, int COLL, bool PEERS, bool CG>
__device__ __forceinline__ void aa_even_node(const SparseParams<T> &sp, long long i, AaStep st, T pulse, double &velsum) {
    const StepParams<T> &p = sp.base;
    // one word per 32 ids says which lanes are fluid and whether any of them needs its node word at all
    // (walls need nothing in the local step): 0.25 B of metadata per node instead of 4
    uint2 cm = make_uint2(0u, 0u);
    if (i < sp.id_end) cm = sp.cmeta[i >> 5];
    if (!((cm.x >> (i & 31)) & 1u)) return;
    uint32_t node = 0u, rest = 0u;  // rest: links that are neither fluid-fed nor walls: inlet / outlet / static
    if (cm.y) node = sp.nodec[i];
    if (!CG) grid_dep_wait();
    T f[Q];
#pragma unroll
    for (int q = 0; q < Q; q++) {
        LBM_CHK(p, p.pull_base[q] + i);
        f[q] = ld_pop<CG>(p.pull_base[q] + i);
    }
    if ((node & NODE_LINKS) && !(node & NODE_WALLS_ONLY)) rest = node & NODE_LINKS & ~sp.wallc[i];
    T rho, ux, uy, uz;
    collide<T, STRICT, COLL>(f, p, rho, ux, uy, uz);
    if (rest == 0u) {
#pragma unroll
        for (int q = 0; q < Q; q++) {
            LBM_CHK(p, p.store_base[q] + i);
            p.store_base[q][i] = f[oppq(q)];
        }
    } else {
#pragma unroll
        for (int q = 0; q < Q; q++)
            if (!(rest & (1u << q))) {
                LBM_CHK(p, p.store_base[q] + i);
                p.store_base[q][i] = f[oppq(q)];
            }
        if (node & NODE_HAS_BC) own_slot_bc<T, COLL>(sp, i, rho, ux, uy, uz, f, pulse);
    }
    if (st.moments) {
        p.rho[i] = rho, p.ux[i] = ux, p.uy[i] = uy, p.uz[i] = uz;
    }
    if (st.resid) velsum += (double)(T)sqrt((double)(ux * ux + uy * uy + uz * uz));
    if (PEERS) push_to_peers<T, MODE_AA_EVEN>(p, i - p.face_c0, node, f);
}

// the neighbour (odd) step of one record: a whole warp calls this with the same `seg`
template <typename T, bool STRICT, int COLL, bool PEERS, bool CG>
__device__ __forceinline__ void aa_odd_record(const SparseParams<T> &sp, long long seg, AaStep st, T pulse, double &velsum) {
    const StepParams<T> &p = sp.base;
    const int lane = threadIdx.x & 31;
    const int32_t r0 = sp.rec[seg * SEG_REC + lane];
    const int32_t r1 = lane < SEG_REC - 32 ? sp.rec[seg * SEG_REC + 32 + lane] : 0;
    // the lane's node word travels with the record (no dependent load): link bits, NODE_SKIP when idle
    const uint32_t node = sp.rec_links[seg * 32 + lane];
    const int mB = __shfl_sync(0xffffffffu, r1, SEG_HALF + 19 - 32);
    const bool two = (mB >> 8) != 0;  // warp-uniform
    const bool inB = two && lane >= (mB & 255) && lane < (mB & 255) + (mB >> 8);
    const bool active = !(node & NODE_SKIP);
    const int i = __shfl_sync(0xffffffffu, r0, 0) + lane;  // compact id: the chunk's first id + lane in both pieces
    // compact id of the node at this lane's x in each of the 8 neighbouring rows
    int j[8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        int b = __shfl_sync(0xffffffffu, r0, row_rep(r));
        if (two) {
            const int bb = SEG_HALF + row_rep(r) < 32 ? __shfl_sync(0xffffffffu, r0, SEG_HALF + row_rep(r))
                                                      : __shfl_sync(0xffffffffu, r1, SEG_HALF + row_rep(r) - 32);
            b = inB ? bb : b;
        }
        j[r] = b + lane;
    }
    if (!active) return;
    if (!CG) grid_dep_wait();
    // ONE element index per direction, used for the load and for the store: inside the array of opp(k),
    // either the source's id or -- for a link -- this node's own slot in the array of k, which lies
    // dk[k] = (k - opp k) * qstride elements away
    int idx[Q];
    T f[Q];
    LBM_CHK(p, p.pull_base[0] + i);
    f[0] = ld_pop<CG>(p.pull_base[0] + i);
#pragma unroll
    for (int k = 1; k < Q; k++) {
        const int n = (k < 3 ? i : j[row_of(k) < 0 ? 0 : row_of(k)]) - cxq(k);
        idx[k] = (node & (1u << k)) ? i + sp.dk[k] : n;
        LBM_CHK(p, p.pull_base[oppq(k)] + idx[k]);
        f[k] = ld_pop<CG>(p.pull_base[oppq(k)] + idx[k]);
    }
    uint32_t rest = 0u;
    if ((node & NODE_LINKS) && !(node & NODE_WALLS_ONLY)) rest = node & NODE_LINKS & ~sp.wallc[i];
    T rho, ux, uy, uz;
    collide<T, STRICT, COLL>(f, p, rho, ux, uy, uz);
    LBM_CHK(p, p.store_base[0] + i);
    p.store_base[0][i] = f[0];
#pragma unroll
    for (int k = 1; k < Q; k++) {
        if (rest & (1u << k)) continue;  // inlet / outlet (written below) or static (kept) link
        if (PEERS && !(node & (1u << k))) {
            if (czq(k) > 0 && p.peer_dn && idx[k] < sp.halo_lo_n) {
                // the target x - c_k lies in the low halo plane: it is a node the neighbour below owns
                p.peer_dn[(long long)oppq(k) * p.peer_dn_qs + p.peer_dn_own + idx[k]] = f[oppq(k)];
                continue;
            }
            if (czq(k) < 0 && p.peer_up && idx[k] >= sp.halo_hi0) {
                p.peer_up[(long long)oppq(k) * p.peer_up_qs + p.peer_up_own + (idx[k] - sp.halo_hi0)] = f[oppq(k)];
                continue;
            }
        }
        LBM_CHK(p, p.store_base[oppq(k)] + idx[k]);
        p.store_base[oppq(k)][idx[k]] = f[oppq(k)];
    }
    if (rest && (node & NODE_HAS_BC)) own_slot_bc<T, COLL>(sp, i, rho, ux, uy, uz, f, pulse);
    if (st.moments) {
        p.rho[i] = rho, p.ux[i] = ux, p.uy[i] = uy, p.uz[i] = uz;
    }
    if (st.resid) velsum += (double)(T)sqrt((double)(ux * ux + uy * uy + uz * uz));
}

// sum|u| of a CTA into one atomic: on a small grid thousands of same-address atomics per step serialise in L2
// and cost more than the step itself.  Every thread of the CTA must call this.
template <int NWARPS>
__device__ __forceinline__ void cta_add(double *dst, double v) {
    __shared__ double ws[NWARPS];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < NWARPS; w++) t += ws[w];
        if (t != 0.0) atomicAdd(dst, t);
    }
}

template <typename T, bool STRICT, int COLL, bool MOMENTS, bool RESID, bool PEERS>
__global__ void __launch_bounds__(SPARSE_BLOCK, sizeof(T) == 8 ? LBM_SPAA64_MINB : LBM_SPAA32_MINB)
    k_sparse_aa_even(const __grid_constant__ SparseParams<T> sp) {
    grid_dep_launch();
    const long long i = sp.id_begin + (long long)blockIdx.x * SPARSE_BLOCK + threadIdx.x;
    double velsum = 0.0;
    aa_even_node<T, STRICT, COLL, PEERS, false>(sp, i, AaStep{MOMENTS, RESID}, sp.base.pulse_scale, velsum);
    if (RESID) cta_add<SPARSE_BLOCK / 32>(sp.base.resid, velsum);
}

template <typename T, bool STRICT, int COLL, bool MOMENTS, bool RESID, bool PEERS>
__global__ void __launch_bounds__(SPARSE_BLOCK, sizeof(T) == 8 ? LBM_SPAA64_ODD_MINB : LBM_SPAA32_ODD_MINB)
    k_sparse_aa_odd(const __grid_constant__ SparseParams<T> sp) {
    grid_dep_launch();
    const long long seg = sp.seg_begin + (long long)blockIdx.x * (SPARSE_BLOCK / 32) + (threadIdx.x >> 5);
    double velsum = 0.0;
    if (seg < sp.seg_end)  // warp-uniform
        aa_odd_record<T, STRICT, COLL, PEERS, false>(sp, seg, AaStep{MOMENTS, RESID}, sp.base.pulse_scale, velsum);
    if (RESID) cta_add<SPARSE_BLOCK / 32>(sp.base.resid, velsum);
}

// ---------------------------------------------------------------------------------------------------------
// Persistent form for grids that live in L2 (64^3 and the like: the reference's own configurations).
// There a time step moves a few MB, so a launch per step spends most of its time in launch latency and in
// the tail of its last wave.  ONE cooperative launch runs `nsteps` steps: every warp walks its share of
// the chunks (even step) or records (odd step), then all CTAs meet at a grid barrier (one monotonic counter
// in global memory; co-residency is guaranteed by cudaLaunchCooperativeKernel).  Populations are read with
// ld.global.cg: between two steps other SMs rewrote them and no kernel boundary invalidated L1.
// Per-step values that the one-step kernels get as launch parameters come from small tables: the
// pulsatile inlet scale of step s (computed by the host exactly as for single launches) and the slot S[s]
// that receives sum|u| of that step.
template <typename T>
struct PersistArgs {
    int nsteps, parity0;
    int moments_last, resid;
    double *S;          // [nsteps] when resid
    const T *pulse;     // [nsteps] or null (scale 1)
    unsigned *barrier;  // BAR_WORDS words, zero at launch
};
// Grid barrier, generation `gen` = 1, 2, ... (counters are monotonic, never reset inside a launch).
// Same-address atomics serialise in L2 at ~27 cycles each and polling loads queue behind them, so a single
// counter for ~300 CTAs made the barrier cost more than the step (19 us per 64^3 step).  Two levels: CTAs
// arrive on the counter of their group of 16, the last arriver of a group arrives on the top counter, the
// last of those publishes `gen` in a release word that everybody polls with plain L1-bypassing loads.
// Every counter sits in its own 128-byte line: bar[0] release, bar[32] top, bar[64 + 32 g] group g.
constexpr int BAR_GROUP = 16, BAR_WORDS = 64 + 32 * 64;
__device__ __forceinline__ void grid_barrier(unsigned *bar, unsigned gen) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned g = blockIdx.x / BAR_GROUP, ngroups = (gridDim.x + BAR_GROUP - 1) / BAR_GROUP;
        const unsigned gsize = min((unsigned)BAR_GROUP, gridDim.x - g * BAR_GROUP);
        if (atomicAdd(bar + 64 + 32 * g, 1u) == gen * gsize - 1u) {
            if (atomicAdd(bar + 32, 1u) == gen * ngroups - 1u) {
                asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(bar), "r"(gen) : "memory");
            }
        }
        unsigned v;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
        } while (v < gen);
    }
    __syncthreads();
}
// Few, large CTAs: the barrier costs one atomic and one polling thread per CTA, all on one L2 line --
// 1480 CTAs of 128 threads made a step 19 us, one or two CTAs of 512 threads per SM keep it near the L2
// round trip (profiles/r02_notes.md).
constexpr int PERSIST_BLOCK = 512;
template <typename T, bool STRICT, int COLL>
__global__ void __launch_bounds__(PERSIST_BLOCK, sizeof(T) == 8 ? 1 : 2)
    k_sparse_aa_persist(const __grid_constant__ SparseParams<T> sp, const __grid_constant__ PersistArgs<T> pa) {
    const long long warp0 = (long long)blockIdx.x * (PERSIST_BLOCK / 32) + (threadIdx.x >> 5);
    const long long nwarps = (long long)gridDim.x * (PERSIST_BLOCK / 32);
    const int lane = threadIdx.x & 31;
    const long long first_chunk = sp.id_begin >> 5, end_chunk = (sp.id_end + 31) >> 5;
    for (int s = 0; s < pa.nsteps; s++) {
        const AaStep st{pa.moments_last && s == pa.nsteps - 1, pa.resid != 0};
        const T pulse = pa.pulse ? pa.pulse[s] : T(1.0);
        double velsum = 0.0;
        if (((pa.parity0 + s) & 1) == 0) {
            for (long long c = first_chunk + warp0; c < end_chunk; c += nwarps) {
                const long long i = c * 32 + lane;
                if (i >= sp.id_begin) aa_even_node<T, STRICT, COLL, false, true>(sp, i, st, pulse, velsum);
            }
        } else {
            for (long long seg = sp.seg_begin + warp0; seg < sp.seg_end; seg += nwarps)
                aa_odd_record<T, STRICT, COLL, false, true>(sp, seg, st, pulse, velsum);
        }
        if (st.resid) cta_add<PERSIST_BLOCK / 32>(pa.S + s, velsum);
        if (s + 1 < pa.nsteps) grid_barrier(pa.barrier, (unsigned)(s + 1));
    }
}

}  // namespace lbm
