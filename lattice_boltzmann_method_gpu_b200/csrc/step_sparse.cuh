// Fused step on the SPARSE storage: populations, moments and node words live in the reference's own
// compact order (one entry per stored node, index_transform numbering, bifurcation.cu:241-252), two
// buffers, addressed through run-segment records instead of a per-node neighbour list.
//
// One warp = one segment = one aligned chunk of 32 compact ids, holding up to two "pieces" (the tail
// of one row's run of fluid nodes and the head of the next; lbm_geo.cu, k_seg_fill).  For each
// direction the sources of a piece are one contiguous range of compact ids, so the warp needs the
// record's 19 base ids per piece (one 192-byte load, broadcast by shuffles) and then issues 19 coalesced
// loads -- 6 B of index traffic per node instead of the 72 B of an 18-entry neighbour list -- and 19
// stores that are full aligned 256-byte rows (fp64) of the destination arrays.
//
// Boundary links work exactly as in step_dense.cuh: the slot of link q is the pull source itself,
// dst[q][base_q + lane] -- wall, inlet/outlet and -1 nodes ARE stored nodes in this layout, as in the
// reference.  The slow path (inlet/outlet/lid/static) is the same out-of-line function, fed with the
// node's Cartesian cell id from the record.
#pragma once
#include "step_dense.cuh"

namespace lbm {

constexpr int SPARSE_BLOCK = 128;
#ifndef LBM_SP64_MINB
#define LBM_SP64_MINB 5
#endif
#ifndef LBM_SP32_MINB
#define LBM_SP32_MINB 10
#endif

template <typename T, bool STRICT, int COLL, bool MOMENTS, bool RESID>
__global__ void __launch_bounds__(SPARSE_BLOCK, sizeof(T) == 8 ? LBM_SP64_MINB : LBM_SP32_MINB)
    k_step_sparse(const __grid_constant__ SparseParams<T> sp) {
    const StepParams<T> &p = sp.base;
    const int lane = threadIdx.x & 31;
    // a warp walks `spw` consecutive records; the next record is fetched while the current one is
    // processed, so only the first record load of a warp is exposed in front of the 19 pulls
    long long seg = sp.seg_begin + ((long long)blockIdx.x * (SPARSE_BLOCK / 32) + (threadIdx.x >> 5)) * sp.spw;
    const long long seg_last = (seg + sp.spw < sp.seg_end ? seg + sp.spw : sp.seg_end) - 1;
    if (seg > seg_last) return;
    int32_t r0 = sp.rec[seg * SEG_REC + lane];
    int32_t r1 = lane < SEG_REC - 32 ? sp.rec[seg * SEG_REC + 32 + lane] : 0;
    double velsum = 0.0;
    for (; seg <= seg_last; seg++) {
        int32_t n0 = 0, n1 = 0;
        if (seg < seg_last) {
            n0 = sp.rec[(seg + 1) * SEG_REC + lane];
            if (lane < SEG_REC - 32) n1 = sp.rec[(seg + 1) * SEG_REC + 32 + lane];
        }
        const int mA = __shfl_sync(0xffffffffu, r0, 19), mB = __shfl_sync(0xffffffffu, r1, SEG_HALF + 19 - 32);
        const bool two = (mB >> 8) != 0;  // warp-uniform
        const bool inB = two && lane >= (mB & 255) && lane < (mB & 255) + (mB >> 8);
        const bool active = inB || (lane >= (mA & 255) && lane < (mA & 255) + (mA >> 8));
        unsigned clo = (unsigned)__shfl_sync(0xffffffffu, r0, 20), chi = (unsigned)__shfl_sync(0xffffffffu, r0, 21);
        int has_links = __shfl_sync(0xffffffffu, r0, 22);
        if (two) {
            const unsigned blo = (unsigned)__shfl_sync(0xffffffffu, r1, SEG_HALF + 20 - 32);
            const unsigned bhi = (unsigned)__shfl_sync(0xffffffffu, r1, SEG_HALF + 21 - 32);
            const int bl = __shfl_sync(0xffffffffu, r1, SEG_HALF + 22 - 32);
            if (inB) clo = blo, chi = bhi, has_links = bl;
        }
        const int i = __shfl_sync(0xffffffffu, r0, 0) + lane;  // compact id: the chunk's first id + lane in both pieces
        uint32_t node = 0u, wl = 0u;
        if (active && has_links) {
            node = sp.nodec[i];
            wl = sp.wallc[i];
        }
        // the 19 source ids are used once (they do not stay in registers next to the populations)
        T f[Q];
        if (!two) {  // warp-uniform: one region around all 19 pulls, not one per direction
#pragma unroll
            for (int q = 0; q < Q; q++) {
                const int bq = __shfl_sync(0xffffffffu, r0, q);
                // idle lanes read their own (stored, unused) slot: no branch between the shuffles
                if (active) LBM_CHK(p, p.pull_base[q] + (bq + lane));  // the idle lanes' dummy reads are not the pull
                f[q] = ld_stream(p.pull_base[q] + (active ? bq + lane : i));
            }
        } else {
#pragma unroll
            for (int q = 0; q < Q; q++) {
                const int ba = __shfl_sync(0xffffffffu, r0, q);
                const int bb = SEG_HALF + q < 32 ? __shfl_sync(0xffffffffu, r0, SEG_HALF + q)
                                                 : __shfl_sync(0xffffffffu, r1, SEG_HALF + q - 32);
                if (active) LBM_CHK(p, p.pull_base[q] + ((inB ? bb : ba) + lane));
                f[q] = ld_stream(p.pull_base[q] + (active ? (inB ? bb : ba) + lane : i));
            }
        }
        T rho, ux, uy, uz;
        if (active) {
            collide<T, STRICT, COLL>(f, p, rho, ux, uy, uz);
#pragma unroll
            for (int q = 0; q < Q; q++) {
                LBM_CHK(p, p.store_base[q] + i);
                p.store_base[q][i] = f[q];
            }
            if (MOMENTS) {
                p.rho[i] = rho, p.ux[i] = ux, p.uy[i] = uy, p.uz[i] = uz;
            }
            if (RESID) velsum += (double)(T)sqrt((double)(ux * ux + uy * uy + uz * uz));
            if (p.peer_up || p.peer_dn) push_to_peers<T, MODE_AB>(p, (long long)i - p.face_c0, node, f);  // compact ids: a plane is one id range
            if (node & NODE_LINKS) {
                // boundary slots are the pull sources themselves; the few lanes that have links re-read
                // their piece's base ids from the record (L1-resident by now)
                const int32_t *mine = sp.rec + seg * SEG_REC + (inB ? SEG_HALF : 0);
                wl = (node & NODE_WALLS_ONLY) ? (node & NODE_LINKS) : (wl & node & NODE_LINKS);
#pragma unroll
                for (int q = 1; q < Q; q++)
                    if (wl & (1u << q)) {
                        LBM_CHK(p, p.store_base[q] + (mine[q] + lane));
                        p.store_base[q][mine[q] + lane] = f[oppq(q)];
                    }
                const uint32_t rest = (node & NODE_HAS_BC) ? (node & NODE_LINKS & ~wl) : 0u;  // inlet/outlet; static links keep their slot
                if (rest) {
                    const long long c = (long long)(((unsigned long long)chi << 32) | clo) + lane;  // Cartesian cell
                    T gl[Q], hv[Q];
#pragma unroll
                    for (int q = 0; q < Q; q++) gl[q] = f[q];
                    const uint32_t wm = boundary_node<T, COLL>(p, c, rest, MODE_AB, rho, ux, uy, uz, gl, gl, hv, p.pulse_scale);
#pragma unroll
                    for (int q = 1; q < Q; q++)
                        if (wm & (1u << q)) {
                            LBM_CHK(p, p.store_base[q] + (mine[q] + lane));
                            p.store_base[q][mine[q] + lane] = hv[q];
                        }
                }
            }
        }
        r0 = n0, r1 = n1;
    }
    if (RESID) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) velsum += __shfl_xor_sync(0xffffffffu, velsum, o);
        if (lane == 0 && velsum != 0.0) atomicAdd(p.resid, velsum);
    }
}

}  // namespace lbm
