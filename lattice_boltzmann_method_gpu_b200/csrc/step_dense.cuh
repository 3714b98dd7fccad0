// Fused pull-stream + collide (BGK or TRT, lattice.cuh) + moment kernel on the box-dense SoA layout,
// with link-wise boundaries evaluated by the FLUID node ("fluid-side push").
//
// Replaces the reference's `update` + `boundary_stream` pair
// (ldc.cu:57-458, Poiseulle.cu:384-893, bifurcation.cu:429-1023,
// coronary.cu:352-944) with one launch per time step.
//
// Layout: f[q][z][y][x], x fastest, x pitch a multiple of 32 cells, one 1-D
// cell id c = x + px*(y + ny*zl).  The pull of direction q reads
// f[q][c - off_q], off_q = cx + px*cy + plane*cz: a constant shift, so a warp
// reads 32 consecutive reals per population (coalesced; the x-shifted ones
// straddle one extra sector).  No thread ever needs its coordinates on the
// bulk path.
//
// Boundaries (SURVEY A.5, proven equivalent to the reference's stored-node
// scheme at every fluid node): only fluid nodes compute.  For a direction q
// whose source s = x - c_q is not fluid, the value the reference's wall / inlet /
// outlet node s would hold in slot (q,s) after `boundary_stream` depends only on
// x's own post-collision state and moments:
//     wall             : g_opp(q)(x)                               (bif:655-798)
//     inlet/outlet, q in its set:
//         feq_q(rho_bc,u_bc(s)) + (g_q(x) - feq_q(rho_x,u_x))(1-1/tau)   (bif:877-1021)
//     otherwise ("static"): the initial equilibrium of s, never rewritten
// so x itself writes it into slot (q,s) of the destination buffer at the end of
// its own update ("push into the solid node's slot").  The next step's pull is
// then uniform for every node: f_q(x) = src[q][x - c_q].
//
// One warp = one 32-cell segment.  seg[] classifies segments: BULK (all 32 are
// fluid with fluid sources only -> no node-word load, no divergence), MIXED, or
// EMPTY (nothing to do).
#pragma once
#include <cstdlib>
#include "lattice.cuh"
#include "lbm_internal.h"
#include "init_rule.cuh"

namespace lbm {

template <typename T>
__device__ __forceinline__ T ld_stream(const T *p) {
    return __ldg(p);
}

// Self-checking build: LBM_CHK(p, address) in front of every population access of the step kernels.
//  - the address must lie inside one of the handle's population buffers (guards included);
//  - within one launch an element may be touched by ONE thread only -- the property that makes the
//    in-place (AA) step race-free and lets the two-buffer step write boundary slots without atomics.
// A normal build compiles the macro away.
#ifdef LBM_SELFCHECK
template <typename T>
__device__ __noinline__ void chk_touch(const StepParams<T> &p, const T *a, bool track = true) {
    if (!p.chk_count) return;
    for (int b = 0; b < 2; b++)
        if (a >= p.chk_lo[b] && a < p.chk_hi[b]) {
            if (!track) return;  // a speculative read whose value is dropped: only its address matters
            const unsigned long long tag = ((unsigned long long)p.chk_launch << 32) |
                                           (unsigned long long)((unsigned)blockIdx.x * blockDim.x + threadIdx.x + 1u);
            const unsigned long long old = atomicExch(p.chk_shadow[b] + (a - p.chk_lo[b]), tag);
            if ((old >> 32) == p.chk_launch && old != tag) atomicAdd(p.chk_count + 1, 1ull);
            return;
        }
    atomicAdd(p.chk_count, 1ull);
}
#define LBM_CHK(p_, a_) chk_touch(p_, a_)
#define LBM_CHK_BOUNDS(p_, a_) chk_touch(p_, a_, false)
#else
#define LBM_CHK(p_, a_) ((void)0)
#define LBM_CHK_BOUNDS(p_, a_) ((void)0)
#endif

// prescribed boundary speed of BC entry `e` at boundary node (gx, gy, gz) (global coords)
template <typename T>
__device__ __forceinline__ T bc_speed(const StepParams<T> &p, const BcEntry &e, int gx, int gz, T pulse) {
    T u = bc_speed_unscaled<T>(e, p.box, p.plane_in, p.plane_out, gx, gz);
    if (e.pulsatile) u = u * pulse;
    return u;
}

// equilibrium of a prescribed axis-aligned velocity, the reference's literal
// polynomials (pos.cu:766, ldc.cu:402,441,454)
template <typename T>
__device__ __forceinline__ T feq_bc_axis(T rw, int cs, T u) {
    if (cs > 0) return rw * (T(1.0) + T(3.0) * u + T(3.0) * u * u);
    if (cs < 0) return rw * (T(1.0) - T(3.0) * u + T(3.0) * u * u);
    return rw * (T(1.0) - T(1.5) * u * u);
}

// Storage modes of the populations
//   MODE_AB      two buffers.  pull  src[q][c - off_q]         store dst[q][c]
//                              boundary slot of link q:        dst[q][c - off_q]
//   MODE_AA_EVEN one buffer, even step (purely local).
//                              pull  a[q][c]                   store a[opp q][c]
//                              boundary slot of link q:        a[opp q][c - off_q]   (read by the odd step)
//   MODE_AA_ODD  one buffer, odd step.
//                              pull  a[opp q][c - off_q]       store a[q][c + off_q] (only into fluid targets)
//                              boundary slot of link q:        a[q][c]               (read by the even step)
// AA-pattern streaming (Bailey et al. 2009) with the fluid-side boundaries of this file: every slot
// a thread touches in a launch is touched by that thread only, so the update is in place.
// The even step overwrites slot (q,c) of a link whose source is not fluid, so in the two in-place
// modes a static link CARRIES its constant along: the value pulled for it (the initial equilibrium of
// its source, whatever that was) is written back, before the collision, into the slot the following
// step pulls from.  Two-buffer storage never writes static slots.
enum { MODE_AB = 0, MODE_AA_EVEN = 1, MODE_AA_ODD = 2 };

// Slow path of a node next to an inlet / outlet / lid: the values this fluid node (cell c, moments
// rho/u, post-collision populations g, pulled populations fpre) must leave in the slots of its links
// `rest`; returns the mask of links to write (a static link of the two-buffer storage keeps its slot).  Out of line, so the bulk path stays small, and one call
// per NODE in three phases -- all source labels, then all prescribed speeds, then the arithmetic --
// so that the dependent loads of the links overlap instead of queueing up link after link: these
// few nodes set the lifetime of their CTA, which is what a small grid's step time consists of.
template <typename T, int COLL>
__device__ __noinline__ uint32_t boundary_node(const StepParams<T> &p, long long c, uint32_t rest, int mode, T rho, T ux,
                                               T uy, T uz, const T *g, const T *fpre, T *out, T pulse) {
    const Box &b = p.box;
    int x, y, zl;  // coordinates of the node, once (32-bit arithmetic when the cell id allows it)
    if (c < 0x7fffffffLL) {
        const unsigned cu = (unsigned)c, px = (unsigned)b.px, ny = (unsigned)b.ny, t = cu / px;
        x = (int)(cu - t * px), zl = (int)(t / ny), y = (int)(t - (unsigned)zl * ny);
    } else {
        const long long t = c / b.px;
        x = (int)(c - t * b.px), zl = (int)(t / b.ny), y = (int)(t - (long long)zl * b.ny);
    }
    int lab[Q];
#pragma unroll
    for (int q = 1; q < Q; q++) {
        lab[q] = 0;
        if (rest & (1u << q)) lab[q] = p.label8[c - ((long long)cxq(q) + (long long)b.px * cyq(q) + b.plane * czq(q))];
    }
    uint32_t bcm = 0;  // links whose source is an inlet/outlet node prescribing this direction
    T ubc[Q];
#pragma unroll
    for (int q = 1; q < Q; q++) {
        ubc[q] = T(0.0);
        const int l = lab[q];
        if ((rest & (1u << q)) && l >= 2 && l < LBM_MAX_BC && p.bc[l].kind != LBM_BC_NONE &&
            caxis(q, p.bc[l].naxis) == p.bc[l].nsign) {
            bcm |= 1u << q;
            // the speed is sampled at the boundary node s = x - c_q itself (pos.cu:597)
            if (p.bc[l].kind != LBM_BC_P) ubc[q] = bc_speed<T>(p, p.bc[l], x - cxq(q), zl - czq(q) + b.z0, pulse);
        }
    }
    const T r3 = rho / T(3.0), r18 = rho / T(18.0), r36 = rho / T(36.0);
    const T one = T(1.0);
    uint32_t wm = 0;
#pragma unroll
    for (int q = 1; q < Q; q++) {
        if (!(rest & (1u << q))) continue;
        const int l = lab[q];
        if (l == 1) {  // half-way bounce-back
            out[q] = g[oppq(q)];
            wm |= 1u << q;
        } else if (bcm & (1u << q)) {
            // feq_q(rho_bc, u_bc(s)) + (g_q(x) - feq_q(rho_x, u_x)) (1 - 1/tau)      (bif:877-1021)
            // TRT: the extrapolated non-equilibrium n_q = g_q(x) - feq_q(rho_x, u_x) relaxes like the collision,
            //      feq_q(rho_bc, u_bc(s)) + (1 - om+) (n_q + n_opp(q))/2 + (1 - om-) (n_q - n_opp(q))/2
            const BcEntry &e = p.bc[l];
            const T feq = feq_lit<T>(q, r3, r18, r36, ux, uy, uz);
            T tmp;
            if (e.kind == LBM_BC_P) {
                tmp = feq_lit<T>(q, one / T(3.0), one / T(18.0), one / T(36.0), ux, uy, uz);
            } else {
                const T rw = e.kind == LBM_BC_V ? (q < 7 ? r18 : r36) : (q < 7 ? one / T(18.0) : one / T(36.0));
                tmp = feq_bc_axis<T>(rw, caxis(q, e.vaxis), ubc[q]);
            }
            if constexpr (COLL == LBM_COLL_TRT) {
                const T nq = g[q] - feq, nb = g[oppq(q)] - feq_lit<T>(oppq(q), r3, r18, r36, ux, uy, uz);
                out[q] = tmp + (p.om1 * (T(0.5) * (nq + nb)) + p.om1_m * (T(0.5) * (nq - nb)));
            } else {
                out[q] = tmp + (g[q] - feq) * p.om1;
            }
            wm |= 1u << q;
        } else if (mode != MODE_AB) {
            out[q] = fpre[q];  // static link, in-place storage: the constant travels with the link
            wm |= 1u << q;
        }
    }
    return wm;
}

// ---------------------------------------------------------------------------
// fused step
// ---------------------------------------------------------------------------
// One warp per 32-cell segment, one CTA per B consecutive cells.  Two forms:
//   SPEC = false : class byte -> (node word) -> 19 population loads.  Nothing is
//                  read for EMPTY segments or non-fluid cells; the class byte
//                  (L2-resident) sits on the critical path.
//   SPEC = true  : the 19 population loads, the class byte and the node word are
//                  all issued up front, for every thread; non-fluid threads drop
//                  the values.  No dependent load precedes the DRAM reads.  Chosen
//                  by the host when >= 90 % of the launched cells are fluid (dense
//                  cavities), where the wasted reads are a few percent.
// The kernel is latency-bound per warp, so resident warps matter more than
// anything else: CTA shape and register cap are picked per precision
// (fp64: 128 threads x 6 CTAs/SM, 80 registers; fp32: 128 x 10, 48 registers; no spills).
// Measurements behind every choice here: profiles/r01_notes.md.
constexpr int DENSE_BLOCK = 128;
#ifndef LBM_F32_MINB
#define LBM_F32_MINB 10
#endif
#ifndef LBM_F64_MINB
#define LBM_F64_MINB 6
#endif

// Loads of the speculative pull.  They have to be ISSUED before the thread knows whether it needs them, and
// ptxas sinks an ordinary ld.global (also .nc, also from `asm volatile`) below the early exit that depends on
// the segment byte -- which puts a dependent L2 round trip in front of every population load (SASS of round 1
// and 2: `LDG.U8 kind ... @!P0 EXIT ; LDG ...`).  A relaxed gpu-scope load must be performed where it
// stands; it is served by L2 like every streaming load of this kernel (in-place storage: 0.975 -> 0.983 fp64).
#ifndef LBM_SPEC_LD
#define LBM_SPEC_LD 1
#endif
// two-buffer storage: the read-only path, sunk or not, measured better than the relaxed load (0.954 / 0.890
// against 0.948 / 0.885 of peak, fp64 / fp32)
__device__ __forceinline__ double ld_spec(const double *p) {
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_spec(const float *p) {
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
// in-place modes read and write the same array in one launch: no read-only (.nc) path there
__device__ __forceinline__ double ld_spec_rw(const double *p) {
    double v;
#if LBM_SPEC_LD == 1
    asm volatile("ld.relaxed.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(p));
#else
    asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(p));
#endif
    return v;
}
__device__ __forceinline__ float ld_spec_rw(const float *p) {
    float v;
#if LBM_SPEC_LD == 1
    asm volatile("ld.relaxed.gpu.global.f32 %0, [%1];" : "=f"(v) : "l"(p));
#else
    asm volatile("ld.global.f32 %0, [%1];" : "=f"(v) : "l"(p));
#endif
    return v;
}

template <int MODE>
__host__ __device__ __forceinline__ long long pull_index(int q, long long c, long long qs, long long off) {
    if (MODE == MODE_AB) return (long long)q * qs + c - off;
    if (MODE == MODE_AA_EVEN) return (long long)q * qs + c;
    return (long long)oppq(q) * qs + c - off;
}
template <int MODE>
__host__ __device__ __forceinline__ long long store_index(int q, long long c, long long qs, long long off) {
    if (MODE == MODE_AB) return (long long)q * qs + c;
    if (MODE == MODE_AA_EVEN) return (long long)oppq(q) * qs + c;
    return (long long)q * qs + c + off;
}
template <int MODE>
__host__ __device__ __forceinline__ long long slot_index(int q, long long c, long long qs, long long off) {
    if (MODE == MODE_AB) return (long long)q * qs + c - off;
    if (MODE == MODE_AA_EVEN) return (long long)oppq(q) * qs + c - off;
    return (long long)q * qs + c;
}

// collide, store, moments, boundary links of one fluid cell whose post-streaming
// populations are already in f[]
// Fused halo exchange: the populations that leave through a z face go straight into the neighbour
// slab's halo plane (same x,y; `i` = offset inside the plane).  c_z=+1: q in {5,11,13,15,16}.
// In-place storage: the even step leaves g_q(x) in slot opp(q) of x, which the neighbour's odd step
// pulls -> the copy goes into slot opp(q) of the neighbour's halo plane; the odd step pushes g_q(x)
// into slot q of the TARGET cell x + c_q, which for a face plane is a cell of the neighbour's
// outermost owned plane (shifted by the in-plane part of c_q), fluid targets only.
template <typename T, int MODE>
__device__ __forceinline__ void push_to_peers(const StepParams<T> &p, long long i, uint32_t node, const T (&f)[Q]) {
#pragma unroll
    for (int q = 1; q < Q; q++) {
        if (czq(q) == 0) continue;
        T *peer = czq(q) > 0 ? p.peer_up : p.peer_dn;
        if (!peer) continue;
        const long long qs = czq(q) > 0 ? p.peer_up_qs : p.peer_dn_qs;
        if (p.peer_mail) {  // the neighbour's mailbox: part A on even steps, part B (shifted in-plane target) on odd ones
            if (MODE == MODE_AA_EVEN) {
                peer[(long long)kslot(q) * qs + (czq(q) > 0 ? p.peer_up_c0 : p.peer_dn_c0) + i] = f[q];
            } else if (MODE == MODE_AA_ODD && !(node & (1u << oppq(q)))) {
                peer[(long long)kslot(q) * qs + (czq(q) > 0 ? p.peer_up_own : p.peer_dn_own) + i + cxq(q) + (long long)p.box.px * cyq(q)] = f[q];
            }
            continue;
        }
        if (MODE == MODE_AB) {
            peer[(long long)q * qs + (czq(q) > 0 ? p.peer_up_c0 : p.peer_dn_c0) + i] = f[q];
        } else if (MODE == MODE_AA_EVEN) {
            peer[(long long)oppq(q) * qs + (czq(q) > 0 ? p.peer_up_c0 : p.peer_dn_c0) + i] = f[q];
        } else if (!(node & (1u << oppq(q)))) {
            peer[(long long)q * qs + (czq(q) > 0 ? p.peer_up_own : p.peer_dn_own) + i + cxq(q) + (long long)p.box.px * cyq(q)] = f[q];
        }
    }
}

// WALL_READY: the caller already holds the node's wall mask in `wallw`; otherwise it is fetched here,
// lazily, by the few nodes that need it
template <typename T, bool STRICT, int COLL, bool MOMENTS, bool RESID, int MODE, bool WALL_READY>
__device__ __forceinline__ void finish_cell(const StepParams<T> &p, long long c, uint32_t node, uint32_t wallw, T (&f)[Q],
                                            double &velsum) {
    T rho, ux, uy, uz;
    // in-place storage: links that are neither walls nor (for nodes without NODE_HAS_BC) boundary links
    // are static -- put the pulled constant back where the next step pulls it, before it is collided
    T fpre[Q];
    bool keep_pre = false;
    if (MODE != MODE_AB && (node & NODE_LINKS) && !(node & NODE_WALLS_ONLY)) {
        if (!WALL_READY) wallw = p.wall[c];
        const uint32_t rest = node & NODE_LINKS & ~wallw;
        if (rest && !(node & NODE_HAS_BC)) {
#pragma unroll
            for (int q = 1; q < Q; q++)
                if (rest & (1u << q)) {
                    LBM_CHK(p, p.slot_base[q] + c);
                    p.slot_base[q][c] = f[q];
                }
        } else if (rest) {
            keep_pre = true;
#pragma unroll
            for (int q = 0; q < Q; q++) fpre[q] = f[q];
        }
    }
    collide<T, STRICT, COLL>(f, p, rho, ux, uy, uz);
#pragma unroll
    for (int q = 0; q < Q; q++) {
        if (MODE == MODE_AA_ODD) {
            // push only into fluid targets: x + c_q is the source of link opp(q); a target beyond a
            // slab face lives in the neighbour's memory (push_to_peers)
            const bool remote = (czq(q) > 0 && p.peer_up) || (czq(q) < 0 && p.peer_dn);
            if (q == 0 || (!(node & (1u << oppq(q))) && !remote)) {
                LBM_CHK(p, p.store_base[q] + c);
                p.store_base[q][c] = f[q];
            }
        } else {
            LBM_CHK(p, p.store_base[q] + c);
            p.store_base[q][c] = f[q];
        }
    }
    if (MOMENTS) {
        p.rho[c] = rho, p.ux[c] = ux, p.uy[c] = uy, p.uz[c] = uz;
    }
    if (RESID) velsum += (double)(T)sqrt((double)(ux * ux + uy * uy + uz * uz));  // |u| as ldc.cu:464 forms it
    if (p.peer_up || p.peer_dn) push_to_peers<T, MODE>(p, (long long)c - p.face_c0, node, f);
    if (node & NODE_LINKS) {
        // wall links: half-way bounce-back, inline: the link's slot <- g_opp(q)(x)   (bif:781-798)
        const uint32_t wl = (node & NODE_WALLS_ONLY) ? (node & NODE_LINKS)
                                                     : ((WALL_READY || MODE != MODE_AB) ? (wallw & node & NODE_LINKS) : p.wall[c]);
#pragma unroll
        for (int q = 1; q < Q; q++) {
            if (wl & (1u << q)) {
                LBM_CHK(p, p.slot_base[q] + c);
                p.slot_base[q][c] = f[oppq(q)];
            }
        }
        // what is left is an inlet/outlet/lid link (slow path) or a static link (handled above)
        const uint32_t rest = node & NODE_LINKS & ~wl;
        if (rest && (node & NODE_HAS_BC)) {
            T gl[Q], hv[Q];  // copies in local memory on this path only: f[] itself stays in registers
#pragma unroll
            for (int q = 0; q < Q; q++) gl[q] = f[q];
            if (!keep_pre) {  // two-buffer storage: never read
#pragma unroll
                for (int q = 0; q < Q; q++) fpre[q] = T(0.0);
            }
            const uint32_t wm = boundary_node<T, COLL>(p, (long long)c, rest, MODE, rho, ux, uy, uz, gl, fpre, hv, p.pulse_scale);
#pragma unroll
            for (int q = 1; q < Q; q++) {
                if (wm & (1u << q)) {
                    LBM_CHK(p, p.slot_base[q] + c);
                    p.slot_base[q][c] = hv[q];
                }
            }
        }
    }
}

// Programmatic dependent launch: a step kernel lets the next launch of the stream start as soon as all of its
// own CTAs are resident (grid_dep_launch, first instruction), and waits for the previous launch to be complete
// and visible only where it first touches populations (grid_dep_wait) -- geometry words, records and link
// lists are never written by a step, so their loads and the launch latency itself (2 - 3 us, a third of a
// 64^3 step) overlap the previous step's tail.  Both are no-ops when the launch does not carry the attribute.
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Used by the in-place storages only: the two-buffer kernels read through the non-coherent path (ld.global.nc),
// whose contract -- read-only for the lifetime of the kernel -- an early-started kernel would break.

template <typename T, bool STRICT, int COLL, bool MOMENTS, bool RESID, bool SPEC, int MODE>
__global__ void __launch_bounds__(DENSE_BLOCK, sizeof(T) == 8 ? LBM_F64_MINB : LBM_F32_MINB)
    k_step_dense(const __grid_constant__ StepParams<T> p) {
    const Box &b = p.box;
    // 64-bit cell ids on purpose: 32-bit ones turn every address into one IMAD.WIDE.U32 instead of an
    // IADD3 pair (-22 instructions per thread), which changes nothing in fp64 and costs 6 % in fp32,
    // where IMAD shares its pipe with the collision's FFMAs (profiles/r01_notes.md)
    if (MODE != MODE_AB) grid_dep_launch();
    const long long c = p.c_begin + (long long)blockIdx.x * DENSE_BLOCK + threadIdx.x;
    if (c >= p.c_end) return;  // ranges are whole planes (multiples of 32 cells): warp-uniform
    T f[Q];
    uint32_t node, wallw = 0u;
    const uint32_t kind = p.seg[c >> 5];
    if (SPEC) {
        // every thread pulls before it knows what its cell is; the buffers carry guards so all addresses are
        // mapped.  The node / wall words are fetched afterwards and for mixed segments only (in a box that is
        // mostly bulk they were 4 of the 156 bytes a fp32 cell moves), while the populations are in flight.
#ifdef LBM_SELFCHECK
        node = p.node[c];  // the checked build wants to know which reads are dropped
#endif
        if (MODE != MODE_AB) grid_dep_wait();
#pragma unroll
        for (int q = 0; q < Q; q++) {
            // every thread pulls, a non-fluid one drops what it read: bounds always, ownership only when used
#ifdef LBM_SELFCHECK
            if (node & NODE_SKIP) LBM_CHK_BOUNDS(p, p.pull_base[q] + c);
            else LBM_CHK(p, p.pull_base[q] + c);
#endif
            f[q] = MODE == MODE_AB ? ld_spec(p.pull_base[q] + c) : ld_spec_rw(p.pull_base[q] + c);
        }
        if (kind == SEG_EMPTY) return;
        node = kind == SEG_MIXED ? p.node[c] : 0u;
        wallw = kind == SEG_MIXED ? p.wall[c] : 0u;
    } else {
        if (kind == SEG_EMPTY) return;
        node = kind == SEG_MIXED ? p.node[c] : 0u;
        wallw = kind == SEG_MIXED ? p.wall[c] : 0u;
        if (MODE != MODE_AB) grid_dep_wait();
    }
    double velsum = 0.0;
    if (!(node & NODE_SKIP)) {
        if (!SPEC) {
#pragma unroll
            for (int q = 0; q < Q; q++) {
                LBM_CHK(p, p.pull_base[q] + c);
                f[q] = MODE == MODE_AB ? ld_stream(p.pull_base[q] + c) : p.pull_base[q][c];
            }
        }
        finish_cell<T, STRICT, COLL, MOMENTS, RESID, MODE, true>(p, c, node, wallw, f, velsum);
    }
    if (RESID) {
        // warp shuffle tree, then one atomic per warp
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) velsum += __shfl_xor_sync(0xffffffffu, velsum, o);
        if ((threadIdx.x & 31) == 0 && velsum != 0.0) atomicAdd(p.resid, velsum);
    }
}

// host: fold the storage mode into the per-direction base pointers
template <typename T, int MODE>
void set_bases(StepParams<T> &p) {
    for (int q = 0; q < Q; q++) {
        const long long off = (long long)cxq(q) + (long long)p.box.px * cyq(q) + p.box.plane * czq(q);
        p.pull_base[q] = p.src + pull_index<MODE>(q, 0, p.qstride, off);
        p.store_base[q] = p.dst + store_index<MODE>(q, 0, p.qstride, off);
        p.slot_base[q] = p.dst + slot_index<MODE>(q, 0, p.qstride, off);
    }
    // mailboxes of the faces this launch covers: the slots of the 5 entering directions live there
    for (int side = 0; side < 2; side++) {
        if (!p.mail[side] || MODE == MODE_AB) continue;
        for (int q = 1; q < Q; q++) {
            if (czq(q) != (side == 0 ? 1 : -1)) continue;  // enters through the low face with c_z = +1, through the high one with -1
            const long long inpl = (long long)cxq(q) + (long long)p.box.px * cyq(q);
            T *A = p.mail[side] + (long long)kslot(q) * p.mail_ms + p.mail_G - p.face_c0;
            T *B = p.mail[side] + (long long)(5 + kslot(q)) * p.mail_ms + p.mail_G - p.face_c0;
            if (MODE == MODE_AA_EVEN) {
                p.pull_base[q] = B;          // a[q][c]: pushed here by the neighbour's odd step / this node's boundary link
                p.slot_base[q] = A - inpl;   // a[opp q][c - off_q]: the halo cell's slot, read by the odd step
            } else {
                p.pull_base[q] = A - inpl;   // a[opp q][c - off_q]
                p.slot_base[q] = B;          // a[q][c]
            }
        }
    }
}

}  // namespace lbm
