// Internal declarations shared by the translation units of liblbm_b200.so.
// Not installed; the public surface is include/lbm_b200.h.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/lbm_b200.h"

namespace lbm {

// node word ("link mask") of the fused kernels
//   bit 0        : node is NOT a fluid node (skip)
//   bit q (1..18): the source x - c_q of direction q is not a fluid node, so the
//                  pulled value is one this node pushed itself last step
constexpr int Q = 19;  // D3Q19
constexpr uint32_t NODE_SKIP = 1u;
constexpr uint32_t NODE_LINKS = 0x7FFFEu;
//   bit 31       : every non-fluid source of this node is a wall (label 1): all its
//                  links are plain half-way bounce-back, handled inline
constexpr uint32_t NODE_WALLS_ONLY = 0x80000000u;
//   bit 30       : at least one link of this node comes from an inlet/outlet/lid node and lies in
//                  that boundary's direction set, i.e. needs the non-equilibrium extrapolation.
//                  Without it every non-wall link is "static" (its slot is never rewritten).
constexpr uint32_t NODE_HAS_BC = 0x40000000u;
// second word per node ("wall mask"): bit q set <=> the source of direction q is a wall.  Only
// read for nodes that have links and are not walls-only (curved walls: -1 outer neighbours).

// per 32-cell segment summary (one warp of the dense kernels)
enum : uint8_t { SEG_BULK = 0, SEG_MIXED = 1, SEG_EMPTY = 2 };

struct BcEntry {
    int kind, naxis, nsign, vaxis, source, pulsatile;
    double value, init_value;
};

// Geometry of a box of cells stored [z][y][x] with padded x pitch.
struct Box {
    int nx, ny, nz;   // GLOBAL dims (reference NX,NY,NZ)
    int px;           // x pitch in cells (multiple of 32)
    int z0, z1;       // global z range [z0,z1) held by this array
    long long plane;  // px*ny
    __host__ __device__ long long cells() const { return plane * (long long)(z1 - z0); }
};

struct GeoRules {
    int case_rule;
    int n_open;
    lbm_opening_rule open[LBM_MAX_OPENINGS];
    unsigned mark_sources;  // bit L set: label L is a marking source
};

// everything the fused step kernels need, passed by value as a __grid_constant__
template <typename T>
struct StepParams {
    const T *src;
    T *dst;
    long long qstride;  // elements between consecutive populations
    const uint32_t *node;
    const uint32_t *wall;  // wall mask per cell (dense) / per compact id (sparse)
    const uint8_t *seg;
    const int8_t *label8;
    T *rho, *ux, *uy, *uz;  // dense moments (written when MOMENTS)
    double *resid;          // [1] accumulator of sum |u| (written when RESID)
    Box box;                // state box
    long long c_begin, c_end;  // cell range processed by this launch
    int fluid_label;
    T tau, inv_tau, om1;  // om1 = 1 - 1/tau
    T pulse_scale;
    BcEntry bc[LBM_MAX_BC];
    const T *plane_in, *plane_out;  // nx * nz(global) each
    int parity;                     // AA: 0 even (local) step, 1 odd (shifted) step
    int speculative;                // issue the population loads before the segment class is known
    // fused halo exchange: when this launch covers a face plane, fluid threads also store their
    // upward (c_z=+1) / downward (c_z=-1) populations into the neighbour slab's halo plane
    T *peer_up, *peer_dn;           // neighbour's destination buffer (peer / same-device memory) or null
    long long peer_up_qs, peer_dn_qs;   // its q stride
    long long peer_up_c0, peer_dn_c0;   // offset of its halo plane (cells, or compact ids for sparse)
    long long peer_up_own, peer_dn_own; // offset of its outermost owned plane (AA odd step pushes there)
    long long face_c0;              // offset of this launch's plane (cell of c_begin / first compact id)
    // Mailboxes (dense in-place storage across processes): the 5 populations that cross a face live in a small
    // separate allocation per side instead of in the halo / face planes of the population buffer, so that a
    // neighbour maps ~80 MB instead of the whole buffer (cudaIpcOpenMemHandle costs ~50-65 ms per GB).
    //   part A [5][mail_ms]: slot opp(q) of the HALO-plane cells  (written by the neighbour's even step and by this
    //                        slab's boundary links there, read by this slab's odd step)
    //   part B [5][mail_ms]: slot q of this slab's outermost OWNED plane  (written by the neighbour's odd step and by
    //                        this slab's boundary links, read by this slab's even step)
    // for the 5 directions q that enter through that face; element G + (in-plane cell index).
    T *mail[2];                     // this slab's own mailboxes (low / high side) when the launch covers that face, else null
    long long mail_ms, mail_G;
    int peer_mail;                  // peer_up / peer_dn point at the neighbour's mailbox (part A on even, part B on odd steps)
    int pdl;                        // in-place storages: launch with programmatic stream serialization (step_launch.cuh)
    // per-direction base pointers of the dense kernels, so that an access is base[q] + c (one 64-bit
    // add) instead of five integer instructions: pull_base[q][c] is the population direction q pulls
    // for cell c, store_base[q][c] the slot its post-collision value goes to (storage mode folded in)
    const T *pull_base[Q];
    T *store_base[Q];
    T *slot_base[Q];                // slot_base[q][c]: where cell c leaves the boundary value of its link q
    int case_rule;                  // lbm_case_rule
    T u_init;                       // lbm_case_desc.u_max
    // self-checking build (-DLBM_SELFCHECK, tools/selfcheck.py; compute-sanitizer is not available on the GPU
    // pool): every population access of the step kernels is checked against the handle's buffers, and a
    // shadow word per element records which thread touched it in this launch
    const T *chk_lo[2], *chk_hi[2];     // the population buffers [lo, hi)
    unsigned long long *chk_shadow[2];  // (launch id << 32) | (thread + 1) per buffer element
    unsigned long long *chk_count;      // [0] accesses outside the buffers, [1] elements touched by two threads in one launch
    unsigned int chk_launch;
    // collision operator (lbm_collision) and, for TRT, its odd-part rate omega- and 1 - omega- (lattice.cuh
    // collide_trt); the even-part rate is inv_tau.  Appended last so that no member above moves.
    int collision;
    T om_m, om1_m;
    // SparseParams embeds this struct: its later members move by what was appended here.  A multiple of 16 bytes
    // keeps their 16-byte alignment, which decides how the kernels merge parameter loads (LDCU.128).
    int align16[sizeof(T) == 4 ? 2 : 4];
};

// Precomputed inlet / outlet links of the in-place sparse storage: per node with NODE_HAS_BC a header
// (mask of the links that take the non-equilibrium extrapolation) followed by one entry per set bit, in
// direction order.  The step kernel then needs no label look-ups, coordinates or profile evaluation.
template <typename T>
struct BcLink {
    uint32_t meta;  // header: link mask.  entry: bits 0-1 lbm_bc_kind, bits 2-3 c_q[vel_axis] + 1, bit 4 pulsatile
    uint32_t pad;
    T ubc;          // prescribed speed at the source node (before the pulsatile scale)
};

template <typename T>
struct InitParams {
    T *fa, *fb;  // both buffers (fb == fa for in-place storage)
    int aa;      // in-place storage: slot (q,c) holds the PRE-STREAMED population feq_q(cell c - c_q)
    long long qstride;
    const int32_t *label;  // state box labels (int32)
    T *rho, *ux, *uy, *uz;
    Box box;
    int case_rule;
    T u_max;
    BcEntry bc[LBM_MAX_BC];
    const T *plane_in, *plane_out;
    int fluid_label;
};

// ---- launchers implemented in the .cu files ----
// geometry (lbm_geo.cu)
cudaError_t launch_make_flag_pos(uint8_t *flag, Box ext, cudaStream_t s);
cudaError_t launch_labels(const uint8_t *flag, int32_t *label, Box ext, GeoRules r, cudaStream_t s);
cudaError_t launch_mark(int32_t *label, Box ext, GeoRules r, cudaStream_t s);
// exclusive scan of (label != 0) over `cells` cells; index = running count + base, or -1
// plane_first_dev (optional, [cells/plane]): compact id each z-plane starts at
cudaError_t launch_compact(const int32_t *label, int32_t *index, long long cells, int px, int nx, int all,
                           long long base, int32_t *scratch, size_t scratch_ints, long long *total_out_dev,
                           long long plane, long long *plane_first_dev, cudaStream_t s);
size_t compact_scratch_ints(long long cells);
// order-independent 64-bit hash of a label field (checkpoint header)
cudaError_t launch_label_hash(const int32_t *label, long long cells, unsigned long long *out_dev, cudaStream_t s);
cudaError_t launch_count_stored(const int32_t *label, long long cells, int px, int nx, int all, long long *out_dev,
                                cudaStream_t s);
cudaError_t launch_node_words(const int32_t *label, uint32_t *node, uint32_t *wall, uint8_t *seg, int8_t *label8, Box box,
                              int own_z0, int own_z1, int fluid_label, const BcEntry *bc, long long *nfluid_dev,
                              cudaStream_t s);
template <typename T>
cudaError_t launch_init(const InitParams<T> &p, cudaStream_t s);
template <typename T>
cudaError_t launch_gather_fields(const T *rho, const T *ux, const T *uy, const T *uz, const int32_t *label,
                                 const int32_t *index, const int32_t *sid, Box box, int own_z0, int own_z1, int fluid_label,
                                 long long first, T *orho, T *oux, T *ouy, T *ouz, cudaStream_t s);
// layout: 0 two-buffer (slot q of cell y), 1 AA before an even step (a[q][y+c_q]), 2 AA before an odd step (a[opp q][y])
template <typename T>
cudaError_t launch_gather_pops(const T *f, long long qstride, const int32_t *index, Box box, int own_z0, int own_z1,
                               long long first, long long count, int layout, T *out, cudaStream_t s);
template <typename T>
cudaError_t launch_reduce_fields(const T *ux, const T *uy, const T *uz, const int32_t *label, Box box, int own_z0,
                                 int own_z1, int kind, int fluid_label, int case_rule, double *out_dev, cudaStream_t s);
template <typename T>
cudaError_t launch_halo_pack(const T *f, long long qstride, Box box, int zl, int side, T *buf, cudaStream_t s);
template <typename T>
cudaError_t launch_halo_unpack(T *f, long long qstride, const int8_t *label8, int fluid_label, Box box, int zl, int side,
                               const T *buf, cudaStream_t s);

// mailbox <-> population buffer (dir 0: fill the mailbox from the buffer, 1: drain it back); see StepParams::mail
template <typename T>
cudaError_t launch_mail_merge(T *mail, const T *in, long long n, cudaStream_t s);
template <typename T>
cudaError_t launch_mail_copy(T *a, long long qstride, T *mail, long long ms, long long G, long long face_c0, long long halo_c0,
                             long long plane, int side, int dir, cudaStream_t s);
// neighbour handshake of z-slabs in different processes (flags in peer memory), lbm_geo.cu
cudaError_t launch_slab_wait(unsigned long long *sync, unsigned long long need_lo, unsigned long long need_hi,
                             unsigned long long timeout_ns, cudaStream_t s);
cudaError_t launch_slab_signal(unsigned long long *peer_lo, unsigned long long *peer_hi, unsigned long long value,
                               cudaStream_t s);

// ---- sparse storage (reference compact order + run segments), lbm_geo.cu
constexpr int SEG_REC = 48;   // int32 per segment record: two pieces of 24, see k_seg_build
constexpr int SEG_HALF = 24;
// Segments over the compact ids [id0, id1) of the owned planes.  pass 1 (rec == nullptr): records per
// aligned 32-id chunk + scan (total to *nseg_dev); pass 2: fill the records and, per owned plane, the
// index of its first record (plane_seg[z], atomicMin; preset to a large value by the caller).
cudaError_t launch_build_segments(const uint32_t *nodec, const long long *cart, const int32_t *index, Box box,
                                  int own_zl0, long long id0, long long id1, long long id_first, int32_t *counts,
                                  long long *offsets, long long *nseg_dev, int32_t *rec, long long *plane_seg,
                                  cudaStream_t s);
cudaError_t launch_compact_maps(const int32_t *index, const uint32_t *node, const uint32_t *wall, const int32_t *label,
                                long long cells, long long id_first, long long *cart, uint32_t *nodec, uint32_t *wallc,
                                int8_t *labelc, cudaStream_t s);
template <typename T>
cudaError_t launch_init_sparse(const InitParams<T> &p, const long long *cart, long long nstored, cudaStream_t s);
// debug view of the in-place sparse storage as the reference's d_scr: out[q][s] = the population the fluid
// node s + c_q pulls next (0 when that node is not fluid)
template <typename T>
cudaError_t launch_gather_pops_sparse_aa(const T *a, long long qstride, const int32_t *label, const int32_t *index,
                                         const int32_t *sid, Box box, int own_z0, int own_z1, int fluid_label, long long first,
                                         long long n, int odd, T *out, cudaStream_t s);
// the in-place sparse storage's own numbering (fluid nodes + single-cell x gaps), its records and chunk masks
cudaError_t launch_span_flags(const int32_t *label, Box box, int fluid_label, int32_t *keep, cudaStream_t s);
cudaError_t launch_chunk_meta(const uint32_t *nodec, long long ns, uint2 *meta, cudaStream_t s);
// pass 1 (links == nullptr): *total_dev += entries needed; pass 2: lists filled, slots handed out by atomics
template <typename T>
cudaError_t launch_bc_links(const uint32_t *nodec, const uint32_t *wallc, const long long *cart, const int8_t *label8, Box box,
                            const BcEntry *bc, const T *plane_in, const T *plane_out, long long i0, long long i1,
                            int *total_dev, int32_t *bcslot, BcLink<T> *links, cudaStream_t s);
cudaError_t launch_rec_links(const int32_t *rec, const uint32_t *nodec, long long nseg, uint32_t *links, cudaStream_t s);
cudaError_t launch_build_segments_rows(const uint32_t *nodec, const long long *cart, const int32_t *sid, const int32_t *label,
                                       int fluid_label, Box box, int own_zl0, long long id0, long long id1, int32_t *counts,
                                       long long *offsets, long long *nseg_dev, int32_t *rec, long long *plane_seg,
                                       cudaStream_t s);
template <typename T>
cudaError_t launch_reduce_fields_sparse(const T *ux, const T *uy, const T *uz, const int8_t *labelc, const long long *cart,
                                        Box box, long long i0, long long i1, int kind, int fluid_label, int case_rule,
                                        double *out_dev, cudaStream_t s);
template <typename T>
cudaError_t launch_halo_pack_sparse(const T *f, long long qstride, long long i0, long long n, int side, T *buf,
                                    long long bufstride, cudaStream_t s);
template <typename T>
cudaError_t launch_halo_unpack_sparse(T *f, long long qstride, const int8_t *labelc, int fluid_label, long long i0,
                                      long long n, int side, const T *buf, long long bufstride, cudaStream_t s);

// everything the sparse step needs
template <typename T>
struct SparseParams {
    StepParams<T> base;      // src/dst (compact), qstride = stored nodes of the state box, box, bc, ...
    const int32_t *rec;      // [nseg][SEG_REC]
    const uint32_t *nodec;   // node words by compact id
    const uint32_t *wallc;   // wall masks by compact id
    long long seg_begin, seg_end;
    int spw;                 // consecutive records per warp
    // in-place sparse storage (step_sparse_aa.cuh)
    const long long *cartc;  // Cartesian cell of a compact id (boundary slow path)
    const uint2 *cmeta;      // per aligned chunk of 32 ids: fluid-lane mask, "some lane has a non-wall link"
    const uint32_t *rec_links;  // [nseg][32] node word of every lane of a record (NODE_SKIP outside its pieces)
    const int32_t *bcslot;      // per id: first BcLink of the node's list (nodes with NODE_HAS_BC only)
    const BcLink<T> *bclinks;
    long long id_begin, id_end;  // compact ids of the even (local) step's launch
    int halo_lo_n, halo_hi0;     // local ids < halo_lo_n lie in the low halo plane, ids >= halo_hi0 in the high one
    int dk[Q];                   // (k - opp k) * qstride: from the array of opp(k) to the same node's slot in the array of k
};

// fused step (step_launch.cuh), instantiated for STRICT = false in lbm_step_fast.cu and true in lbm_step_strict.cu
// one step over the range of sp, which the caller checked is not empty; the dense storages read sp.base only
template <typename T, bool STRICT>
cudaError_t launch_step(const SparseParams<T> &sp, int storage, bool moments, bool resid, cudaStream_t s);
// nsteps steps of a single-domain in-place sparse handle in ONE cooperative launch (grids that live in L2)
template <typename T, bool STRICT>
cudaError_t launch_persist(const SparseParams<T> &sp, int nsteps, int parity0, int moments_last, double *S, const T *pulse,
                           unsigned *barrier, int sm_count, cudaStream_t s);
// loads the step kernels a run loop is about to launch
template <typename T, bool STRICT>
cudaError_t preload_step_kernels(int storage, int collision, bool speculative, bool resid, bool persist);

}  // namespace lbm
