/*
 * lbm_b200.h -- C ABI of liblbm_b200.so, a B200-native (sm_100a) D3Q19 BGK
 * Lattice-Boltzmann solver that is a drop-in for the *case interface* of
 * Xinhuan-Imperial/Lattice-Boltzmann-Method-GPU.
 *
 * The reference has no library / FFI surface: its "API" is the sequence of
 * file-scope functions each of its four programs calls from main()
 * (bifurcation.cu:1177-1326):
 *      geo_pre(); index_transform(); read_vel(); initialize();
 *      loop { update<<<>>>; boundary_stream<<<>>>; swap; } calc_res(); outputSave(t);
 * Every entry point below names the reference function it replaces
 * (file:line into /root/reference; ldc = Lid_driven_cavity/ldc.cu,
 * pos = Poiseulle_flow/Poiseulle.cu, bif = bifurcation/bifurcation.cu,
 * cor = coronary_cfd/coronary.cu).
 *
 * Conventions
 *  - plain C types only; every function returns 0 on success, a negative
 *    lbm_status otherwise; lbm_last_error(h) gives the message.  No exceptions
 *    cross the ABI.  One caller thread per handle; handles are independent.
 *  - "Cartesian" arrays are int32/real [nz][ny][nx], x fastest (the order of
 *    geo.txt, bif:50-61).  "Compact" arrays have NLATTICE entries in the
 *    reference's own numbering (running count over z,y,x of geo != 0,
 *    bif:241-252; for the LDC rule every node is stored, ldc:54).
 *  - real = float (LBM_F32, the reference's precision) or double (LBM_F64).
 *  - the library owns all device memory; the caller owns the host buffers it
 *    passes in.
 */
#ifndef LBM_B200_H
#define LBM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LBM_B200_ABI_VERSION 3

typedef struct lbm_solver_s *lbm_handle;

typedef enum {
    LBM_OK = 0,
    LBM_ERR_ARG = -1,     /* bad argument / descriptor */
    LBM_ERR_STATE = -2,   /* call out of order (e.g. step before initialize) */
    LBM_ERR_IO = -3,      /* file missing / short */
    LBM_ERR_CUDA = -4,    /* a CUDA call failed */
    LBM_ERR_NOMEM = -5,
    LBM_ERR_NO_DEVICE = -6 /* no CUDA device: there is deliberately no CPU fallback */
} lbm_status;

/* which reference program's geometry / initial-state / boundary rules apply */
typedef enum {
    LBM_CASE_LDC = 0,          /* ldc:468-580  lid-driven cavity, labels 0 ghost,1 wall,2 lid,3 fluid, dense */
    LBM_CASE_POISEUILLE = 1,   /* pos:52-382   circular pipe along y, analytic in/outlet velocity */
    LBM_CASE_GEO_Y_INOUT = 2,  /* bif:36-427   geo.txt voxels, inlet y=1 (bc.txt velocity), outlet y=NY-2 (pressure) */
    LBM_CASE_GEO_OPENINGS = 3  /* cor:31-350   geo.txt voxels, list of opening planes, constant BC speeds */
} lbm_case_rule;

typedef enum { LBM_F32 = 0, LBM_F64 = 1 } lbm_precision;

/* distribution storage */
typedef enum {
    LBM_STORE_DENSE_AB = 0,  /* box-dense SoA, two buffers, fused pull step            */
    LBM_STORE_DENSE_AA = 1,  /* box-dense SoA, ONE buffer, in-place AA-pattern streaming */
    LBM_STORE_SPARSE_AB = 2, /* reference compact order (NLATTICE entries), run-segment indirect addressing, two buffers */
    LBM_STORE_SPARSE_AA = 3  /* the same compact order, ONE buffer streamed in place; boundary links live in the fluid
                                node's own slot, so solid nodes are never touched by a step */
} lbm_storage;

/* arithmetic of the fused kernel */
typedef enum {
    LBM_MATH_FAST = 0,   /* FMA-contracted, reciprocal-multiply BGK (default, the measured path) */
    LBM_MATH_STRICT = 1  /* the reference's expression order, no contraction: bit-identical to the CPU oracle */
} lbm_math;

/* collision operator of the fused kernel (lbm_set_collision) */
typedef enum {
    LBM_COLL_BGK = 0, /* single relaxation time 1/tau (default, the reference's operator) */
    LBM_COLL_TRT = 1  /* two relaxation times: even part 1/tau, odd part set by the magic parameter; FAST only */
} lbm_collision;

/* boundary-condition kinds of the non-equilibrium extrapolation (SURVEY A.4) */
typedef enum {
    LBM_BC_NONE = 0,
    LBM_BC_V = 1,  /* rho from the fluid neighbour, prescribed u   (ldc:391-456, pos:748-891, bif:950-1021, cor:795-942) */
    LBM_BC_P = 2,  /* rho = 1, u from the fluid neighbour          (bif:877-948) */
    LBM_BC_VP = 3  /* rho = 1, prescribed u                        (cor:716-792) */
} lbm_bc_kind;

typedef enum {
    LBM_SRC_CONST = 0,        /* value                                        (ldc:378, cor:717) */
    LBM_SRC_PARABOLA = 1,     /* value*(1-((i-cx)^2+(k-cz)^2)/R^2), R=cx=(NX-1)/2, cz=(NZ-1)/2  (pos:597) */
    LBM_SRC_PLANE_INLET = 2,  /* inlet plane[i + k*NX] from bc.txt            (bif:650,951) */
    LBM_SRC_PLANE_OUTLET = 3  /* outlet plane[i + k*NX]                       (bif:296-325) */
} lbm_bc_source;

/* one boundary label.  Direction set = { q : c_q[normal_axis] == normal_sign }. */
typedef struct {
    int32_t label;       /* node label the entry applies to (1..7) */
    int32_t kind;        /* lbm_bc_kind */
    int32_t normal_axis; /* 0 x, 1 y, 2 z */
    int32_t normal_sign; /* +1 / -1: points from the boundary node into the fluid */
    int32_t vel_axis;    /* axis of the prescribed velocity */
    int32_t source;      /* lbm_bc_source */
    int32_t pulsatile;   /* != 0: multiply by 1 + pulse_amp*sin(2 pi t / pulse_period), t = step index.
                            No reference code exists for this (curved vessel/README.md:1): parity unpinned. */
    int32_t reserved;
    double value;        /* speed used by the boundary kernel, lattice units (pos:590, cor:717) */
    double init_value;   /* speed `initialize` gives nodes of this label (cor:302-306); the reference
                            computes the two with different float expressions, so both are carried */
} lbm_bc_desc;

/* one "opening plane" of the GEO_OPENINGS rule (cor:77-141): on plane
 * axis=coord, inside the inclusive window [lo_a,hi_a]x[lo_b,hi_b] of the two
 * in-plane axes (in x,y,z order), label += reps * min4(in-plane neighbours of flag) */
typedef struct {
    int32_t axis, coord, lo_a, hi_a, lo_b, hi_b, reps, reserved;
} lbm_opening_rule;

#define LBM_MAX_BC 8
#define LBM_MAX_OPENINGS 8

typedef struct {
    int32_t struct_size; /* sizeof(lbm_case_desc), checked */
    int32_t case_rule;   /* lbm_case_rule */
    int32_t nx, ny, nz;  /* GLOBAL box, the reference's NX,NY,NZ (bif:19) */
    int32_t precision;   /* lbm_precision */
    int32_t storage;     /* lbm_storage */
    int32_t math;        /* lbm_math */
    int32_t device;      /* CUDA device ordinal */
    int32_t geo_yfast;   /* geo.txt stored y-fastest (cor:45-56) instead of x-fastest (bif:50-61) */
    /* z-slab decomposition (new; the reference is single-GPU): this handle owns
     * global planes [z_begin, z_end); 0,nz for a single domain. */
    int32_t z_begin, z_end;
    int32_t n_bc, n_openings;
    double tau;          /* ldc:55, pos:39, bif:434 */
    double u_max;        /* LDC lid speed (ldc:52) / Poiseuille peak used by initialize (pos:44) */
    double C_U, C_rho, CH; /* unit converters used by the writers (bif:20) */
    double pulse_amp, pulse_period;
    lbm_bc_desc bc[LBM_MAX_BC];
    lbm_opening_rule openings[LBM_MAX_OPENINGS];
    char geo_path[256];  /* "./geo.txt" (bif:49) */
    char bc_path[256];   /* "./bc.txt"  (bif:294) */
    char out_dir[256];   /* "./out"     (bif:15) */
    char out_name[32];   /* "lid","pos","bif","coronary" (ldc:585, pos:906, bif:1097, cor:950) */
} lbm_case_desc;

/* Fill `d` with the constants hard-coded in the reference program for `rule`
 * (SURVEY A.7): dims, tau, u_max, unit converters, BC table, paths, names. */
int lbm_case_defaults(int32_t case_rule, lbm_case_desc *d);

/* replaces the global malloc/cudaMalloc block of main() (bif:1185-1222) */
int lbm_create(const lbm_case_desc *desc, lbm_handle *out);
/* replaces the free/cudaFree block (bif:1294-1322) */
int lbm_destroy(lbm_handle h);
const char *lbm_last_error(lbm_handle h); /* h may be NULL: last create() error */

/* Supply the binary voxel field from memory instead of geo_path (Cartesian,
 * GLOBAL box; host pointer).  Optional. */
int lbm_set_flag(lbm_handle h, const int32_t *flag_cartesian);
/* Same for one z-slab of a large box: `flag` holds planes [z_first, z_first+z_count) only, one byte
 * per voxel, [z][y][x].  The planes must cover this handle's owned range extended by 3 planes on
 * each interior side (labels look 1 plane, the -1 marking 1 more, the halo 1 more).  The planes are
 * uploaded to the device before the call returns; the caller's buffer is not referenced afterwards. */
int lbm_set_flag_slab(lbm_handle h, const uint8_t *flag, int32_t z_first, int32_t z_count);

/* geo_pre(): ldc:468-502, pos:52-254, bif:36-239, cor:31-260.  Reads geo_path
 * unless lbm_set_flag was called (LDC / POISEUILLE masks are analytic).  Label
 * stencil + outer-wall-neighbour marking run as CUDA kernels. */
int lbm_geo_pre(lbm_handle h);

/* index_transform(): pos:257-271, bif:241-252, cor:262-273.  GPU stream
 * compaction (flag -> exclusive scan -> scatter).  *nlattice = stored nodes of
 * the GLOBAL box when compact_offset/total were supplied, else of this slab. */
int lbm_index_transform(lbm_handle h, int64_t *nlattice);
/* multi-slab: stored-node count of the owned planes (call after geo_pre), then
 * tell the handle the running offset of its slab and the global total, so that
 * compact indices equal the single-domain z,y,x numbering. */
int lbm_local_stored_count(lbm_handle h, int64_t *count);
int lbm_set_compact_offset(lbm_handle h, int64_t offset, int64_t total);

/* read_vel(): bif:255-327 (bc_path) -- or the planes directly (host, float[nz*nx] each, GLOBAL) */
int lbm_read_vel(lbm_handle h);
int lbm_set_bc_planes(lbm_handle h, const float *inlet_uy, const float *outlet_uy);

/* initialize(): ldc:504-580, pos:273-382, bif:329-427, cor:277-350 */
int lbm_initialize(lbm_handle h);

/* n iterations of { update; boundary_stream; swap }: ldc:654-666, bif:1249-1257.
 * Macroscopic moments (bif:592-595) are materialised on the last of the n steps. */
int lbm_step(lbm_handle h, int32_t n);
/* same, timed with CUDA events on the library's own stream (ms for the n steps) */
int lbm_step_timed(lbm_handle h, int32_t n, float *elapsed_ms);
int64_t lbm_step_count(lbm_handle h);
/* number of kernels the library has launched on this handle so far */
int64_t lbm_launch_count(lbm_handle h);

typedef enum {
    LBM_RES_VELSUM = 0, /* S = sum_i sqrt(ux^2+uy^2+uz^2) over all stored entries   (ldc:460-466,662; pos:895-901,996) */
    LBM_RES_U2SUM = 1   /* sum of |u|^2 over fluid nodes of the trimmed box          (bif:1158-1175, cor:1013-1030) */
} lbm_residual_kind;
/* value of the reduction for the current moments (device reduction, double) */
int lbm_residual(lbm_handle h, int32_t kind, double *value);

/* copies of h_geo / h_index (Cartesian int32, this handle's owned planes
 * [z_begin,z_end) ) */
int lbm_get_geo(lbm_handle h, int32_t *geo_cartesian);
int lbm_get_index(lbm_handle h, int32_t *index_cartesian);
/* D2H of d_rho,d_ux,d_uy,d_uz (bif:1261-1264): compact order, entries of the
 * owned planes only, `real` = handle precision, never-updated entries are 0.
 * `first`/`count` receive the compact range written (may be NULL). */
int lbm_get_fields(lbm_handle h, void *rho, void *ux, void *uy, void *uz, int64_t *first, int64_t *count);
/* debug: the 19 populations "as if in d_scr after the swap", real[19][count], compact order */
int lbm_debug_get_populations(lbm_handle h, void *f);
int64_t lbm_num_fluid(lbm_handle h); /* fluid nodes owned by this handle */
int64_t lbm_device_bytes(lbm_handle h);

/* outputSave(t): ldc:582-610, pos:903-938, bif:1095-1156, cor:948-1011 --
 * byte-compatible ASCII legacy VTK under out_dir.  Single-domain handles only. */
int lbm_output_save(lbm_handle h, int32_t t);

/* Output format of lbm_output_save and of the run loops (SURVEY 8f.2: at 512^3 the ASCII writer
 * dominates wall time).  LBM_OUT_ASCII_VTK (default) is the reference's format, byte for byte.
 * LBM_OUT_BINARY_VTK writes the same points, fields and unit conversions as legacy-VTK BINARY
 * (big-endian float32) to <out_dir>/<out_name>_<t>_bin.vtk; a z-slab handle writes its own planes
 * to <out_name>_<t>_bin.z<first plane>.vtk with ORIGIN shifted accordingly, so the ranks of a
 * multi-GPU run write in parallel and the pieces tile the single-domain file. */
enum { LBM_OUT_ASCII_VTK = 0, LBM_OUT_BINARY_VTK = 1 };
int lbm_set_output_format(lbm_handle h, int32_t format);

/* The reference main loops, including CONVERGENCE.log and the stdout lines:
 *  fixed:    for i in 0..repeat inclusive, save every time_save      (bif:1246-1274, cor:1100-1132)
 *  converge: while k<=max_it && tol_count<=stag_max, residual each step (ldc:653-685, pos:986-1019) */
int lbm_run_fixed(lbm_handle h, int32_t repeat, int32_t time_save, int32_t write_files);
int lbm_run_converge(lbm_handle h, int32_t max_it, double tol, int32_t stag_max, int32_t time_save,
                     int32_t write_files, int32_t *iterations, double *residual);

/* ---- checkpoint / restart (the reference has none: its periodic VTK is output only) ----
 * Binary dump of the population buffer(s) this handle needs to continue, the step counter and a
 * header that pins case rule, dims, slab range, precision and storage; lbm_checkpoint_load restores
 * a handle that was set up (geo_pre .. initialize) for the same case.  A restarted run continues
 * bit-identically. */
int lbm_checkpoint_save(lbm_handle h, const char *path);
int lbm_checkpoint_load(lbm_handle h, const char *path);

/* ---- z-slab halo exchange (SURVEY 8e): the 5 populations crossing each face ----
 * side 0 = low-z face (sends q with c_z=-1, receives c_z=+1), side 1 = high-z.
 * lbm_halo_buffers returns DEVICE pointers to the contiguous send / receive
 * staging buffers of that side (dense storage: 5 * nx_pitch * ny reals each; sparse storage: 5 reals per
 * stored node of the outermost owned plane / of the halo plane, so the two sizes differ) for the caller's
 * transport (NCCL send/recv, or a peer GPU's kernel storing straight into it).
 * lbm_step_begin .. lbm_step_end bracket one step:
 *   begin:    face planes computed first, send buffers packed (async on the handle's stream)
 *   <caller posts the transfers send->recv between neighbouring handles on its transport stream>
 *   interior: the remaining planes, overlapping the transfer (implied by end if omitted)
 *   <caller makes the handle's stream wait for the transfers>
 *   end:      received populations unpacked into the halo planes, buffers swap. */
int lbm_halo_buffers(lbm_handle h, int32_t side, void **send_dev, void **recv_dev, size_t *send_bytes,
                     size_t *recv_bytes);
#define LBM_STEP_MOMENTS 1 /* materialise rho,u on this step (bif:592-595) */
#define LBM_STEP_VELSUM 2  /* also accumulate S = sum|u| for lbm_last_velsum (ldc:660-662) */
int lbm_step_begin(lbm_handle h, int32_t flags);
int lbm_step_interior(lbm_handle h);
int lbm_step_end(lbm_handle h);
/* S of the most recent step run with LBM_STEP_VELSUM (this slab's share) */
int lbm_last_velsum(lbm_handle h, double *value);
/* ---- fused peer-to-peer halo exchange ----
 * Instead of pack -> transport -> unpack, the step kernel itself stores the 5 crossing populations of
 * every FLUID node of a face plane straight into the neighbouring slab's halo plane (device memory of
 * another GPU mapped over NVLink, or of another handle on the same GPU).  Only fluid threads exist,
 * so solid halo slots are never clobbered and no unpack mask is needed.  The caller still has to
 * order the steps: a slab may start step t+1 only after both neighbours finished step t.
 *   lbm_p2p_export: IPC handles + raw pointers of the two population buffers, the byte offset of each
 *                   buffer inside the allocation its handle maps (small cudaMalloc blocks are
 *                   sub-allocated: two buffers can share one handle), their q stride, and the
 *                   cell/compact offset of this slab's low and high halo planes;
 *   lbm_p2p_open / lbm_p2p_close: map / unmap another process's buffer (cudaIpcOpenMemHandle);
 *   lbm_p2p_attach: side 0/1 now pushes into the neighbour's buffers (peer_a/peer_b in the same order
 *                   as exported) at peer_halo_c0 = the neighbour's halo-plane offset facing this slab;
 *                   peer_face_c0 = offset of the neighbour's outermost OWNED plane on that side, which
 *                   the odd step of the in-place (AA) storage pushes into.  With in-place storage the
 *                   peer stores are the only transport: attach before stepping a slab.  Null buffers
 *                   detach.  While either side of the slab holds a mailbox (lbm_mail_attach or
 *                   lbm_mail_stage), this returns LBM_ERR_STATE: detach it first. */
typedef struct {
    unsigned char bytes[64];
} lbm_ipc_handle;
int lbm_p2p_export(lbm_handle h, lbm_ipc_handle handles[2], void *ptrs[2], int64_t byte_offset[2], int64_t *qstride,
                   int64_t halo_c0[2], int64_t face_c0[2]);
int lbm_p2p_open(const lbm_ipc_handle *handle, void **dev_ptr);
int lbm_p2p_close(void *dev_ptr);
int lbm_p2p_attach(lbm_handle h, int32_t side, void *peer_a, void *peer_b, int64_t peer_qstride, int64_t peer_halo_c0,
                   int64_t peer_face_c0);

/* ---- a slab's time loop entirely inside the library ----
 * lbm_slab_step runs n steps of a z-slab with nothing but kernel launches on the host: the crossing
 * populations travel by the fused peer stores above and the ORDERING with the two neighbours (a slab may
 * touch the planes it shares with a neighbour only after that neighbour finished the face launches of the
 * previous step) is decided on the device -- no global barrier, no NCCL, no host thread in the loop.
 * Between processes (one rank per GPU) the neighbours report their progress into a small sync block in
 * this slab's memory: lbm_sync_export publishes it like lbm_p2p_export publishes the buffers,
 * lbm_sync_attach(side, pointer to the NEIGHBOUR's block as mapped here by lbm_p2p_open) connects one
 * side; attach on every slab before any of them steps again (it also restarts the step count the two
 * sides compare, so repeat it after lbm_checkpoint_load).  A wait that sees no progress for 20 s gives up
 * and the call returns LBM_ERR_CUDA instead of hanging the device.
 * flags_last: LBM_STEP_MOMENTS materialises rho,u on the last step.  S_out (optional, n doubles) receives
 * this slab's share of S = sum|u| of every step (ldc.cu:660-662); the caller all-reduces it. */
int lbm_slab_step(lbm_handle h, int32_t n, int32_t flags_last, double *S_out, float *elapsed_ms);
int lbm_sync_export(lbm_handle h, lbm_ipc_handle *handle, void **ptr, int64_t *byte_offset);
int lbm_sync_attach(lbm_handle h, int32_t side, void *peer_sync);

/* ---- mailboxes: the fused exchange of the dense in-place storage without mapping the population buffers ----
 * cudaIpcOpenMemHandle costs 50-65 ms per GB of the allocation it maps (0.74 s for a 512^3 fp64 slab), and a
 * neighbour only ever writes the 5 populations that cross the face.  lbm_mail_export(side) creates this slab's
 * mailbox of that side -- 10 planes: the entering populations as its odd step pulls them from the halo plane and as
 * its even step reads them in its outermost owned plane -- and publishes it like lbm_p2p_export publishes the
 * buffers; lbm_mail_attach(side, the NEIGHBOUR's mailbox of the facing side as mapped here) switches that face over:
 * the face launches read the entering populations from the own mailbox (base-pointer redirection, the kernel does
 * not know) and store the leaving ones into the neighbour's.  Both slabs of a face switch together, between two
 * steps; checkpoints and lbm_debug_get_populations see the complete population buffer (the mailbox is drained and
 * re-filled around them).  LBM_STORE_DENSE_AA only.  A null peer_mail detaches either kind of mailbox; while either side
 * of the slab holds mapped buffers (lbm_p2p_attach) or a staged mailbox, this returns LBM_ERR_STATE: detach it first. */
int lbm_mail_export(lbm_handle h, int32_t side, lbm_ipc_handle *handle, void **ptr, int64_t *byte_offset, int64_t *stride,
                    int64_t *guard);
int lbm_mail_attach(lbm_handle h, int32_t side, void *peer_mail);
/* The same exchange where the neighbour's memory cannot be mapped (no peer access: the NCCL / copy transport).
 * lbm_mail_stage(side) creates the mailbox of that side and two staging buffers; from then on the face launches
 * store the leaving populations into the local send part, lbm_halo_buffers(side) returns the send / receive part
 * of the current step (5 planes each), the caller moves send -> the neighbour's receive between lbm_step_begin and
 * lbm_step_end (ordered on lbm_stream), and lbm_step_end merges what arrived into the mailbox.  Steps are driven
 * with lbm_step_begin / lbm_step_interior / lbm_step_end as for the two-buffer storage; lbm_mail_attach(side, NULL) ends
 * it.  While either side of the slab holds mapped buffers or a mapped mailbox, this returns LBM_ERR_STATE: detach it. */
int lbm_mail_stage(lbm_handle h, int32_t side);

/* ---- several z-slabs driven from ONE process: the multi-GPU form of the reference's main() ----
 * (SURVEY 8b `lbm_create_distributed`; the reference is single-GPU, ldc.cu:612-717.)
 * nslabs contiguous z ranges of desc's box, slab r on CUDA device devices[r] (NULL: r modulo the device
 * count; several slabs may share a device).  lbm_group_setup = geo_pre, index_transform (numbering
 * continued across slabs: bif:241-252), read_vel, initialize on every slab, then peer access + fused
 * peer-store exchange + event ordering between neighbours.  flag_cartesian / the bc planes are optional
 * (NULL: geo_path / bc_path as in the single-domain calls).  The run loops and writers below are the
 * single-domain ones with "all-reduced" reductions: S and sum(u^2) are the sums of the slabs' shares. */
typedef struct lbm_group_s *lbm_group;
int lbm_create_distributed(const lbm_case_desc *desc, int32_t nslabs, const int32_t *devices, lbm_group *out);
int lbm_group_destroy(lbm_group g);
const char *lbm_group_last_error(lbm_group g); /* g may be NULL: last lbm_create_distributed error */
int32_t lbm_group_size(lbm_group g);
lbm_handle lbm_group_slab(lbm_group g, int32_t r); /* the r-th slab's handle (owned by the group) */
int lbm_group_setup(lbm_group g, const int32_t *flag_cartesian, const float *inlet_uy, const float *outlet_uy,
                    int64_t *nlattice);
int lbm_group_step(lbm_group g, int32_t n, float *elapsed_ms); /* ms: host clock around the synchronised loop */
int64_t lbm_group_num_fluid(lbm_group g);
int lbm_group_residual(lbm_group g, int32_t kind, double *value);
int lbm_group_get_fields(lbm_group g, void *rho, void *ux, void *uy, void *uz); /* NLATTICE entries each */
int lbm_group_get_index(lbm_group g, int32_t *index_cartesian);                 /* whole box */
int lbm_group_set_output_format(lbm_group g, int32_t format);
int lbm_group_output_save(lbm_group g, int32_t t); /* ASCII: ONE file, byte-identical to the single-domain one */
int lbm_group_run_fixed(lbm_group g, int32_t repeat, int32_t time_save, int32_t write_files);
int lbm_group_run_converge(lbm_group g, int32_t max_it, double tol, int32_t stag_max, int32_t time_save,
                           int32_t write_files, int32_t *iterations, double *residual);
/* lbm_set_collision on every slab of the group (all or none: the arguments are checked before any slab changes) */
int lbm_group_set_collision(lbm_group g, int32_t model, double magic);

/* Tuning knobs that are not part of a case description.  "persistent": 1 runs batches of steps of the in-place
 * sparse storage in one cooperative launch with a grid barrier between steps (for grids that live in L2); 0 or
 * -1 (the default): one launch per step, which measured as fast or faster on the reference's 64^3 cases.
 * "overlap_launches": 1 (default) launches the step kernels of the in-place storages with programmatic stream
 * serialization, so that a step's launch latency and geometry loads overlap the previous step's tail (a 64^3
 * step: 9.9 -> 7.6 us); 0 serialises launches the ordinary way.  Single-domain handles only. */
int lbm_set_option(lbm_handle h, const char *name, double value);

/* Collision operator.  LBM_COLL_BGK (the default; a handle that never calls this steps exactly as before):
 *     f_q <- f_q - (f_q - feq_q) / tau.
 * LBM_COLL_TRT, two relaxation times (Ginzburg, Verhaeghe & d'Humieres, Commun. Comput. Phys. 3, 2008): with
 * the opposite direction qbar of q,
 *     n+ = (f_q + f_qbar)/2 - (feq_q + feq_qbar)/2      n- = (f_q - f_qbar)/2 - (feq_q - feq_qbar)/2
 *     f_q <- f_q - om+ n+ - om- n-                      f_0 <- f_0 - om+ (f_0 - feq_0)
 * om+ = 1/tau sets the viscosity as for BGK; om- = 1 / (1/2 + magic / (tau - 1/2)), i.e. the magic parameter
 * Lambda = (1/om+ - 1/2)(1/om- - 1/2) = magic.  At fixed Lambda the steady bounce-back solution does not depend on
 * tau: Lambda = 3/16 puts a straight wall exactly half-way for Poiseuille flow, Lambda = 1/4 is the usual choice
 * for stability.  Lambda = (tau - 1/2)^2 gives om- = om+, i.e. BGK.
 * Inlet / outlet / lid links under TRT: the node's post-collision non-equilibrium n_q = g_q - feq_q(rho_x, u_x) is
 * split with the opposite link and relaxed like the collision,
 *     feq_q(rho_bc, u_bc) + (1 - om+) (n_q + n_qbar)/2 + (1 - om-) (n_q - n_qbar)/2,
 * which is the BGK rule feq_q(rho_bc, u_bc) + n_q (1 - 1/tau) when om- = om+.  Bounce-back and static links are
 * unchanged.  TRT exists in LBM_MATH_FAST arithmetic only (STRICT is the reference's expression order, and the
 * reference has no TRT).
 * Callable any time after lbm_create; takes effect from the next step.  LBM_ERR_STATE inside lbm_step_begin ..
 * lbm_step_end; LBM_ERR_ARG for an unknown model, a magic parameter that is not finite and > 0 (TRT; ignored for
 * BGK), tau <= 1/2 with TRT, or TRT on an LBM_MATH_STRICT handle -- the handle then keeps its operator.
 * Checkpoints of a TRT run carry the operator and Lambda: only a handle with the same ones loads them. */
int lbm_set_collision(lbm_handle h, int32_t model, double magic);

/* Self-checking build of the library (-DLBM_SELFCHECK; tools/selfcheck.py builds and runs it -- the stand-in for
 * compute-sanitizer, which the GPU pool does not offer): out[0] = population accesses of the step kernels that
 * fell outside the handle's buffers, out[1] = buffer elements touched by two different threads within one launch
 * (the in-place storage relies on there being none), out[2] = step-kernel launches checked.  A normal build
 * returns LBM_ERR_STATE. */
int lbm_debug_selfcheck(lbm_handle h, uint64_t out[3]);

/* write_once(): cor.cu:1033-1051 -- "x,y,z,ux,uy,uz" (%f) of every inlet / outlet node (labels 2,3,5,6,7) */
int lbm_write_bc_csv(lbm_handle h, const char *path);

/* cudaStream_t of the handle as an opaque pointer (for event / NCCL interop) */
void *lbm_stream(lbm_handle h);
int lbm_sync(lbm_handle h);

/* ---- geometry front end: STL surface -> binary voxel field (what geo.txt holds before geo_pre).
 * Replaces the MATLAB pre-processing step the reference does not ship (bifurcation/README.md:1-5:
 * bif.stl -> geo.txt).  Voxel (i,j,k) has its centre at origin + (i+.5, j+.5, k+.5) * spacing; a voxel
 * is inside when the +x ray from -inf to its centre crosses the surface an odd number of times, so
 * the surface must be closed around x (open vessel ends along y or z are fine).  flag_out receives
 * planes [z_begin, z_end) as [z][y][x] bytes (1 inside) -- the layout lbm_set_flag_slab takes, so every
 * rank of a z-slab run voxelises only its own planes.  Deterministic (order-independent XOR marking). */
typedef struct lbm_voxel_grid {
    double origin[3];
    double spacing;
    int32_t nx, ny, nz;
    int32_t reserved;
} lbm_voxel_grid;
int lbm_voxelize_stl(const char *stl_path, const lbm_voxel_grid *grid, int32_t z_begin, int32_t z_end, int32_t device,
                     uint8_t *flag_out);
/* same from memory: tri = [ntri][3 vertices][x,y,z] floats */
int lbm_voxelize_triangles(const float *tri, int64_t ntri, const lbm_voxel_grid *grid, int32_t z_begin, int32_t z_end,
                           int32_t device, uint8_t *flag_out);
const char *lbm_voxel_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* LBM_B200_H */
