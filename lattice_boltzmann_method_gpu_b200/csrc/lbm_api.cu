// Host side of liblbm_b200.so: the solver object behind the opaque handle, the
// C ABI of include/lbm_b200.h, the geo.txt / bc.txt readers and the
// byte-compatible VTK / CONVERGENCE.log writers.
//
// There is deliberately no CPU fallback: without a CUDA device lbm_create
// fails with LBM_ERR_NO_DEVICE.
#include <algorithm>
#include <charconv>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <fstream>
#include <iostream>
#include <new>
#include <sstream>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "lbm_internal.h"
#include "geo_text.h"
#include "vtk_format.h"

namespace lbm {

static thread_local std::string g_create_error;

static std::string fmt(const char *f, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, f);
    vsnprintf(buf, sizeof buf, f, ap);
    va_end(ap);
    return buf;
}

// the argument rules of lbm_set_collision (include/lbm_b200.h); empty: accepted
static std::string collision_refusal(const lbm_case_desc &d, int model, double magic) {
    if (model == LBM_COLL_BGK) return "";
    if (model != LBM_COLL_TRT) return fmt("unknown collision model %d (LBM_COLL_BGK = 0, LBM_COLL_TRT = 1)", model);
    if (!std::isfinite(magic) || !(magic > 0.0)) return fmt("TRT magic parameter must be finite and > 0 (got %g)", magic);
    if (!(d.tau > 0.5)) return fmt("TRT needs tau > 1/2 (tau = %g)", d.tau);
    if (d.math == LBM_MATH_STRICT)
        return "TRT exists in LBM_MATH_FAST arithmetic only (STRICT is the reference's expression order, which has no TRT)";
    return "";
}

struct SolverBase {
    virtual ~SolverBase() {}
    std::string err;
    lbm_case_desc d{};
    virtual int set_flag(const int32_t *flag) = 0;
    virtual int set_flag_slab(const uint8_t *flag, int z_first, int z_count) = 0;
    virtual int geo_pre() = 0;
    virtual int index_transform(int64_t *nlat) = 0;
    virtual int local_stored_count(int64_t *n) = 0;
    virtual int set_compact_offset(int64_t off, int64_t total) = 0;
    virtual int read_vel() = 0;
    virtual int set_bc_planes(const float *in, const float *out) = 0;
    virtual int initialize() = 0;
    virtual int step(int n, float *ms) = 0;
    virtual int step_begin(int flags) = 0;
    virtual int step_interior() = 0;
    virtual int step_end() = 0;
    virtual int last_velsum(double *v) = 0;
    // n steps of a z-slab with every ordering decision on the device (flags in peer memory across
    // processes, events inside one process); S_out (optional, n doubles): this slab's share of sum|u| per step
    virtual int slab_steps(int n, int flags_last, double *S_out, float *ms) = 0;
    virtual int sync_export(lbm_ipc_handle *h, void **ptr, int64_t *boff) = 0;
    virtual int sync_attach(int side, void *peer_sync) = 0;
    virtual int mail_export(int side, lbm_ipc_handle *h, void **ptr, int64_t *boff, int64_t *ms, int64_t *guard) = 0;
    virtual int mail_attach(int side, void *peer_mail) = 0;
    virtual int mail_stage(int side) = 0;
    virtual void set_inproc_neighbour(int side, SolverBase *nb) = 0;
    virtual cudaEvent_t face_event(int k) = 0;
    virtual int enqueue_step(int flags, double *acc_slot) = 0;  // begin + interior + end, no host sync
    virtual int fetch_acc(int first, int n, double *out) = 0;
    virtual int zero_acc(int first, int n) = 0;
    virtual double *acc_slot(int k) = 0;
    virtual int write_global(int t, const int32_t *index_global, const void *rho, const void *ux, const void *uy,
                             const void *uz, int64_t nlattice) = 0;
    virtual int residual(int kind, double *v) = 0;
    virtual int get_geo(int32_t *g) = 0;
    virtual int get_index(int32_t *g) = 0;
    virtual int get_fields(void *rho, void *ux, void *uy, void *uz, int64_t *first, int64_t *count) = 0;
    virtual int get_populations(void *f) = 0;
    virtual int output_save(int t) = 0;
    virtual int write_bc_csv(const char *path) = 0;
    int out_format = LBM_OUT_ASCII_VTK;
    virtual int run_fixed(int repeat, int time_save, int write_files) = 0;
    virtual int run_converge(int max_it, double tol, int stag_max, int time_save, int write_files, int *its,
                             double *res) = 0;
    virtual int checkpoint(const char *path, bool save) = 0;
    virtual int p2p_export(lbm_ipc_handle *h2, void **ptrs, int64_t *boff, int64_t *qs, int64_t *halo_c0, int64_t *face_c0) = 0;
    virtual int p2p_attach(int side, void *pa, void *pb, int64_t pqs, int64_t pc0, int64_t pown) = 0;
    virtual int halo_buffers(int side, void **send, void **recv, size_t *send_bytes, size_t *recv_bytes) = 0;
    virtual int sync() = 0;
    virtual void *stream_ptr() = 0;
    virtual int selfcheck(uint64_t *out2) = 0;
    virtual int set_option(const char *name, double value) = 0;
    virtual int set_collision(int model, double magic) = 0;
    int64_t steps = 0, launches = 0, nfluid = 0, dev_bytes = 0;
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            err = fmt("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return e_ == cudaErrorMemoryAllocation ? LBM_ERR_NOMEM : LBM_ERR_CUDA;                 \
        }                                                                                          \
    } while (0)
#define FAIL(code, ...)         \
    do {                        \
        err = fmt(__VA_ARGS__); \
        return code;            \
    } while (0)

template <typename T>
struct Solver final : SolverBase {
    cudaStream_t st = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    Box ext{}, box{};
    int own_z0 = 0, own_z1 = 0;
    bool lo_halo = false, hi_halo = false;
    int fluid_label = 4;
    GeoRules rules{};
    BcEntry bc[LBM_MAX_BC]{};
    // stage flags
    bool have_flag = false, have_geo = false, have_index = false, have_init = false, have_planes = false;
    bool have_moments = false, in_step = false;
    int step_flags = 0;
    // host
    std::vector<int32_t> h_flag;  // global Cartesian, optional
    bool flag_on_device = false;       // d_flag holds the planes lbm_set_flag_slab was given
    std::vector<float> h_in, h_out;
    // device
    uint8_t *d_flag = nullptr;
    int32_t *d_label_ext = nullptr, *d_label = nullptr, *d_index = nullptr, *d_scratch = nullptr;
    uint32_t *d_node = nullptr, *d_wall = nullptr, *d_wallc = nullptr;
    uint8_t *d_seg = nullptr;
    int8_t *d_label8 = nullptr;
    T *d_fa = nullptr, *d_fb = nullptr, *d_cur = nullptr, *d_nxt = nullptr;
    T *d_rho = nullptr, *d_ux = nullptr, *d_uy = nullptr, *d_uz = nullptr;
    T *d_plane_in = nullptr, *d_plane_out = nullptr;
    double *d_acc = nullptr;      // [ACC_SLOTS] reduction slots
    long long *d_cnt = nullptr;   // small device counters
    static constexpr int ACC_SLOTS = 64;
    long long qstride = 0;
    int64_t stored_own = 0, compact_first = 0, compact_total = -1;
    bool offset_set = false;
    size_t scratch_ints = 0;
    double last_S = 0.0;
    std::vector<long long> plane_first;  // [planes of the state box + 1] global compact id each plane starts at
    T *d_stage = nullptr;                // staging of get_fields (dense storage), two plane groups in flight
    size_t stage_elems = 0;
    cudaStream_t st_copy = nullptr;
    cudaEvent_t ev_gathered[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    long long pend_i0 = 0, pend_i1 = 0;
    bool interior_pending = false;
    // How the populations crossing one z face reach the neighbour (include/lbm_b200.h, "z-slab halo exchange" on):
    //   PACKED          the step packs them into `send` and unpacks the neighbour's from `recv`; the caller moves the bytes
    //   PEER_BUFFERS    the face launches store into the neighbour's population buffers (lbm_p2p_attach)
    //   MAILBOX         ... into the neighbour's mailbox, and read the entering ones from `mail` (lbm_mail_attach)
    //   STAGED_MAILBOX  ... into `stage_out`; the caller moves it to the neighbour's `stage_in`, which lbm_step_end
    //                   merges into `mail` (lbm_mail_stage)
    // The kinds change only in the "slab faces" section (relink, unlink_*); a step asks the face what to do there too.
    enum class Link { PACKED, PEER_BUFFERS, MAILBOX, STAGED_MAILBOX };
    struct Face {
        Link kind = Link::PACKED;
        T *send = nullptr, *recv = nullptr;       // pack / unpack buffers, allocated by initialize for every kind
        T *peer_buf[2] = {nullptr, nullptr};      // PEER_BUFFERS: the neighbour's two buffers in export order,
        long long peer_qs = 0, peer_c0 = 0, peer_own = 0;  // their q stride, halo-plane and outermost-owned-plane offsets
        T *mail = nullptr;                        // own mailbox (lbm_mail_export, 10 planes), kept when the kind changes
        T *peer_mail = nullptr;                   // MAILBOX: the neighbour's mailbox as mapped here; STAGED: stage_out
        bool mail_live = false;  // the mailbox, not the population buffer, holds the current values of its slots
        T *stage_out = nullptr, *stage_in = nullptr;  // STAGED_MAILBOX: send / receive parts, A and B halves each
        unsigned long long *peer_sync = nullptr;  // ordering: where this slab reports its progress (other process), or
        SolverBase *inproc_nb = nullptr;          // the neighbour whose face events it waits for (same process)
        bool mailbox() const { return kind == Link::MAILBOX || kind == Link::STAGED_MAILBOX; }
    };
    Face face[2];                                       // [0] low-z side, [1] high-z side
    long long mail_ms = 0, mail_G = 0;                  // mailbox plane stride and guard (StepParams::mail)
    unsigned long long *d_sync = nullptr;               // [0] low neighbour's progress, [1] high neighbour's, [2] timeout
    int64_t sync_base = 0;                              // step count at which the progress counters were zero
    cudaEvent_t ev_face[2] = {nullptr, nullptr};        // recorded after the face launches of even / odd steps
    // sparse storage (reference compact order + run segments)
    bool sparse = false;
    long long n_lo_stored = 0, stored_box = 0;   // stored nodes of the low halo plane / of the whole state box
    long long sp_first = 0;                      // global compact id of the first stored node of the state box
    long long nseg = 0;
    long long *d_cart = nullptr, *d_chunk_off = nullptr, *d_plane_seg = nullptr;
    uint32_t *d_nodec = nullptr;
    int8_t *d_labelc = nullptr;
    int32_t *d_rec = nullptr, *d_chunk_cnt = nullptr;
    std::vector<long long> seg_plane_start;      // [owned planes + 1]
    // in-place sparse storage: its own numbering (fluid nodes + single-cell x gaps), see lbm_geo.cu k_span_flags
    int32_t *d_sid = nullptr;
    uint2 *d_cmeta = nullptr;
    uint32_t *d_rec_links = nullptr;
    int32_t *d_bcslot = nullptr;     // in-place sparse storage: precomputed inlet / outlet link lists (k_bc_links)
    BcLink<T> *d_bclinks = nullptr;
    std::vector<long long> sid_plane_first;      // [planes of the state box + 1] first own-numbering id of each plane
    long long own_id0 = 0, own_id1 = 0;          // ids (storage numbering, local) of the owned planes
    long long halo_id0[2] = {0, 0}, halo_n[2] = {0, 0};   // compact range of the halo plane per side
    long long face_id0[2] = {0, 0}, face_n[2] = {0, 0};   // compact range of the outermost owned plane per side

    ~Solver() override {
        join_writer();
        cudaSetDevice(d.device);
        auto fr = [](void *p) {
            if (p) cudaFree(p);
        };
        fr(d_flag), fr(d_label_ext), fr(d_label), fr(d_index), fr(d_scratch), fr(d_node), fr(d_seg), fr(d_label8);
        fr(d_fa), fr(d_fb == d_fa ? nullptr : d_fb), fr(d_rho), fr(d_ux), fr(d_uy), fr(d_uz), fr(d_plane_in), fr(d_plane_out);
        fr(d_acc), fr(d_cnt);
        fr(d_sid), fr(d_cmeta), fr(d_rec_links), fr(d_bcslot), fr(d_bclinks);
        fr(d_stage), fr(d_wall), fr(d_wallc), fr(d_cart), fr(d_chunk_off), fr(d_nodec), fr(d_labelc), fr(d_rec), fr(d_chunk_cnt), fr(d_plane_seg);
        for (Face &f : face) fr(f.send), fr(f.recv), fr(f.mail), fr(f.stage_out), fr(f.stage_in);
        fr(d_sync), fr(d_chk_shadow[0]), fr(d_chk_shadow[1]), fr(d_chk_count), fr(d_pulse), fr(d_barrier);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        for (auto &e : ev_face)
            if (e) cudaEventDestroy(e);
        for (int k = 0; k < 2; k++) {
            if (ev_gathered[k]) cudaEventDestroy(ev_gathered[k]);
            if (ev_copied[k]) cudaEventDestroy(ev_copied[k]);
        }
        if (st_copy) cudaStreamDestroy(st_copy);
        if (st) cudaStreamDestroy(st);
    }

    // the LDC rule stores every node of the box (ldc.cu:54); the others store geo != 0
    int store_all() const { return d.case_rule == LBM_CASE_LDC ? 1 : 0; }

    std::vector<std::pair<void *, size_t>> allocs;  // what dalloc handed out (for dev_bytes and dfree)
    template <typename U>
    int dalloc(U **p, size_t n) {
        CK(cudaMalloc((void **)p, std::max<size_t>(n, 1) * sizeof(U)));
        dev_bytes += (int64_t)(n * sizeof(U));
        allocs.emplace_back((void *)*p, n * sizeof(U));
        return 0;
    }
    template <typename U>
    void dfree(U **p) {
        if (!*p) return;
        for (auto &a : allocs)
            if (a.first == (void *)*p) {
                dev_bytes -= (int64_t)a.second;
                a = allocs.back();
                allocs.pop_back();
                break;
            }
        cudaFree((void *)*p);
        *p = nullptr;
    }
    // Buffers whose size depends on the GEOMETRY (stored-node counts, records, face sizes) and not only
    // on the box: released whenever geo_pre runs again, so that a handle re-initialised with a larger
    // mask never writes past allocations sized for the previous one.
    void release_geometry_sized() {
        if (d_fb == d_fa) d_fb = nullptr;
        dfree(&d_fa), dfree(&d_fb), dfree(&d_rho), dfree(&d_ux), dfree(&d_uy), dfree(&d_uz);
        dfree(&d_cart), dfree(&d_nodec), dfree(&d_wallc), dfree(&d_labelc), dfree(&d_rec), dfree(&d_chunk_cnt);
        dfree(&d_cmeta), dfree(&d_rec_links), dfree(&d_bcslot), dfree(&d_bclinks);
        dfree(&d_chunk_off), dfree(&d_plane_seg);
        if (d_stage) cudaFree(d_stage), d_stage = nullptr, stage_elems = 0;
        d_cur = d_nxt = nullptr;
        unlink_geometry_sized();
    }

    int setup() {
        CK(cudaSetDevice(d.device));
        CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        CK(cudaEventCreate(&ev0));
        CK(cudaEventCreate(&ev1));
        for (auto &e : ev_face) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        fluid_label = d.case_rule == LBM_CASE_LDC ? 3 : 4;
        own_z0 = d.z_begin, own_z1 = d.z_end;
        lo_halo = own_z0 > 0, hi_halo = own_z1 < d.nz;
        const int px = ((d.nx + 31) / 32) * 32;
        box.nx = d.nx, box.ny = d.ny, box.nz = d.nz, box.px = px, box.plane = (long long)px * d.ny;
        box.z0 = own_z0 - (lo_halo ? 1 : 0), box.z1 = own_z1 + (hi_halo ? 1 : 0);
        ext = box;
        ext.z0 = std::max(0, own_z0 - 3), ext.z1 = std::min(d.nz, own_z1 + 3);
        // compact indices are int32, like the reference's h_index (bifurcation.cu:22)
        if (box.cells() >= (1LL << 31)) FAIL(LBM_ERR_ARG, "slab of %lld cells exceeds the int32 index range: use more z-slabs", box.cells());
        rules.case_rule = d.case_rule;
        rules.n_open = d.n_openings;
        for (int i = 0; i < d.n_openings; i++) rules.open[i] = d.openings[i];
        rules.mark_sources = d.case_rule == LBM_CASE_LDC ? 0u
                             : d.case_rule == LBM_CASE_POISEUILLE ? ((1u << 1) | (1u << 2) | (1u << 3))
                                                                  : (1u << 1);
        for (auto &e : bc) e = BcEntry{LBM_BC_NONE, 0, 0, 0, 0, 0, 0.0, 0.0};
        for (int i = 0; i < d.n_bc; i++) {
            const lbm_bc_desc &s = d.bc[i];
            if (s.label < 1 || s.label >= LBM_MAX_BC || s.label == fluid_label)
                FAIL(LBM_ERR_ARG, "bc[%d]: label %d not a boundary label", i, s.label);
            if (s.normal_axis < 0 || s.normal_axis > 2 || s.vel_axis < 0 || s.vel_axis > 2 ||
                (s.normal_sign != 1 && s.normal_sign != -1))
                FAIL(LBM_ERR_ARG, "bc[%d]: bad axis/sign", i);
            bc[s.label] = BcEntry{s.kind, s.normal_axis, s.normal_sign, s.vel_axis, s.source, s.pulsatile, s.value,
                                  s.init_value};
        }
        if (dalloc(&d_acc, ACC_SLOTS) || dalloc(&d_cnt, 8) || dalloc(&d_sync, 8)) return LBM_ERR_NOMEM;
        CK(cudaMemset(d_sync, 0, 8 * sizeof(unsigned long long)));
        return 0;
    }

    // ------------------------------------------------------------ geometry
    int set_flag(const int32_t *flag) override {
        if (!flag) FAIL(LBM_ERR_ARG, "null flag");
        h_flag.assign(flag, flag + (size_t)d.nx * d.ny * d.nz);
        flag_on_device = false;
        have_flag = true;
        return 0;
    }

    int set_flag_slab(const uint8_t *flag, int z_first, int z_count) override {
        if (!flag || z_count <= 0) FAIL(LBM_ERR_ARG, "null / empty flag slab");
        if (z_first > ext.z0 || z_first + z_count < ext.z1)
            FAIL(LBM_ERR_ARG, "flag slab [%d,%d) does not cover the planes [%d,%d) this handle needs", z_first,
                 z_first + z_count, ext.z0, ext.z1);
        // the planes this handle reads go straight into the padded device rows: no host copy is kept (a copy of a
        // 512^3 field alone took 59 ms, more than geo_pre + index_transform + initialize together)
        CK(cudaSetDevice(d.device));
        if (!d_flag && dalloc(&d_flag, (size_t)ext.cells())) return LBM_ERR_NOMEM;
        CK(cudaMemsetAsync(d_flag, 0, (size_t)ext.cells(), st));
        CK(cudaMemcpy2DAsync(d_flag, (size_t)ext.px, flag + (size_t)d.nx * (size_t)d.ny * (size_t)(ext.z0 - z_first), (size_t)d.nx,
                             (size_t)d.nx, (size_t)d.ny * (size_t)(ext.z1 - ext.z0), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
        h_flag.clear();
        flag_on_device = true;
        have_flag = true;
        return 0;
    }

    int load_flag_file() {
        // bif.cu:50-61 (x fastest) or cor.cu:45-56 (y fastest); mapped and parsed by several threads (geo_text.h)
        MappedFile f;
        if (!f.open_ro(d.geo_path)) FAIL(LBM_ERR_IO, "cannot open geometry file '%s'", d.geo_path);
        const long total = (long)d.nx * d.ny * d.nz;
        h_flag.assign((size_t)total, 0);
        int32_t *out = h_flag.data();
        const long nx = d.nx, ny = d.ny, plane = nx * ny;
        long cnt;
        if (!d.geo_yfast) {
            cnt = parse_int_tokens(f.p, f.n, total, 16, [out](long t, int v) { out[t] = v; });
        } else {  // token t = (z * nx + x) * ny + y
            cnt = parse_int_tokens(f.p, f.n, total, 16, [out, nx, ny, plane](long t, int v) {
                const long z = t / plane, r = t - z * plane, x = r / ny, y = r - x * ny;
                out[x + nx * (y + ny * z)] = v;
            });
        }
        if (cnt < total)
            FAIL(LBM_ERR_IO, "geometry file '%s' holds %ld tokens, expected %ld", d.geo_path, cnt, total);
        have_flag = true;
        return 0;
    }

    int geo_pre() override {
        CK(cudaSetDevice(d.device));
        const bool needs_file = d.case_rule == LBM_CASE_GEO_Y_INOUT || d.case_rule == LBM_CASE_GEO_OPENINGS;
        if (needs_file && !have_flag) {
            int r = load_flag_file();
            if (r) return r;
        }
        if (!d_flag && dalloc(&d_flag, (size_t)ext.cells())) return LBM_ERR_NOMEM;
        if (!d_label_ext && dalloc(&d_label_ext, (size_t)ext.cells())) return LBM_ERR_NOMEM;
        if (needs_file && flag_on_device) {
            // lbm_set_flag_slab already put the planes there
        } else if (needs_file) {
            // ext slab of the global int32 field (geo.txt / lbm_set_flag), padded pitch, one byte per voxel
            std::vector<uint8_t> tmp((size_t)ext.cells(), 0);
            const int nthr = std::max(1, std::min({(int)std::thread::hardware_concurrency(), 16, ext.z1 - ext.z0}));
            auto work = [&](int t) {
                const int za = ext.z0 + (int)((long long)(ext.z1 - ext.z0) * t / nthr), zb = ext.z0 + (int)((long long)(ext.z1 - ext.z0) * (t + 1) / nthr);
                for (int z = za; z < zb; z++)
                    for (int y = 0; y < d.ny; y++) {
                        uint8_t *drow = &tmp[(size_t)ext.px * ((size_t)y + (size_t)d.ny * (z - ext.z0))];
                        const int32_t *srow = &h_flag[(size_t)d.nx * ((size_t)y + (size_t)d.ny * z)];
                        for (int x = 0; x < d.nx; x++) drow[x] = (uint8_t)srow[x];
                    }
            };
            std::vector<std::thread> pool;
            for (int t = 1; t < nthr; t++) pool.emplace_back(work, t);
            work(0);
            for (auto &th : pool) th.join();
            CK(cudaMemcpyAsync(d_flag, tmp.data(), tmp.size(), cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));
        } else if (d.case_rule == LBM_CASE_POISEUILLE) {
            CK(launch_make_flag_pos(d_flag, ext, st));
            launches++;
        } else {
            CK(cudaMemsetAsync(d_flag, 0, (size_t)ext.cells(), st));
        }
        CK(launch_labels(d_flag, d_label_ext, ext, rules, st));
        CK(launch_mark(d_label_ext, ext, rules, st));
        launches += 2;
        if (!d_label && dalloc(&d_label, (size_t)box.cells())) return LBM_ERR_NOMEM;
        CK(cudaMemcpyAsync(d_label, d_label_ext + (long long)(box.z0 - ext.z0) * ext.plane,
                           (size_t)box.cells() * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        // owned stored-node count (needed by multi-slab callers before index_transform)
        CK(launch_count_stored(d_label + (long long)(own_z0 - box.z0) * box.plane,
                               (long long)(own_z1 - own_z0) * box.plane, box.px, box.nx, store_all(), d_cnt, st));
        launches++;
        long long c = 0;
        CK(cudaMemcpyAsync(&c, d_cnt, sizeof c, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        stored_own = c;
        join_writer();
        if (have_init && sparse) release_geometry_sized();
        have_geo = true, have_index = false, have_init = false, have_moments = false;
        w_index.clear(), w_rho.clear(), w_ux.clear(), w_uy.clear(), w_uz.clear();  // host mirrors of the old tables
        return 0;
    }

    int local_stored_count(int64_t *n) override {
        if (!have_geo) FAIL(LBM_ERR_STATE, "geo_pre has not run");
        *n = stored_own;
        return 0;
    }
    int set_compact_offset(int64_t off, int64_t total) override {
        compact_first = off, compact_total = total, offset_set = true;
        have_index = false, have_init = false;  // the index table is numbered from `off`
        w_index.clear();
        return 0;
    }

    int index_transform(int64_t *nlat) override {
        if (!have_geo) FAIL(LBM_ERR_STATE, "index_transform before geo_pre");
        CK(cudaSetDevice(d.device));
        if ((lo_halo || hi_halo) && !offset_set)
            FAIL(LBM_ERR_STATE, "slab handle: call lbm_set_compact_offset before lbm_index_transform");
        if (!offset_set) compact_first = 0, compact_total = stored_own;
        if (!d_index && dalloc(&d_index, (size_t)box.cells())) return LBM_ERR_NOMEM;
        long long n_lo = 0;
        if (lo_halo) {
            CK(launch_count_stored(d_label, box.plane, box.px, box.nx, store_all(), d_cnt + 1, st));
            launches++;
            CK(cudaMemcpyAsync(&n_lo, d_cnt + 1, sizeof n_lo, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        scratch_ints = compact_scratch_ints(box.cells());
        if (!d_scratch && dalloc(&d_scratch, scratch_ints)) return LBM_ERR_NOMEM;
        const int nzl = box.z1 - box.z0;
        long long *d_pf = nullptr;
        CK(cudaMalloc((void **)&d_pf, (size_t)nzl * sizeof(long long)));
        cudaError_t ce = launch_compact(d_label, d_index, box.cells(), box.px, box.nx, store_all(),
                                        (long long)compact_first - n_lo, d_scratch, scratch_ints, d_cnt + 2, box.plane, d_pf, st);
        plane_first.assign((size_t)nzl + 1, 0);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(plane_first.data(), d_pf, (size_t)nzl * sizeof(long long), cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        cudaFree(d_pf);
        CK(ce);
        launches += 3;
        // node words, segment classes, int8 labels
        if (!d_node) {
            if (dalloc(&d_node, (size_t)box.cells()) || dalloc(&d_wall, (size_t)box.cells()) || dalloc(&d_seg, (size_t)(box.cells() / 32 + 1)) ||
                dalloc(&d_label8, (size_t)box.cells()))
                return LBM_ERR_NOMEM;
        }
        CK(launch_node_words(d_label, d_node, d_wall, d_seg, d_label8, box, own_z0, own_z1, fluid_label, bc, d_cnt + 3, st));
        launches++;
        long long nf = 0, nbox = 0;
        CK(cudaMemcpyAsync(&nf, d_cnt + 3, sizeof nf, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&nbox, d_cnt + 2, sizeof nbox, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        nfluid = nf;
        n_lo_stored = n_lo, stored_box = nbox, sp_first = (long long)compact_first - n_lo;
        plane_first[(size_t)(box.z1 - box.z0)] = sp_first + nbox;
        have_index = true, have_init = false;
        w_index.clear();
        if (nlat) *nlat = compact_total;
        return 0;
    }

    // label of global cell (x,y,z) for host-side masking; 0 when outside the state box
    int fetch_label_rows(int y, std::vector<int32_t> &rows) {
        // rows[z_local*px + x] for all planes of the state box
        const int nzl = box.z1 - box.z0;
        rows.assign((size_t)nzl * box.px, 0);
        CK(cudaMemcpy2DAsync(rows.data(), (size_t)box.px * sizeof(int32_t), d_label + (long long)y * box.px,
                             (size_t)box.plane * sizeof(int32_t), (size_t)box.px * sizeof(int32_t), nzl,
                             cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return 0;
    }

    int upload_planes() {
        const size_t n = (size_t)d.nx * d.nz;
        if (!d_plane_in && (dalloc(&d_plane_in, n) || dalloc(&d_plane_out, n))) return LBM_ERR_NOMEM;
        std::vector<T> a(n), b(n);
        for (size_t i = 0; i < n; i++) a[i] = (T)h_in[i], b[i] = (T)h_out[i];
        CK(cudaMemcpyAsync(d_plane_in, a.data(), n * sizeof(T), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_plane_out, b.data(), n * sizeof(T), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
        have_planes = true;
        return 0;
    }

    // read_vel(): bif.cu:255-327.  raw planes are masked by the labels at y=1 / y=NY-2.
    int mask_and_store_planes(const float *in, const float *out) {
        if (!have_geo) FAIL(LBM_ERR_STATE, "read_vel before geo_pre");
        std::vector<int32_t> r1, r2;
        int r = fetch_label_rows(1, r1);
        if (r) return r;
        r = fetch_label_rows(d.ny - 2, r2);
        if (r) return r;
        const size_t n = (size_t)d.nx * d.nz;
        h_in.assign(n, 0.f), h_out.assign(n, 0.f);
        for (int z = box.z0; z < box.z1; z++)
            for (int x = 0; x < d.nx; x++) {
                size_t i = (size_t)x + (size_t)z * d.nx, j = (size_t)(z - box.z0) * box.px + x;
                h_in[i] = r1[j] == 2 ? in[i] : 0.f;
                h_out[i] = r2[j] == 3 ? out[i] : 0.f;
            }
        return upload_planes();
    }
    int read_vel() override {
        FILE *f = fopen(d.bc_path, "r");
        if (!f) FAIL(LBM_ERR_IO, "cannot open boundary file '%s'", d.bc_path);
        const size_t n = (size_t)d.nx * d.nz;
        std::vector<float> a(n, 0.f), b(n, 0.f);
        float tmp;
        for (size_t i = 0; i < n; i++) a[i] = fscanf(f, "%f ", &tmp) == 1 ? tmp : 0.f;
        for (size_t i = 0; i < n; i++) b[i] = fscanf(f, "%f ", &tmp) == 1 ? tmp : 0.f;
        fclose(f);
        return mask_and_store_planes(a.data(), b.data());
    }
    int set_bc_planes(const float *in, const float *out) override {
        if (!in || !out) FAIL(LBM_ERR_ARG, "null plane");
        return mask_and_store_planes(in, out);
    }

    // ------------------------------------------------------------ state
    int initialize() override {
        if (!have_index) FAIL(LBM_ERR_STATE, "initialize before index_transform");
        CK(cudaSetDevice(d.device));
        if (d.storage == LBM_STORE_SPARSE_AB || d.storage == LBM_STORE_SPARSE_AA) return initialize_sparse();
        if (d.storage != LBM_STORE_DENSE_AB && d.storage != LBM_STORE_DENSE_AA)
            FAIL(LBM_ERR_ARG, "unknown storage %d", d.storage);
        const bool aa = d.storage == LBM_STORE_DENSE_AA;
        if (d.case_rule == LBM_CASE_GEO_Y_INOUT && !have_planes) {
            h_in.assign((size_t)d.nx * d.nz, 0.f), h_out = h_in;
            int r = upload_planes();
            if (r) return r;
        }
        if (!d_plane_in) {
            h_in.assign((size_t)d.nx * d.nz, 0.f), h_out = h_in;
            int r = upload_planes();
            if (r) return r;
        }
        const long long cells = box.cells();
        qstride = cells + 64;  // de-phase the 19 streams a little; keeps 256-B alignment
        if (!d_fa) {
            // tail guard: the speculative step form pulls for every cell, up to plane+px beyond the last one
            const size_t fsize = (size_t)qstride * Q + (size_t)box.plane + box.px + 64;
            if (dalloc(&d_fa, fsize)) return LBM_ERR_NOMEM;
            CK(cudaMemsetAsync(d_fa, 0, fsize * sizeof(T), st));
            if (aa) {
                d_fb = d_fa;  // one buffer, streamed in place
            } else {
                if (dalloc(&d_fb, fsize)) return LBM_ERR_NOMEM;
                CK(cudaMemsetAsync(d_fb, 0, fsize * sizeof(T), st));
            }
            if (dalloc(&d_rho, (size_t)cells) || dalloc(&d_ux, (size_t)cells) || dalloc(&d_uy, (size_t)cells) ||
                dalloc(&d_uz, (size_t)cells))
                return LBM_ERR_NOMEM;
            for (Face &f : face)
                if (dalloc(&f.send, (size_t)box.plane * 5) || dalloc(&f.recv, (size_t)box.plane * 5)) return LBM_ERR_NOMEM;
        }
        InitParams<T> ip{};
        ip.fa = d_fa, ip.fb = d_fb, ip.aa = aa ? 1 : 0, ip.qstride = qstride, ip.label = d_label;
        ip.rho = d_rho, ip.ux = d_ux, ip.uy = d_uy, ip.uz = d_uz;
        ip.box = box, ip.case_rule = d.case_rule, ip.u_max = (T)d.u_max;
        for (int i = 0; i < LBM_MAX_BC; i++) ip.bc[i] = bc[i];
        ip.plane_in = d_plane_in, ip.plane_out = d_plane_out, ip.fluid_label = fluid_label;
        CK(launch_init<T>(ip, st));
        launches++;
        CK(cudaStreamSynchronize(st));
        d_cur = d_fa, d_nxt = d_fb;
        steps = 0;
        have_init = true, have_moments = false, in_step = false;
        unlink_initialized();
        return 0;
    }

    long long count_plane(int zl) {
        long long c = 0;
        if (launch_count_stored(d_label + (long long)zl * box.plane, box.plane, box.px, box.nx, store_all(), d_cnt + 4, st) !=
            cudaSuccess)
            return -1;
        launches++;
        cudaMemcpyAsync(&c, d_cnt + 4, sizeof c, cudaMemcpyDeviceToHost, st);
        cudaStreamSynchronize(st);
        return c;
    }

    // populations / moments / node words in the reference's compact order, run-segment records
    int initialize_sparse() {
        sparse = true;
        if (!d_plane_in) {
            if (!have_planes) h_in.assign((size_t)d.nx * d.nz, 0.f), h_out = h_in;
            int r = upload_planes();
            if (r) return r;
        }
        const bool aa = d.storage == LBM_STORE_SPARSE_AA;
        const int nzl = box.z1 - box.z0, nown = own_z1 - own_z0;
        const int zl_first = own_z0 - box.z0, zl_last = own_z1 - 1 - box.z0;
        long long ns = stored_box;            // entries of the storage's arrays
        const int32_t *numidx = d_index;      // cell -> id of the storage's numbering (+ num_first)
        long long num_first = sp_first;
        std::vector<long long> pfirst((size_t)nzl + 1);  // first local id of every plane of the state box
        if (aa) {
            // own numbering: fluid nodes and single-cell x gaps, z,y,x order (k_span_flags)
            if (!d_sid && dalloc(&d_sid, (size_t)box.cells())) return LBM_ERR_NOMEM;
            int32_t *keep = nullptr;
            long long *d_pf = nullptr;
            CK(cudaMalloc((void **)&keep, (size_t)box.cells() * sizeof(int32_t)));
            cudaError_t ce = cudaMalloc((void **)&d_pf, (size_t)nzl * sizeof(long long));
            if (ce == cudaSuccess) ce = launch_span_flags(d_label, box, fluid_label, keep, st);
            if (ce == cudaSuccess)
                ce = launch_compact(keep, d_sid, box.cells(), box.px, box.nx, 0, 0, d_scratch, scratch_ints, d_cnt + 7, box.plane, d_pf, st);
            if (ce == cudaSuccess) ce = cudaMemcpyAsync(pfirst.data(), d_pf, (size_t)nzl * sizeof(long long), cudaMemcpyDeviceToHost, st);
            if (ce == cudaSuccess) ce = cudaMemcpyAsync(&ns, d_cnt + 7, sizeof ns, cudaMemcpyDeviceToHost, st);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
            cudaFree(keep), cudaFree(d_pf);
            CK(ce);
            launches += 4;
            pfirst[(size_t)nzl] = ns;
            numidx = d_sid, num_first = 0;
        } else {
            for (int z = 0; z <= nzl; z++) pfirst[(size_t)z] = plane_first[(size_t)z] - sp_first;
        }
        sid_plane_first = pfirst;
        if (!d_cart) {
            if (dalloc(&d_cart, (size_t)ns) || dalloc(&d_nodec, (size_t)ns) || dalloc(&d_wallc, (size_t)ns) ||
                dalloc(&d_labelc, (size_t)ns))
                return LBM_ERR_NOMEM;
        }
        if (aa) {  // gap cells are not fluid: they must read as "skip" whatever the cell's own node word says
            CK(cudaMemsetAsync(d_nodec, 0xff, (size_t)ns * sizeof(uint32_t), st));
        }
        CK(launch_compact_maps(numidx, d_node, d_wall, d_label, box.cells(), num_first, d_cart, d_nodec, d_wallc, d_labelc, st));
        launches++;
        // id ranges of the halo planes and of the outermost owned planes (a plane is one contiguous range)
        auto plane_n = [&](int zl) { return pfirst[(size_t)zl + 1] - pfirst[(size_t)zl]; };
        halo_id0[0] = 0, halo_n[0] = lo_halo ? plane_n(0) : 0;
        face_id0[0] = pfirst[(size_t)zl_first], face_n[0] = lo_halo ? plane_n(zl_first) : 0;
        halo_n[1] = hi_halo ? plane_n(nzl - 1) : 0, halo_id0[1] = ns - halo_n[1];
        face_n[1] = hi_halo ? plane_n(zl_last) : 0, face_id0[1] = pfirst[(size_t)zl_last];
        // segments: aligned 32-id chunks of the owned planes' id range
        own_id0 = pfirst[(size_t)zl_first], own_id1 = pfirst[(size_t)zl_last + 1];
        const long long nchunks = (own_id1 - (own_id0 & ~31LL) + 31) / 32 + 1;
        if (!d_chunk_cnt && (dalloc(&d_chunk_cnt, (size_t)nchunks) || dalloc(&d_chunk_off, (size_t)nchunks) ||
                             dalloc(&d_plane_seg, (size_t)nown + 1)))
            return LBM_ERR_NOMEM;
        auto build = [&](int32_t *rec, long long *plane_seg) {
            return aa ? launch_build_segments_rows(d_nodec, d_cart, d_sid, d_label, fluid_label, box, zl_first, own_id0, own_id1,
                                                   d_chunk_cnt, d_chunk_off, d_cnt + 5, rec, plane_seg, st)
                      : launch_build_segments(d_nodec, d_cart, d_index, box, zl_first, own_id0, own_id1, sp_first, d_chunk_cnt,
                                              d_chunk_off, d_cnt + 5, rec, plane_seg, st);
        };
        CK(build(nullptr, nullptr));
        launches += 2;
        CK(cudaMemcpyAsync(&nseg, d_cnt + 5, sizeof nseg, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (own_id1 <= own_id0) nseg = 0;
        dfree(&d_rec);
        if (dalloc(&d_rec, (size_t)std::max<long long>(nseg, 1) * SEG_REC)) return LBM_ERR_NOMEM;
        CK(cudaMemsetAsync(d_rec, 0, (size_t)std::max<long long>(nseg, 1) * SEG_REC * sizeof(int32_t), st));
        CK(cudaMemsetAsync(d_plane_seg, 0x7f, ((size_t)nown + 1) * sizeof(long long), st));  // "no record yet"
        CK(build(d_rec, d_plane_seg));
        launches++;
        {
            // first record of every owned plane (records are in plane order); planes without fluid take the next one's
            seg_plane_start.assign((size_t)nown + 1, nseg);
            CK(cudaMemcpyAsync(seg_plane_start.data(), d_plane_seg, (size_t)nown * sizeof(long long), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            seg_plane_start[(size_t)nown] = nseg;
            for (int z = nown - 1; z >= 0; z--)
                if (seg_plane_start[(size_t)z] > nseg) seg_plane_start[(size_t)z] = seg_plane_start[(size_t)z + 1];
        }
        if (aa) {
            if (!d_cmeta && dalloc(&d_cmeta, (size_t)(ns / 32 + 2))) return LBM_ERR_NOMEM;
            CK(launch_chunk_meta(d_nodec, ns, d_cmeta, st));
            dfree(&d_rec_links);
            if (dalloc(&d_rec_links, (size_t)std::max<long long>(nseg, 1) * 32)) return LBM_ERR_NOMEM;
            CK(launch_rec_links(d_rec, d_nodec, nseg, d_rec_links, st));
            launches += 2;
            // inlet / outlet link lists (two passes: size, fill)
            int *d_tot = (int *)(d_cnt + 7), total = 0;
            CK(cudaMemsetAsync(d_tot, 0, sizeof(int), st));
            CK(launch_bc_links<T>(d_nodec, d_wallc, d_cart, d_label8, box, bc, d_plane_in, d_plane_out, own_id0, own_id1, d_tot, nullptr,
                                  nullptr, st));
            CK(cudaMemcpyAsync(&total, d_tot, sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            dfree(&d_bcslot), dfree(&d_bclinks);
            if (dalloc(&d_bcslot, (size_t)std::max<long long>(ns, 1)) || dalloc(&d_bclinks, (size_t)std::max(total, 1))) return LBM_ERR_NOMEM;
            CK(cudaMemsetAsync(d_tot, 0, sizeof(int), st));
            CK(launch_bc_links<T>(d_nodec, d_wallc, d_cart, d_label8, box, bc, d_plane_in, d_plane_out, own_id0, own_id1, d_tot, d_bcslot,
                                  d_bclinks, st));
            launches += 2;
        }
        qstride = (ns + 64 + 31) & ~31LL;  // every direction's array starts 256-byte aligned
        if (aa && qstride >= (1LL << 31) / 3) FAIL(LBM_ERR_ARG, "slab of %lld nodes is too large for 32-bit element offsets: use more z-slabs", ns);
        if (!d_fa) {
            const size_t fsize = (size_t)qstride * Q + 64;
            if (dalloc(&d_fa, fsize)) return LBM_ERR_NOMEM;
            if (aa) d_fb = d_fa;  // one buffer, streamed in place
            else if (dalloc(&d_fb, fsize)) return LBM_ERR_NOMEM;
            if (dalloc(&d_rho, (size_t)ns) || dalloc(&d_ux, (size_t)ns) || dalloc(&d_uy, (size_t)ns) || dalloc(&d_uz, (size_t)ns))
                return LBM_ERR_NOMEM;
            for (int sd = 0; sd < 2; sd++) {
                const size_t nb = (size_t)std::max(face_n[sd], halo_n[sd]) * 5;
                if (dalloc(&face[sd].send, nb) || dalloc(&face[sd].recv, nb)) return LBM_ERR_NOMEM;
            }
        }
        InitParams<T> ip{};
        ip.fa = d_fa, ip.fb = d_fb, ip.aa = aa ? 1 : 0, ip.qstride = qstride, ip.label = d_label;
        ip.rho = d_rho, ip.ux = d_ux, ip.uy = d_uy, ip.uz = d_uz;
        ip.box = box, ip.case_rule = d.case_rule, ip.u_max = (T)d.u_max;
        for (int i = 0; i < LBM_MAX_BC; i++) ip.bc[i] = bc[i];
        ip.plane_in = d_plane_in, ip.plane_out = d_plane_out, ip.fluid_label = fluid_label;
        CK(launch_init_sparse<T>(ip, d_cart, ns, st));
        launches++;
        CK(cudaStreamSynchronize(st));
        d_cur = d_fa, d_nxt = d_fb;
        steps = 0;
        have_init = true, have_moments = false, in_step = false;
        unlink_initialized();
        return 0;
    }

    // dense cavities: >= 90 % of the launched cells are fluid -> pull before classifying
    bool speculative_pull() const {
        static const char *const force = getenv("LBM_SPECULATIVE");  // tuning knob, read once
        return force ? atoi(force) != 0 : (nfluid * 10 >= (int64_t)(own_z1 - own_z0) * box.plane * 9);
    }
    // f(std::bool_constant<STRICT>) for this handle's arithmetic: the step entry points are instantiated per arithmetic
    template <typename F>
    cudaError_t with_math(F f) const {
        if (d.math == LBM_MATH_STRICT) return f(std::true_type{});
        return f(std::false_type{});
    }
    // the run loops load the step kernels they are about to launch before they start their clock (lazy module
    // loading would otherwise put 5 - 10 ms per kernel variant into the loop: step_launch.cuh preload_step_kernels)
    int preload_kernels(bool resid) {
        CK(cudaSetDevice(d.device));
        CK(with_math([&](auto S) { return preload_step_kernels<T, S>(d.storage, collision, speculative_pull(), resid, use_persist()); }));
        return 0;
    }

    StepParams<T> make_params(long long c0, long long c1, double *acc) {
        StepParams<T> p{};
        p.src = d_cur, p.dst = d_nxt, p.qstride = qstride;
        p.node = d_node, p.wall = d_wall, p.seg = d_seg, p.label8 = d_label8;
        p.rho = d_rho, p.ux = d_ux, p.uy = d_uy, p.uz = d_uz;
        p.resid = acc;
        p.box = box, p.c_begin = c0, p.c_end = c1;
        p.pdl = opt_pdl && !lo_halo && !hi_halo && in_place();  // single domain only: slab launches alternate with flag kernels
        p.fluid_label = fluid_label;
        p.tau = (T)d.tau;
        p.inv_tau = T(1.0) / p.tau;
        p.om1 = T(1.0) - T(1.0) / p.tau;
        p.collision = collision;
        if (collision == LBM_COLL_TRT) {
            const double om_m = 1.0 / (0.5 + trt_magic / (d.tau - 0.5));  // Lambda = (1/om+ - 1/2)(1/om- - 1/2)
            p.om_m = (T)om_m, p.om1_m = (T)(1.0 - om_m);
        }
        double sc = 1.0;
        if (d.pulse_amp != 0.0) sc = 1.0 + d.pulse_amp * std::sin(2.0 * M_PI * (double)steps / d.pulse_period);
        p.pulse_scale = (T)sc;
        for (int i = 0; i < LBM_MAX_BC; i++) p.bc[i] = bc[i];
        p.plane_in = d_plane_in, p.plane_out = d_plane_out;
        p.parity = (int)(steps & 1);
        p.case_rule = d.case_rule;
        p.u_init = (T)d.u_max;
#ifdef LBM_SELFCHECK
        if (chk_prepare() == 0) {
            p.chk_lo[0] = d_fa, p.chk_hi[0] = d_fa + chk_elems, p.chk_lo[1] = d_fb, p.chk_hi[1] = d_fb + chk_elems;
            p.chk_shadow[0] = d_chk_shadow[0], p.chk_shadow[1] = d_fb == d_fa ? d_chk_shadow[0] : d_chk_shadow[1];
            p.chk_count = d_chk_count, p.chk_launch = ++chk_launch_id;
        }
#endif
        p.speculative = speculative_pull();
        return p;
    }
    // the parameters of a launch over the cells [c0, c1) of the state box; a sparse storage adds its records and id
    // ranges, the dense ones use .base only.  face_sides bit 0: the range is the lowest owned plane, bit 1: the highest
    SparseParams<T> launch_params(long long c0, long long c1, double *acc, int face_sides) {
        SparseParams<T> sp{};
        sp.base = make_params(c0, c1, acc);
        for (int sd = 0; sd < 2; sd++)
            if (face_sides & (1 << sd)) link_params(sp.base, sd, c0);
        if (!sparse) return sp;
        static const int spw_env = getenv("LBM_SPW") ? atoi(getenv("LBM_SPW")) : 0;  // tuning knob
        sp.spw = spw_env > 0 ? spw_env : 1;  // measured: 1 is fastest (profiles/r01_notes.md)
        sp.rec = d_rec, sp.nodec = d_nodec, sp.wallc = d_wallc;
        sp.cartc = d_cart, sp.cmeta = d_cmeta, sp.rec_links = d_rec_links, sp.bcslot = d_bcslot, sp.bclinks = d_bclinks;
        const long long zA = c0 / box.plane - (own_z0 - box.z0), zB = c1 / box.plane - (own_z0 - box.z0);
        sp.seg_begin = seg_plane_start[(size_t)zA], sp.seg_end = seg_plane_start[(size_t)zB];
        sp.id_begin = sid_plane_first[(size_t)(c0 / box.plane)], sp.id_end = sid_plane_first[(size_t)(c1 / box.plane)];
        sp.halo_lo_n = (int)halo_n[0], sp.halo_hi0 = (int)halo_id0[1];
        return sp;
    }
    int launch_range(long long c0, long long c1, bool moments, bool resid, double *acc, int face_sides = 0) {
        if (c1 <= c0) return 0;
        const SparseParams<T> sp = launch_params(c0, c1, acc, face_sides);
        // a sparse kernel walks records (ids on even steps of the in-place storage): planes without fluid have none
        const bool walks_ids = d.storage == LBM_STORE_SPARSE_AA && sp.base.parity == 0;
        if (sparse && (walks_ids ? sp.id_end <= sp.id_begin : sp.seg_end <= sp.seg_begin)) return 0;
        CK(with_math([&](auto S) { return launch_step<T, S>(sp, d.storage, moments, resid, st); }));
        launches++;
        return 0;
    }
    long long plane_c(int z_global) const { return (long long)(z_global - box.z0) * box.plane; }

    // ---- persistent multi-step launches for grids that live in L2 (step_sparse_aa.cuh, k_sparse_aa_persist)
    T *d_pulse = nullptr;
    size_t pulse_cap = 0;
    unsigned *d_barrier = nullptr;
    int sm_count = 0;
    static constexpr int PERSIST_MAX_STEPS = 2048, PERSIST_BAR_WORDS = 64 + 32 * 64;  // = BAR_WORDS of step_sparse_aa.cuh
    int opt_persist = -1;  // lbm_set_option("persistent", 0 / 1); -1: by size
    int collision = LBM_COLL_BGK;  // lbm_set_collision
    double trt_magic = 0.0;        // TRT: Lambda
    int opt_pdl = 1;       // lbm_set_option("overlap_launches", 0 / 1)
    bool use_persist() {
        if (d.storage != LBM_STORE_SPARSE_AA || lo_halo || hi_halo) return false;
#ifdef LBM_SELFCHECK
        return false;  // the shadow tags are per launch: a launch must be one step
#endif
        // opt-in (lbm_set_option("persistent", 1)): measured on the reference's 64^3 configurations one launch per
        // step is as fast or faster (10.1 vs 12.2 us per step, profiles/r02_notes.md section 5) -- the grid barrier
        // costs what the launch gap saves
        return opt_persist > 0;
    }
    // n <= PERSIST_MAX_STEPS steps in one cooperative launch; S_dev: n device slots receiving sum|u| per step, or null
    int persist_steps(int n, bool moments_last, double *S_dev) {
        if (n <= 0) return 0;
        if (!sm_count) {
            cudaDeviceProp prop;
            CK(cudaGetDeviceProperties(&prop, d.device));
            sm_count = prop.multiProcessorCount;
            CK(cudaMalloc((void **)&d_barrier, PERSIST_BAR_WORDS * sizeof(unsigned)));
        }
        const T *pulse_dev = nullptr;
        if (d.pulse_amp != 0.0) {  // the same scale the single launches get, step by step (make_params)
            std::vector<T> tab((size_t)n);
            for (int k = 0; k < n; k++) tab[(size_t)k] = (T)(1.0 + d.pulse_amp * std::sin(2.0 * M_PI * (double)(steps + k) / d.pulse_period));
            if ((size_t)n > pulse_cap) {
                if (d_pulse) cudaFree(d_pulse), d_pulse = nullptr;
                pulse_cap = (size_t)std::max(n, 256);
                CK(cudaMalloc((void **)&d_pulse, pulse_cap * sizeof(T)));
            }
            CK(cudaMemcpyAsync(d_pulse, tab.data(), (size_t)n * sizeof(T), cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));  // `tab` is pageable and goes out of scope
            pulse_dev = d_pulse;
        }
        CK(cudaMemsetAsync(d_barrier, 0, PERSIST_BAR_WORDS * sizeof(unsigned), st));
        const SparseParams<T> sp = launch_params(plane_c(own_z0), plane_c(own_z1), nullptr, 0);
        const int parity0 = (int)(steps & 1);
        CK(with_math([&](auto S) {
            return launch_persist<T, S>(sp, n, parity0, moments_last ? 1 : 0, S_dev, pulse_dev, d_barrier, sm_count, st);
        }));
        launches++;
        steps += n;
        return 0;
    }

    // single-domain step loop
    int step(int n, float *ms) override {
        if (!have_init) FAIL(LBM_ERR_STATE, "step before initialize");
        if (lo_halo || hi_halo) FAIL(LBM_ERR_STATE, "slab handle: use lbm_step_begin / lbm_step_end");
        if (n < 0) FAIL(LBM_ERR_ARG, "negative step count");
        CK(cudaSetDevice(d.device));
        if (ms) CK(cudaEventRecord(ev0, st));
        if (use_persist()) {
            for (int done = 0; done < n; done += PERSIST_MAX_STEPS) {
                const int nb = std::min(PERSIST_MAX_STEPS, n - done);
                int r = persist_steps(nb, done + nb == n, nullptr);
                if (r) return r;
            }
        } else {
            for (int i = 0; i < n; i++) {
                int r = launch_range(plane_c(own_z0), plane_c(own_z1), i == n - 1, false, nullptr);
                if (r) return r;
                std::swap(d_cur, d_nxt);
                steps++;
            }
        }
        if (n > 0) have_moments = true;
        if (ms) {
            CK(cudaEventRecord(ev1, st));
            CK(cudaEventSynchronize(ev1));
            CK(cudaEventElapsedTime(ms, ev0, ev1));
        } else {
            CK(cudaStreamSynchronize(st));
        }
        return 0;
    }

    // one step with an optional velsum slot; used by run_converge and the slab protocol
    double *step_acc = nullptr;
    bool step_nosync = false;
    static constexpr unsigned long long SYNC_TIMEOUT_NS = 20ull * 1000000000ull;
    int step_begin(int flags) override { return step_begin_ex(flags, nullptr); }
    int step_begin_ex(int flags, double *acc) {
        if (!have_init) FAIL(LBM_ERR_STATE, "step before initialize");
        if (in_step) FAIL(LBM_ERR_STATE, "lbm_step_begin called twice");
        CK(cudaSetDevice(d.device));
        const bool mom = flags & LBM_STEP_MOMENTS, res = flags & LBM_STEP_VELSUM;
        if (in_place() && ((lo_halo && !fused(0)) || (hi_halo && !fused(1))))
            FAIL(LBM_ERR_STATE, "in-place storage exchanges slab faces by peer stores only: call lbm_p2p_attach first");
        step_flags = flags;
        step_acc = acc ? acc : d_acc, step_nosync = acc != nullptr;
        if (res && !acc) CK(cudaMemsetAsync(d_acc, 0, sizeof(double), st));
        // a slab may touch the planes it shares with a neighbour only after that neighbour finished the
        // face launches of the previous step (flags across processes, events inside one)
        const unsigned long long done = (unsigned long long)(steps - sync_base);
        if (face[0].peer_sync || face[1].peer_sync) {
            CK(launch_slab_wait(d_sync, face[0].peer_sync ? done : 0ull, face[1].peer_sync ? done : 0ull, SYNC_TIMEOUT_NS, st));
            launches++;
        }
        for (const Face &f : face)
            if (f.inproc_nb) CK(cudaStreamWaitEvent(st, f.inproc_nb->face_event((int)((steps + 1) & 1)), 0));
        int r;
        const int zt = own_z1 - 1, zb = own_z0;
        long long i0 = plane_c(own_z0), i1 = plane_c(own_z1);
        if (hi_halo) {
            const int sides = 2 | ((lo_halo && zb == zt) ? 1 : 0);
            if ((r = launch_range(plane_c(zt), plane_c(zt + 1), mom, res, step_acc, sides))) return r;
            if ((r = after_face_launch(1))) return r;
            i1 = plane_c(zt);
        }
        if (lo_halo && !(hi_halo && zb == zt)) {
            if ((r = launch_range(plane_c(zb), plane_c(zb + 1), mom, res, step_acc, 1))) return r;
            i0 = plane_c(zb + 1);
        }
        if (lo_halo && (r = after_face_launch(0))) return r;
        if (face[0].peer_sync || face[1].peer_sync) {
            CK(launch_slab_signal(face[0].peer_sync, face[1].peer_sync, done + 1ull, st));
            launches++;
        }
        if (face[0].inproc_nb || face[1].inproc_nb) CK(cudaEventRecord(ev_face[steps & 1], st));
        pend_i0 = i0, pend_i1 = i1, interior_pending = true;
        in_step = true;
        return 0;
    }
    // the interior planes: queued AFTER the caller posted the halo transfers, so that the
    // transfer (on the transport's stream) overlaps this launch
    int step_interior() override {
        if (!in_step) FAIL(LBM_ERR_STATE, "lbm_step_interior without lbm_step_begin");
        if (!interior_pending) return 0;
        CK(cudaSetDevice(d.device));
        interior_pending = false;
        return launch_range(pend_i0, pend_i1, step_flags & LBM_STEP_MOMENTS, step_flags & LBM_STEP_VELSUM, step_acc);
    }
    int step_end() override {
        if (!in_step) FAIL(LBM_ERR_STATE, "lbm_step_end without lbm_step_begin");
        CK(cudaSetDevice(d.device));
        if (interior_pending) {
            int r = step_interior();
            if (r) return r;
        }
        for (int sd = 0; sd < 2; sd++) {
            int r = has_nb(sd) ? at_step_end(sd) : 0;
            if (r) return r;
        }
        if ((step_flags & LBM_STEP_VELSUM) && !step_nosync) {
            CK(cudaMemcpyAsync(&last_S, d_acc, sizeof(double), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        if (step_flags & LBM_STEP_MOMENTS) have_moments = true;
        std::swap(d_cur, d_nxt);
        steps++;
        in_step = false;
        return 0;
    }
    bool in_place() const { return d.storage == LBM_STORE_DENSE_AA || d.storage == LBM_STORE_SPARSE_AA; }
    int enqueue_step(int flags, double *acc) override {
        int r = step_begin_ex(flags, acc);
        if (r) return r;
        if ((r = step_interior())) return r;
        return step_end();
    }
    double *acc_slot(int k) override { return d_acc + 2 + (k % (ACC_SLOTS - 2)); }
    int zero_acc(int first, int n) override {
        CK(cudaSetDevice(d.device));
        CK(cudaMemsetAsync(d_acc + 2 + first, 0, sizeof(double) * (size_t)n, st));
        return 0;
    }
    int fetch_acc(int first, int n, double *out) override {
        CK(cudaSetDevice(d.device));
        CK(cudaMemcpyAsync(out, d_acc + 2 + first, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return check_sync_error();
    }
    int check_sync_error() {
        if (!face[0].peer_sync && !face[1].peer_sync) return 0;
        unsigned long long flag = 0;
        CK(cudaMemcpyAsync(&flag, d_sync + 2, sizeof flag, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (flag) FAIL(LBM_ERR_CUDA, "a neighbouring slab did not report its step within %.0f s", SYNC_TIMEOUT_NS * 1e-9);
        return 0;
    }
    cudaEvent_t face_event(int k) override { return ev_face[k & 1]; }
    void set_inproc_neighbour(int side, SolverBase *nb) override { face[side].inproc_nb = nb; }
    // lbm_slab_step: n steps of this slab, neighbours ordered on the device, nothing but launches on the host
    int slab_steps(int n, int flags_last, double *S_out, float *ms) override {
        if (!have_init) FAIL(LBM_ERR_STATE, "step before initialize");
        if (n < 0) FAIL(LBM_ERR_ARG, "negative step count");
        for (int sd = 0; sd < 2; sd++) {
            if (!has_nb(sd)) continue;
            if (!fused(sd)) FAIL(LBM_ERR_STATE, "lbm_slab_step needs the fused peer-store exchange: lbm_p2p_attach side %d first", sd);
            if (!face[sd].peer_sync && !face[sd].inproc_nb)
                FAIL(LBM_ERR_STATE, "lbm_slab_step: no ordering with the neighbour on side %d (lbm_sync_attach)", sd);
        }
        CK(cudaSetDevice(d.device));
        if (ms) CK(cudaEventRecord(ev0, st));
        const int nslots = ACC_SLOTS - 2;
        for (int i0 = 0; i0 < n; i0 += nslots) {
            const int nb = std::min(nslots, n - i0);
            if (S_out) CK(cudaMemsetAsync(d_acc + 2, 0, sizeof(double) * (size_t)nb, st));
            for (int j = 0; j < nb; j++) {
                const int flags = (i0 + j == n - 1 ? (flags_last & LBM_STEP_MOMENTS) : 0) | (S_out ? LBM_STEP_VELSUM : 0);
                int r = enqueue_step(flags, S_out ? d_acc + 2 + j : d_acc + 1);
                if (r) return r;
            }
            if (S_out) {
                CK(cudaMemcpyAsync(S_out + i0, d_acc + 2, sizeof(double) * (size_t)nb, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
            }
        }
        if (ms) {
            CK(cudaEventRecord(ev1, st));
            CK(cudaEventSynchronize(ev1));
            CK(cudaEventElapsedTime(ms, ev0, ev1));
        } else {
            CK(cudaStreamSynchronize(st));
        }
        return check_sync_error();
    }
    // ------------------------------------------------------------ slab faces (Face, Link)
    bool has_nb(int sd) const { return sd == 0 ? lo_halo : hi_halo; }
    // the step kernels store the leaving populations of this face themselves: no pack, no unpack
    bool fused(int sd) const { return face[sd].kind != Link::PACKED; }
    // the StepParams peer fields of a launch that covers side sd's face plane (c0: the launch's first cell)
    void link_params(StepParams<T> &p, int sd, long long c0) const {
        const Face &f = face[sd];
        T *peer = nullptr;
        long long qs = 0, pc0 = 0, own = 0;
        switch (f.kind) {
        case Link::PACKED:
            return;
        case Link::PEER_BUFFERS:
            peer = f.peer_buf[d_nxt == d_fa ? 0 : 1], qs = f.peer_qs, pc0 = f.peer_c0, own = f.peer_own;
            p.face_c0 = sparse ? face_id0[sd] : c0;
            break;
        case Link::MAILBOX:
        case Link::STAGED_MAILBOX:
            // the neighbour's mailbox: part A (its halo replica) on even steps, part B (its owned face plane) on odd ones
            peer = f.peer_mail + (p.parity ? 5 * mail_ms : 0), qs = mail_ms, pc0 = own = mail_G;
            p.peer_mail = 1, p.face_c0 = c0;
            p.mail[sd] = f.mail, p.mail_ms = mail_ms, p.mail_G = mail_G;
            break;
        }
        if (sd == 1) p.peer_up = peer, p.peer_up_qs = qs, p.peer_up_c0 = pc0, p.peer_up_own = own;
        else p.peer_dn = peer, p.peer_dn_qs = qs, p.peer_dn_c0 = pc0, p.peer_dn_own = own;
    }
    // queued right after the launch of side sd's face plane: the pack of a PACKED face
    int after_face_launch(int sd) {
        const Face &f = face[sd];
        if (f.kind != Link::PACKED) return 0;
        if (sparse) CK(launch_halo_pack_sparse<T>(d_nxt, qstride, face_id0[sd], face_n[sd], sd, f.send, face_n[sd], st));
        else CK(launch_halo_pack<T>(d_nxt, qstride, box, (sd == 0 ? own_z0 : own_z1 - 1) - box.z0, sd, f.send, st));
        launches++;
        return 0;
    }
    // queued by lbm_step_end, after the caller's transfers into the receive buffers
    int at_step_end(int sd) {
        const Face &f = face[sd];
        if (f.kind == Link::PACKED) {
            if (sparse) CK(launch_halo_unpack_sparse<T>(d_nxt, qstride, d_labelc, fluid_label, halo_id0[sd], halo_n[sd], sd, f.recv, halo_n[sd], st));
            else CK(launch_halo_unpack<T>(d_nxt, qstride, d_label8, fluid_label, box, sd == 0 ? 0 : box.z1 - box.z0 - 1, sd, f.recv, st));
            launches++;
        } else if (f.kind == Link::STAGED_MAILBOX) {
            // take over what the neighbour stored (the transfer into the receive part is complete on this stream),
            // and give the part that was sent its "nothing written" pattern back
            const size_t off = (steps & 1) ? (size_t)mail_ms * 5 : 0;
            CK(launch_mail_merge<T>(f.mail + off, f.stage_in + off, mail_ms * 5, st));
            CK(cudaMemsetAsync(f.stage_out + off, 0xFF, (size_t)mail_ms * 5 * sizeof(T), st));
            launches++;
        }
        return 0;
    }
    // Every attach and detach of the C ABI, between two steps; the caller fills in the new kind's peer pointers.
    // Both faces of a slab hold the same fused kind: a one-plane slab's launch covers both with one StepParams, whose
    // peer_mail flag tells the kernel how to address both peers.  So changing the kind needs a detach first.
    int relink(int sd, Link kind) {
        static const char *const names[] = {"packed", "peer-buffer", "mailbox", "staged-mailbox"};
        for (int s = 0; s < 2; s++)
            if (kind != Link::PACKED && face[s].kind != Link::PACKED && face[s].kind != kind)
                FAIL(LBM_ERR_STATE, "side %d holds a %s link: detach it before attaching a %s link to side %d", s,
                     names[(int)face[s].kind], names[(int)kind], sd);
        CK(cudaSetDevice(d.device));
        CK(cudaStreamSynchronize(st));
        int r = mail_place(sd, kind == Link::MAILBOX || kind == Link::STAGED_MAILBOX);
        if (r) return r;
        CK(cudaStreamSynchronize(st));
        Face &f = face[sd];
        f.kind = kind;
        f.peer_buf[0] = f.peer_buf[1] = f.peer_mail = nullptr;
        f.peer_qs = f.peer_c0 = f.peer_own = 0;
        return 0;
    }
    // Where the current values of side sd's mailbox slots (the entering directions) are: in its mailbox (live) or in
    // the population buffer.  The population buffer is made whole before it is read as a whole (checkpoints,
    // lbm_debug_get_populations) and handed back to the mailboxes afterwards: mail_place_all(false / true).
    int mail_place(int sd, bool live) {
        Face &f = face[sd];
        if (f.mail_live == live) return 0;
        const long long halo_c0 = sd == 0 ? 0 : (long long)(box.z1 - box.z0 - 1) * box.plane;
        const long long face_c0 = sd == 0 ? plane_c(own_z0) : plane_c(own_z1 - 1);
        CK(launch_mail_copy<T>(d_fa, qstride, f.mail, mail_ms, mail_G, face_c0, halo_c0, box.plane, sd, live ? 0 : 1, st));
        launches++;
        f.mail_live = live;
        return 0;
    }
    int mail_place_all(bool live) {
        for (int sd = 0; sd < 2; sd++) {
            int r = mail_place(sd, live && face[sd].mailbox());
            if (r) return r;
        }
        return 0;
    }
    // initialize: the population buffer was just written whole, so mailbox links end without moving slots back;
    // mapped peer buffers stay, and the ordering with the neighbours is wired again (lbm_sync_attach / the group)
    void unlink_initialized() {
        for (Face &f : face) {
            if (f.mailbox()) f.kind = Link::PACKED, f.peer_mail = nullptr;
            f.mail_live = false, f.peer_sync = nullptr, f.inproc_nb = nullptr;
        }
        sync_base = 0;
    }
    // geo_pre of an initialised sparse slab: the pack buffers and the neighbours' buffers fit the old geometry
    void unlink_geometry_sized() {
        for (Face &f : face) {
            dfree(&f.send), dfree(&f.recv);
            if (f.kind == Link::PEER_BUFFERS) f.kind = Link::PACKED, f.peer_buf[0] = f.peer_buf[1] = nullptr;
        }
    }
    int mail_export(int side, lbm_ipc_handle *h, void **ptr, int64_t *boff, int64_t *ms, int64_t *guard) override {
        if (side < 0 || side > 1) FAIL(LBM_ERR_ARG, "side must be 0 or 1");
        if (!have_init) FAIL(LBM_ERR_STATE, "mail_export before initialize");
        if (d.storage != LBM_STORE_DENSE_AA) FAIL(LBM_ERR_STATE, "mailboxes exist for the dense in-place storage only");
        if (!has_nb(side)) FAIL(LBM_ERR_ARG, "no neighbour on side %d", side);
        CK(cudaSetDevice(d.device));
        mail_G = box.px + 32, mail_ms = box.plane + 2 * mail_G;
        T *&mail = face[side].mail;
        if (!mail) {
            if (dalloc(&mail, (size_t)mail_ms * 10)) return LBM_ERR_NOMEM;
            CK(cudaMemsetAsync(mail, 0, (size_t)mail_ms * 10 * sizeof(T), st));
        }
        if (h) {
            cudaIpcMemHandle_t ih;
            CK(cudaIpcGetMemHandle(&ih, mail));
            memset(h, 0, sizeof(lbm_ipc_handle));
            memcpy(h, &ih, sizeof ih);
        }
        if (ptr) *ptr = mail;
        if (boff) {
            int r = alloc_offset(mail, boff);
            if (r) return r;
        }
        if (ms) *ms = mail_ms;
        if (guard) *guard = mail_G;
        return 0;
    }
    // peer_mail: the NEIGHBOUR's mailbox of the side facing this slab, as mapped here (null detaches a mailbox link of
    // either kind).  From now on this slab reads the entering populations of that face from its own mailbox and
    // stores the leaving ones into the neighbour's: both sides of a face must switch together, between two steps.
    int mail_attach(int side, void *pm) override {
        if (side < 0 || side > 1) FAIL(LBM_ERR_ARG, "side must be 0 or 1");
        if (!have_init || (pm && !face[side].mail)) FAIL(LBM_ERR_STATE, "lbm_mail_attach before lbm_mail_export of that side");
        if (!pm && !face[side].mailbox()) return 0;
        int r = relink(side, pm ? Link::MAILBOX : Link::PACKED);
        if (r) return r;
        face[side].peer_mail = (T *)pm;
        return 0;
    }
    // pa / pb: the neighbour's two population buffers as mapped here (both null detach a peer-buffer link)
    int p2p_attach(int side, void *pa, void *pb, int64_t pqs, int64_t pc0, int64_t pown) override {
        if (side < 0 || side > 1) FAIL(LBM_ERR_ARG, "side must be 0 or 1");
        if (!have_init) FAIL(LBM_ERR_STATE, "p2p_attach before initialize");
        if (!has_nb(side)) FAIL(LBM_ERR_ARG, "no neighbour on side %d", side);
        if ((pa == nullptr) != (pb == nullptr)) FAIL(LBM_ERR_ARG, "both peer buffers or none");
        Face &f = face[side];
        if (!pa && f.kind != Link::PEER_BUFFERS) return 0;
        int r = relink(side, pa ? Link::PEER_BUFFERS : Link::PACKED);
        if (r) return r;
        f.peer_buf[0] = (T *)pa, f.peer_buf[1] = (T *)pb, f.peer_qs = pqs, f.peer_c0 = pc0, f.peer_own = pown;
        return 0;
    }
    // Mailbox transport WITHOUT peer mapping: the leaving populations of this side go into a local staging buffer
    // (lbm_halo_buffers: send part), the caller moves it to the neighbour's receive part by whatever means it has
    // (NCCL send/recv: slab.py; a device copy: tests) between lbm_step_begin and lbm_step_end, and lbm_step_end
    // merges what arrived into the mailbox (k_mail_merge).  The step kernel is the one of the mapped transport.
    int mail_stage(int side) override {
        int r = mail_export(side, nullptr, nullptr, nullptr, nullptr, nullptr);
        if (r) return r;
        Face &f = face[side];
        const size_t n = (size_t)mail_ms * 10;
        if (!f.stage_out && (dalloc(&f.stage_out, n) || dalloc(&f.stage_in, n))) return LBM_ERR_NOMEM;
        CK(cudaMemsetAsync(f.stage_out, 0xFF, n * sizeof(T), st));
        CK(cudaMemsetAsync(f.stage_in, 0xFF, n * sizeof(T), st));
        if ((r = relink(side, Link::STAGED_MAILBOX))) return r;
        f.peer_mail = f.stage_out;
        return 0;
    }
    int sync_export(lbm_ipc_handle *h, void **ptr, int64_t *boff) override {
        CK(cudaSetDevice(d.device));
        if (h) {
            cudaIpcMemHandle_t ih;
            CK(cudaIpcGetMemHandle(&ih, d_sync));
            memset(h, 0, sizeof(lbm_ipc_handle));
            memcpy(h, &ih, sizeof ih);
        }
        if (ptr) *ptr = d_sync;
        if (boff) {
            int r = alloc_offset(d_sync, boff);
            if (r) return r;
        }
        return 0;
    }
    // peer_sync: the NEIGHBOUR's sync block as mapped into this process (null detaches).  Collective in
    // effect: both sides reset their counters here, so attach on all slabs before any of them steps.
    int sync_attach(int side, void *peer) override {
        if (side < 0 || side > 1) FAIL(LBM_ERR_ARG, "side must be 0 or 1");
        if (!has_nb(side)) FAIL(LBM_ERR_ARG, "no neighbour on side %d", side);
        CK(cudaSetDevice(d.device));
        CK(cudaStreamSynchronize(st));
        // this slab is the HIGH neighbour of the slab below it and the LOW neighbour of the one above
        face[side].peer_sync = peer ? (unsigned long long *)peer + (side == 0 ? 1 : 0) : nullptr;
        CK(cudaMemsetAsync(d_sync + side, 0, sizeof(unsigned long long), st));
        CK(cudaMemsetAsync(d_sync + 2, 0, sizeof(unsigned long long), st));
        CK(cudaStreamSynchronize(st));
        sync_base = steps;
        return 0;
    }
    // byte offset of a device pointer inside the cudaMalloc block its IPC handle stands for
    int alloc_offset(const void *p, int64_t *off) {
        typedef int (*range_fn)(unsigned long long *, size_t *, unsigned long long);
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qr;
        CK(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &qr));
        unsigned long long base = 0;
        size_t sz = 0;
        if (!fn || ((range_fn)fn)(&base, &sz, (unsigned long long)(uintptr_t)p) != 0) FAIL(LBM_ERR_CUDA, "cuMemGetAddressRange failed");
        *off = (int64_t)((unsigned long long)(uintptr_t)p - base);
        return 0;
    }
    int last_velsum(double *v) override {
        *v = last_S;
        return 0;
    }
    // ------------------------------------------------------------ checkpoint / restart
    struct CkptHeader {
        char magic[8];
        int32_t version, case_rule, nx, ny, nz, z_begin, z_end, precision, storage, reserved;
        int64_t steps, qstride, elems;
        uint64_t case_hash;  // labels of the state box, tau, BC table, pulse parameters
    };
    // FNV-1a over the parameters a continued run depends on, seeded with an order-independent
    // device-side hash of the label field
    int case_hash(uint64_t *out) {
        CK(cudaMemsetAsync(d_cnt + 6, 0, sizeof(long long), st));
        CK(launch_label_hash(d_label, box.cells(), (unsigned long long *)(d_cnt + 6), st));
        launches++;
        unsigned long long hv = 0;
        CK(cudaMemcpyAsync(&hv, d_cnt + 6, sizeof hv, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        uint64_t h = 1469598103934665603ull ^ hv;
        auto mix = [&h](const void *p, size_t n) {
            const unsigned char *b = (const unsigned char *)p;
            for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 1099511628211ull;
        };
        mix(&d.tau, sizeof d.tau), mix(&d.u_max, sizeof d.u_max);
        mix(&d.pulse_amp, sizeof d.pulse_amp), mix(&d.pulse_period, sizeof d.pulse_period);
        for (int i = 0; i < LBM_MAX_BC; i++) {
            const BcEntry &e = bc[i];
            const int v[6] = {e.kind, e.naxis, e.nsign, e.vaxis, e.source, e.pulsatile};
            mix(v, sizeof v), mix(&e.value, sizeof e.value), mix(&e.init_value, sizeof e.init_value);
        }
        mix(&nfluid, sizeof nfluid), mix(&stored_box, sizeof stored_box);
        if (have_planes) mix(h_in.data(), h_in.size() * sizeof(float)), mix(h_out.data(), h_out.size() * sizeof(float));
        if (collision != LBM_COLL_BGK) mix(&collision, sizeof collision), mix(&trt_magic, sizeof trt_magic);  // BGK keeps its old hash
        *out = h;
        return 0;
    }
    // The population buffer travels through a bounded pinned staging buffer (two halves, the copy of one
    // overlapping the file I/O of the other): at 512^3 fp64 the buffer is 20 GB, which must not be mirrored
    // in pageable host memory.
    int checkpoint(const char *path, bool save) override {
        if (!have_init) FAIL(LBM_ERR_STATE, "checkpoint before initialize");
        if (in_step) FAIL(LBM_ERR_STATE, "checkpoint inside lbm_step_begin / lbm_step_end");
        if (!path) FAIL(LBM_ERR_ARG, "null path");
        CK(cudaSetDevice(d.device));
        {
            int r = mail_place_all(false);  // the population buffer is whole again; done() hands the slots back
            if (r) return r;
        }
        CK(cudaStreamSynchronize(st));
        // the buffer the next step pulls from holds the whole state (the other one is overwritten),
        // except for the never-rewritten static slots, which initialize() put into both
        const size_t elems = (size_t)qstride * Q;
        CkptHeader hd{};
        memcpy(hd.magic, "LBMB200", 8);
        hd.version = 2, hd.case_rule = d.case_rule, hd.nx = d.nx, hd.ny = d.ny, hd.nz = d.nz;
        hd.z_begin = d.z_begin, hd.z_end = d.z_end, hd.precision = d.precision, hd.storage = d.storage;
        hd.steps = steps, hd.qstride = qstride, hd.elems = (int64_t)elems;
        int r = case_hash(&hd.case_hash);
        if (r) return r;
        const size_t half = (size_t)(32u << 20) / sizeof(T);  // elements per staging half (32 MiB)
        T *stage = nullptr;
        CK(cudaMallocHost((void **)&stage, 2 * half * sizeof(T)));
        cudaEvent_t evh[2] = {nullptr, nullptr};
        FILE *f = nullptr;
        int rc = 0;
        auto done = [&](int code, const std::string &msg) {
            if (have_init) {  // hand the mailbox slots back whatever happened to the file
                const int r2 = mail_place_all(true);
                if (!code) code = r2;
            }
            if (f) fclose(f);
            for (auto &e : evh)
                if (e) cudaEventDestroy(e);
            cudaFreeHost(stage);
            if (code) err = msg;
            return code;
        };
        for (auto &e : evh)
            if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return done(LBM_ERR_CUDA, "cudaEventCreate failed");
        const size_t nchunk = (elems + half - 1) / half;
        auto chunk_len = [&](size_t k) { return std::min(half, elems - k * half); };
        if (save) {
            f = fopen(path, "wb");
            if (!f) return done(LBM_ERR_IO, fmt("cannot write '%s'", path));
            if (fwrite(&hd, sizeof hd, 1, f) != 1) return done(LBM_ERR_IO, fmt("short write to '%s'", path));
            for (size_t k = 0; k <= nchunk; k++) {
                if (k < nchunk) {  // start the copy of chunk k ...
                    if (cudaMemcpyAsync(stage + (k & 1) * half, d_cur + k * half, chunk_len(k) * sizeof(T), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                        cudaEventRecord(evh[k & 1], st) != cudaSuccess)
                        return done(LBM_ERR_CUDA, "checkpoint: device-to-host copy failed");
                }
                if (k > 0) {  // ... while chunk k-1 goes to the file
                    if (cudaEventSynchronize(evh[(k - 1) & 1]) != cudaSuccess) return done(LBM_ERR_CUDA, "checkpoint: copy failed");
                    const size_t n = chunk_len(k - 1);
                    if (fwrite(stage + ((k - 1) & 1) * half, sizeof(T), n, f) != n) return done(LBM_ERR_IO, fmt("short write to '%s'", path));
                }
            }
            rc = fclose(f), f = nullptr;
            return done(rc ? LBM_ERR_IO : 0, fmt("short write to '%s'", path));
        }
        f = fopen(path, "rb");
        if (!f) return done(LBM_ERR_IO, fmt("cannot open '%s'", path));
        CkptHeader in{};
        if (fread(&in, sizeof in, 1, f) != 1) return done(LBM_ERR_IO, fmt("short read from '%s'", path));
        if (memcmp(in.magic, hd.magic, 8) || in.version != hd.version || in.case_rule != hd.case_rule || in.nx != hd.nx ||
            in.ny != hd.ny || in.nz != hd.nz || in.z_begin != hd.z_begin || in.z_end != hd.z_end ||
            in.precision != hd.precision || in.storage != hd.storage || in.qstride != hd.qstride || in.elems != hd.elems)
            return done(LBM_ERR_ARG, fmt("checkpoint '%s' was written for a different case / slab / precision / storage", path));
        if (in.case_hash != hd.case_hash)
            return done(LBM_ERR_ARG, fmt("checkpoint '%s' was written for a different geometry, tau or boundary table", path));
        // two-buffer storage alternates with the step parity; keep "current" consistent with it
        T *target = (d_fb != d_fa && (in.steps & 1)) ? d_fb : d_fa;
        for (size_t k = 0; k < nchunk; k++) {
            if (k >= 2 && cudaEventSynchronize(evh[k & 1]) != cudaSuccess) return done(LBM_ERR_CUDA, "checkpoint: copy failed");
            const size_t n = chunk_len(k);
            if (fread(stage + (k & 1) * half, sizeof(T), n, f) != n) {
                cudaStreamSynchronize(st);
                have_init = false;  // the state is partly overwritten
                return done(LBM_ERR_IO, fmt("short read from '%s' (the handle must be re-initialised)", path));
            }
            if (cudaMemcpyAsync(target + k * half, stage + (k & 1) * half, n * sizeof(T), cudaMemcpyHostToDevice, st) != cudaSuccess ||
                cudaEventRecord(evh[k & 1], st) != cudaSuccess)
                return done(LBM_ERR_CUDA, "checkpoint: host-to-device copy failed");
        }
        if (cudaStreamSynchronize(st) != cudaSuccess) return done(LBM_ERR_CUDA, "checkpoint: copy failed");
        steps = in.steps;
        d_cur = target;
        d_nxt = d_cur == d_fa ? d_fb : d_fa;
        have_moments = false;
        return done(0, "");
    }

    int p2p_export(lbm_ipc_handle *h2, void **ptrs, int64_t *boff, int64_t *qs, int64_t *halo_c0, int64_t *face_c0) override {
        if (!have_init) FAIL(LBM_ERR_STATE, "p2p_export before initialize");
        CK(cudaSetDevice(d.device));
        static_assert(sizeof(cudaIpcMemHandle_t) <= sizeof(lbm_ipc_handle), "handle size");
        T *bufs[2] = {d_fa, d_fb};
        for (int k = 0; k < 2; k++) {
            if (h2) {
                cudaIpcMemHandle_t ih;
                CK(cudaIpcGetMemHandle(&ih, bufs[k]));
                memset(&h2[k], 0, sizeof(lbm_ipc_handle));
                memcpy(&h2[k], &ih, sizeof ih);
            }
            if (ptrs) ptrs[k] = bufs[k];
            if (boff) {
                int r = alloc_offset(bufs[k], &boff[k]);
                if (r) return r;
            }
        }
        if (qs) *qs = qstride;
        if (halo_c0) {
            halo_c0[0] = sparse ? halo_id0[0] : 0;
            halo_c0[1] = sparse ? halo_id0[1] : (long long)(box.z1 - box.z0 - 1) * box.plane;
        }
        if (face_c0) {
            face_c0[0] = sparse ? face_id0[0] : plane_c(own_z0);
            face_c0[1] = sparse ? face_id0[1] : plane_c(own_z1 - 1);
        }
        return 0;
    }
    int halo_buffers(int side, void **send, void **recv, size_t *send_bytes, size_t *recv_bytes) override {
        if (side < 0 || side > 1) FAIL(LBM_ERR_ARG, "side must be 0 or 1");
        if (!have_init) FAIL(LBM_ERR_STATE, "halo_buffers before initialize");
        const bool present = has_nb(side);
        const Face &f = face[side];
        if (present && f.kind == Link::STAGED_MAILBOX) {  // the part of the current step's parity: A on even, B on odd steps
            const size_t off = (steps & 1) ? (size_t)mail_ms * 5 : 0, bytes = (size_t)mail_ms * 5 * sizeof(T);
            if (send) *send = f.stage_out + off;
            if (recv) *recv = f.stage_in + off;
            if (send_bytes) *send_bytes = bytes;
            if (recv_bytes) *recv_bytes = bytes;
            return 0;
        }
        if (send) *send = present ? f.send : nullptr;
        if (recv) *recv = present ? f.recv : nullptr;
        const size_t dense_b = (size_t)box.plane * 5 * sizeof(T);
        if (send_bytes) *send_bytes = !present ? 0 : (sparse ? (size_t)face_n[side] * 5 * sizeof(T) : dense_b);
        if (recv_bytes) *recv_bytes = !present ? 0 : (sparse ? (size_t)halo_n[side] * 5 * sizeof(T) : dense_b);
        return 0;
    }

    int residual(int kind, double *v) override {
        if (!have_moments) FAIL(LBM_ERR_STATE, "no moments yet: run lbm_step first");
        CK(cudaSetDevice(d.device));
        if (sparse)
            CK(launch_reduce_fields_sparse<T>(d_ux, d_uy, d_uz, d_labelc, d_cart, box, own_id0, own_id1, kind, fluid_label,
                                              d.case_rule, d_acc + 1, st));
        else
            CK(launch_reduce_fields<T>(d_ux, d_uy, d_uz, d_label, box, own_z0, own_z1, kind, fluid_label, d.case_rule,
                                       d_acc + 1, st));
        launches++;
        CK(cudaMemcpyAsync(v, d_acc + 1, sizeof(double), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return 0;
    }

    // ------------------------------------------------------------ readback
    int get_box_i32(const int32_t *dev, int32_t *out) {
        CK(cudaSetDevice(d.device));
        const int nzo = own_z1 - own_z0;
        CK(cudaMemcpy2DAsync(out, (size_t)d.nx * sizeof(int32_t), dev + plane_c(own_z0), (size_t)box.px * sizeof(int32_t),
                             (size_t)d.nx * sizeof(int32_t), (size_t)d.ny * nzo, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return 0;
    }
    int get_geo(int32_t *g) override {
        if (!have_geo) FAIL(LBM_ERR_STATE, "get_geo before geo_pre");
        return get_box_i32(d_label, g);
    }
    int get_index(int32_t *g) override {
        if (!have_index) FAIL(LBM_ERR_STATE, "get_index before index_transform");
        return get_box_i32(d_index, g);
    }
    int get_fields(void *rho, void *ux, void *uy, void *uz, int64_t *first, int64_t *count) override {
        if (!have_init) FAIL(LBM_ERR_STATE, "get_fields before initialize");
        CK(cudaSetDevice(d.device));
        const size_t n = (size_t)stored_own;
        if (sparse && d.storage != LBM_STORE_SPARSE_AA) {  // the device arrays already are in compact order
            const T *srcs[4] = {d_rho, d_ux, d_uy, d_uz};
            void *dsts[4] = {rho, ux, uy, uz};
            for (int k = 0; k < 4; k++)
                if (dsts[k]) CK(cudaMemcpyAsync(dsts[k], srcs[k] + n_lo_stored, n * sizeof(T), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (first) *first = compact_first;
            if (count) *count = stored_own;
            return 0;
        }
        if (store_all() && !sparse) {
            // every node of the box is stored (ldc.cu:54): the moment arrays ARE in compact order, row by row
            const T *srcs[4] = {d_rho, d_ux, d_uy, d_uz};
            void *dsts[4] = {rho, ux, uy, uz};
            const size_t rows = (size_t)d.ny * (size_t)(own_z1 - own_z0);
            for (int k = 0; k < 4; k++)
                if (dsts[k])
                    CK(cudaMemcpy2DAsync(dsts[k], (size_t)d.nx * sizeof(T), srcs[k] + plane_c(own_z0), (size_t)box.px * sizeof(T),
                                         (size_t)d.nx * sizeof(T), rows, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (first) *first = compact_first;
            if (count) *count = stored_own;
            return 0;
        }
        // dense storage: gather into compact order one group of planes at a time through two small
        // persistent staging buffers -- the gather of group g+1 runs while group g crosses PCIe on a
        // second stream
        const long long group_cells = 4LL << 20;  // small groups: the staging buffers are allocated on first use, inside the caller's timed region
        const int gplanes = (int)std::max<long long>(1, group_cells / box.plane);
        long long maxn = 1;
        for (int z = own_z0; z < own_z1; z += gplanes) {
            const int zb = std::min(own_z1, z + gplanes);
            maxn = std::max(maxn, plane_first[(size_t)(zb - box.z0)] - plane_first[(size_t)(z - box.z0)]);
        }
        if ((size_t)maxn * 8 > stage_elems) {
            if (d_stage) cudaFree(d_stage), d_stage = nullptr;
            stage_elems = (size_t)maxn * 8;
            CK(cudaMalloc((void **)&d_stage, stage_elems * sizeof(T)));
        }
        if (!st_copy) {
            CK(cudaStreamCreateWithFlags(&st_copy, cudaStreamNonBlocking));
            for (int k = 0; k < 2; k++) {
                CK(cudaEventCreateWithFlags(&ev_gathered[k], cudaEventDisableTiming));
                CK(cudaEventCreateWithFlags(&ev_copied[k], cudaEventDisableTiming));
            }
        }
        char *outs[4] = {(char *)rho, (char *)ux, (char *)uy, (char *)uz};
        int g = 0;
        for (int z = own_z0; z < own_z1; z += gplanes) {
            const int zb = std::min(own_z1, z + gplanes);
            const long long f0 = plane_first[(size_t)(z - box.z0)], cnt = plane_first[(size_t)(zb - box.z0)] - f0;
            if (cnt <= 0) continue;
            T *buf = d_stage + (size_t)(g & 1) * 4 * maxn;
            if (g >= 2) CK(cudaStreamWaitEvent(st, ev_copied[g & 1], 0));  // the copy out of this half is done
            CK(launch_gather_fields<T>(d_rho, d_ux, d_uy, d_uz, d_label, d_index, sparse ? d_sid : nullptr, box, z, zb, fluid_label,
                                       f0, buf, buf + maxn, buf + 2 * maxn, buf + 3 * maxn, st));
            launches++;
            CK(cudaEventRecord(ev_gathered[g & 1], st));
            CK(cudaStreamWaitEvent(st_copy, ev_gathered[g & 1], 0));
            for (int k = 0; k < 4; k++)
                if (outs[k])
                    CK(cudaMemcpyAsync(outs[k] + (size_t)(f0 - compact_first) * sizeof(T), buf + (size_t)k * maxn,
                                       (size_t)cnt * sizeof(T), cudaMemcpyDeviceToHost, st_copy));
            CK(cudaEventRecord(ev_copied[g & 1], st_copy));
            g++;
        }
        CK(cudaStreamSynchronize(st_copy));
        CK(cudaStreamSynchronize(st));
        if (first) *first = compact_first;
        if (count) *count = stored_own;
        return 0;
    }
    int get_populations(void *f) override {
        if (!have_init) FAIL(LBM_ERR_STATE, "get_populations before initialize");
        CK(cudaSetDevice(d.device));
        {
            int r = mail_place_all(false);
            if (r) return r;
        }
        struct Refill {
            Solver *s;
            ~Refill() { s->mail_place_all(true); }
        } refill{this};
        const size_t n = (size_t)stored_own;
        if (d.storage == LBM_STORE_SPARSE_AA) {
            T *tmp = nullptr;
            CK(cudaMalloc((void **)&tmp, std::max<size_t>(n, 1) * Q * sizeof(T)));
            cudaError_t e = cudaMemsetAsync(tmp, 0, std::max<size_t>(n, 1) * Q * sizeof(T), st);
            if (e == cudaSuccess)
                e = launch_gather_pops_sparse_aa<T>(d_cur, qstride, d_label, d_index, d_sid, box, own_z0, own_z1, fluid_label,
                                                    compact_first, (long long)n, (int)(steps & 1), tmp, st);
            launches++;
            if (e == cudaSuccess) e = cudaMemcpyAsync(f, tmp, n * Q * sizeof(T), cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            cudaFree(tmp);
            CK(e);
            return 0;
        }
        if (sparse) {  // d_scr itself, q-major
            for (int q = 0; q < Q; q++)
                CK(cudaMemcpyAsync((T *)f + (size_t)q * n, d_cur + (size_t)q * qstride + n_lo_stored, n * sizeof(T),
                                   cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            return 0;
        }
        T *tmp = nullptr;
        CK(cudaMalloc((void **)&tmp, std::max<size_t>(n, 1) * Q * sizeof(T)));
        const int layout = d.storage == LBM_STORE_DENSE_AA ? ((steps & 1) ? 2 : 1) : 0;
        cudaError_t e = launch_gather_pops<T>(d_cur, qstride, d_index, box, own_z0, own_z1, compact_first, (long long)n,
                                              layout, tmp, st);
        launches++;
        if (e == cudaSuccess) e = cudaMemcpyAsync(f, tmp, n * Q * sizeof(T), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        cudaFree(tmp);
        CK(e);
        return 0;
    }

    // ------------------------------------------------------------ writers
    // Host copies in Cartesian order for the writers (single-domain handles).
    std::vector<int32_t> w_index;
    std::vector<T> w_rho, w_ux, w_uy, w_uz;
    int fetch_for_output() {
        if ((lo_halo || hi_halo) && out_format == LBM_OUT_ASCII_VTK)
            FAIL(LBM_ERR_STATE, "the ASCII writer needs a single-domain handle (slabs: LBM_OUT_BINARY_VTK)");
        if (w_index.empty()) {
            w_index.resize((size_t)d.nx * d.ny * (size_t)(own_z1 - own_z0));
            int r = get_index(w_index.data());
            if (r) return r;
        }
        const size_t n = (size_t)stored_own;
        w_rho.resize(n), w_ux.resize(n), w_uy.resize(n), w_uz.resize(n);
        return get_fields(w_rho.data(), w_ux.data(), w_uy.data(), w_uz.data(), nullptr, nullptr);
    }

    // outputSave: ldc.cu:582-610, pos:903-938, bif:1095-1156, cor:948-1011.
    // Same loops, same `ofstream <<` formatting of float values.
    // Legacy-VTK BINARY: same header, points, fields and unit factors as the ASCII writer, values as
    // big-endian float32.  A slab handle writes its own planes (ORIGIN shifted in z).
    int output_save_binary(int t) {
        const int NX = d.nx, NY = d.ny, NZ = d.nz;
        const float CH = (float)d.CH, C_U = (float)d.C_U, C_rho = (float)d.C_rho;
        const float C_pre = C_rho * C_U * C_U;
        const bool ldc = d.case_rule == LBM_CASE_LDC;
        const int x0 = ldc ? 2 : 1, x1 = ldc ? NX - 2 : NX - 1, y0 = 2, y1 = NY - 2, zt0 = ldc ? 2 : 1,
                  zt1 = ldc ? NZ - 2 : NZ - 1;
        const int z0 = std::max(zt0, own_z0), z1 = std::min(zt1, own_z1);
        const bool piece = lo_halo || hi_halo;
        std::string path = std::string(d.out_dir) + "/" + d.out_name + "_" + std::to_string(t) + "_bin";
        if (piece) path += ".z" + std::to_string(own_z0);
        path += ".vtk";
        const long long npts = z1 > z0 ? (long long)(x1 - x0) * (y1 - y0) * (z1 - z0) : 0;
        std::ofstream ofs(path, std::ios::binary);
        if (!ofs) FAIL(LBM_ERR_IO, "cannot write '%s'", path.c_str());
        ofs << "# vtk DataFile Version 2.0\n";
        ofs << "<-- LBM flow with UIV acceleration, http://www.bg.ic.ac.uk/research/m.tang/ulis/ -->\n";
        ofs << "BINARY\nDATASET STRUCTURED_POINTS\n";
        ofs << "DIMENSIONS " << (x1 - x0) << ' ' << (y1 - y0) << ' ' << std::max(0, z1 - z0) << "\n";
        ofs << "SPACING " << CH << ' ' << CH << ' ' << CH << "\n";
        const float oz = (float)(std::max(z0, zt0) - zt0) * CH;
        if (ldc) ofs << "ORIGIN " << std::round(NX / 2 - 1) * CH << ' ' << std::round(NY / 2 - 1) * CH << ' ' << oz << "\n";
        else ofs << "ORIGIN " << std::round(NX / 2) * CH << ' ' << std::round(NY / 2) * CH << ' ' << oz << "\n";
        ofs << "POINT_DATA  " << npts << "\n";
        if (npts == 0) return 0;
        auto be = [](float v) {
            uint32_t u;
            memcpy(&u, &v, 4);
            return __builtin_bswap32(u);
        };
        // w_index holds the owned planes only; field arrays start at this handle's first compact id
        auto idx_of = [&](int x, int y, int z) {
            const int g = w_index[(size_t)x + (size_t)NX * ((size_t)y + (size_t)NY * (size_t)(z - own_z0))];
            return g < 0 ? (long long)-1 : (long long)g - compact_first;
        };
        const int nzp = z1 - z0;
        const int nthr = std::max(1, std::min({(int)std::thread::hardware_concurrency(), 16, nzp}));
        std::vector<uint32_t> buf;
        // kind 0: density, 1: pressure, 2: velocity
        auto section = [&](int kind) {
            const int ncomp = kind == 2 ? 3 : 1;
            buf.resize((size_t)npts * ncomp);
            auto work = [&](int th) {
                const int za = z0 + (int)((long long)nzp * th / nthr), zb = z0 + (int)((long long)nzp * (th + 1) / nthr);
                size_t o = (size_t)(za - z0) * (y1 - y0) * (x1 - x0) * ncomp;
                for (int z = za; z < zb; z++)
                    for (int y = y0; y < y1; y++)
                        for (int x = x0; x < x1; x++) {
                            const long long i = idx_of(x, y, z);
                            if (kind == 0) buf[o++] = be(i >= 0 ? (float)w_rho[i] * C_rho : 0.0f);
                            else if (kind == 1) buf[o++] = be(i >= 0 ? (float)((float)w_rho[i] * C_pre / 3.0) : 0.0f);
                            else {
                                buf[o++] = be(i >= 0 ? (float)w_ux[i] * C_U : 0.0f);
                                buf[o++] = be(i >= 0 ? (float)w_uy[i] * C_U : 0.0f);
                                buf[o++] = be(i >= 0 ? (float)w_uz[i] * C_U : 0.0f);
                            }
                        }
            };
            std::vector<std::thread> pool;
            for (int th = 1; th < nthr; th++) pool.emplace_back(work, th);
            work(0);
            for (auto &thd : pool) thd.join();
            ofs.write((const char *)buf.data(), (std::streamsize)(buf.size() * sizeof(uint32_t)));
        };
        if (d.case_rule == LBM_CASE_GEO_OPENINGS) {
            ofs << "SCALARS DENSITY float\nLOOKUP_TABLE default\n";
            section(0);
            ofs << "\nSCALARS PRESSURE float\nLOOKUP_TABLE default\n";
            section(1);
            ofs << "\n";
        }
        ofs << "VECTORS VELOCITY float\n";
        section(2);
        ofs << "\n";
        ofs.close();
        if (!ofs) FAIL(LBM_ERR_IO, "short write to '%s'", path.c_str());
        return 0;
    }

    int output_save(int t) override {
        int r = join_writer();
        if (r) return r;
        if ((r = fetch_for_output())) return r;
        if (out_format == LBM_OUT_BINARY_VTK) return output_save_binary(t);
        return write_ascii(t);
    }
    // ONE byte-compatible ASCII file for a run sharded over several slabs: the group gathers the
    // index table (Cartesian, whole box) and the fields (compact order, NLATTICE entries) and any slab
    // handle formats them -- same code as the single-domain writer
    int write_global(int t, const int32_t *index_global, const void *rho, const void *ux, const void *uy, const void *uz,
                     int64_t nlattice) override {
        int jr = join_writer();
        if (jr) return jr;
        std::vector<int32_t> si;
        std::vector<T> sr, sx, sy, sz;
        si.swap(w_index), sr.swap(w_rho), sx.swap(w_ux), sy.swap(w_uy), sz.swap(w_uz);
        w_index.assign(index_global, index_global + (size_t)d.nx * d.ny * d.nz);
        const size_t n = (size_t)nlattice;
        w_rho.assign((const T *)rho, (const T *)rho + n), w_ux.assign((const T *)ux, (const T *)ux + n);
        w_uy.assign((const T *)uy, (const T *)uy + n), w_uz.assign((const T *)uz, (const T *)uz + n);
        int r = write_ascii(t);
        si.swap(w_index), sr.swap(w_rho), sx.swap(w_ux), sy.swap(w_uy), sz.swap(w_uz);
        return r;
    }
    int write_ascii(int t) { return write_ascii_from(t, w_rho.data(), w_ux.data(), w_uy.data(), w_uz.data(), err); }
    // formats and writes one file from host arrays; touches no other member that a running time loop changes
    int write_ascii_from(int t, const T *prho, const T *pux, const T *puy, const T *puz, std::string &errout, int max_threads = 16) {
        const int NX = d.nx, NY = d.ny, NZ = d.nz;
        const float CH = (float)d.CH, C_U = (float)d.C_U, C_rho = (float)d.C_rho;
        const float C_pre = C_rho * C_U * C_U;
        std::string path = std::string(d.out_dir) + "/" + d.out_name + "_" + std::to_string(t) + ".vtk";
        std::ofstream ofs(path);
        if (!ofs) {
            errout = fmt("cannot write '%s'", path.c_str());
            return LBM_ERR_IO;
        }
        using std::endl;
        ofs << "# vtk DataFile Version 2.0" << endl;
        ofs << "<-- LBM flow with UIV acceleration, http://www.bg.ic.ac.uk/research/m.tang/ulis/ -->" << endl;
        ofs << "ASCII" << endl;
        ofs << "DATASET STRUCTURED_POINTS" << endl;
        const bool ldc = d.case_rule == LBM_CASE_LDC;
        const int x0 = ldc ? 2 : 1, x1 = ldc ? NX - 2 : NX - 1, y0 = 2, y1 = NY - 2, z0 = ldc ? 2 : 1,
                  z1 = ldc ? NZ - 2 : NZ - 1;
        ofs << "DIMENSIONS " << (x1 - x0) << ' ' << (y1 - y0) << ' ' << (z1 - z0) << endl;
        ofs << "SPACING " << CH << ' ' << CH << ' ' << CH << endl;
        if (ldc) ofs << "ORIGIN " << std::round(NX / 2 - 1) * CH << ' ' << std::round(NY / 2 - 1) * CH << ' ' << .0 << endl;
        else ofs << "ORIGIN " << std::round(NX / 2) * CH << ' ' << std::round(NY / 2) * CH << ' ' << .0 << endl;
        ofs << "POINT_DATA  " << (x1 - x0) * (y1 - y0) * (z1 - z0) << endl;
        auto idx_of = [&](int x, int y, int z) { return w_index[(size_t)x + (size_t)NX * ((size_t)y + (size_t)NY * z)]; };
        // The bodies: the same characters `ofs << value << ' '` produces (default ostream float format =
        // %g with 6 significant digits = std::to_chars general/6), formatted into one buffer -- at 512^3
        // the reference's ASCII writer would otherwise dominate the run (SURVEY 8f.2).
        // z-planes are formatted by several host threads into their own buffers and written in order.
        const int nzp = z1 - z0;
        const int nthr = std::max(1, std::min({(int)std::thread::hardware_concurrency(), max_threads, nzp}));
        // kind 0: density, 1: pressure, 2: velocity.  A value takes at most 15 characters with its blank
        // ("-1.23457e-308 "), so a part's buffer is sized for the worst case and never grows; only the pages
        // that are written become resident.
        struct Part {
            std::unique_ptr<char[]> data;
            size_t len = 0;
        };
        auto format_planes = [&](int kind, std::vector<Part> &parts) {
            parts.clear();
            parts.resize((size_t)nthr);
            auto work = [&](int t) {
                const int za = z0 + (int)((long long)nzp * t / nthr), zb = z0 + (int)((long long)nzp * (t + 1) / nthr);
                Part &part = parts[(size_t)t];
                part.data.reset(new char[(size_t)(x1 - x0) * (y1 - y0) * (zb - za) * (kind == 2 ? 45 : 15) + VTK_MAX_CHARS]);
                char *p = part.data.get();
                for (int z = za; z < zb; z++)
                    for (int y = y0; y < y1; y++)
                        for (int x = x0; x < x1; x++) {
                            const int i = idx_of(x, y, z);
                            if (kind == 0) p = vtk_write(p, i >= 0 ? (float)prho[i] * C_rho : 0.0f);
                            else if (kind == 1) {
                                if (i >= 0) p = vtk_write(p, (float)prho[i] * C_pre / 3.0);  // double, as in cor.cu:983
                                else p = vtk_write(p, 0.0f);
                            } else if (i >= 0) {
                                p = vtk_write(p, (float)pux[i] * C_U), p = vtk_write(p, (float)puy[i] * C_U);
                                p = vtk_write(p, (float)puz[i] * C_U);
                            } else {
                                std::memcpy(p, "0 0 0 ", 6), p += 6;
                            }
                        }
                part.len = (size_t)(p - part.data.get());
            };
            std::vector<std::thread> pool;
            for (int t = 1; t < nthr; t++) pool.emplace_back(work, t);
            work(0);
            for (auto &th : pool) th.join();
        };
        std::vector<Part> parts;
        auto flush = [&]() {
            for (auto &s : parts) ofs.write(s.data.get(), (std::streamsize)s.len);
        };
        if (d.case_rule == LBM_CASE_GEO_OPENINGS) {
            ofs << "SCALARS DENSITY float\nLOOKUP_TABLE default\n";
            format_planes(0, parts), flush();
            ofs << "\nSCALARS PRESSURE float\nLOOKUP_TABLE default\n";
            format_planes(1, parts), flush();
            ofs << "\n";
        }
        ofs << "VECTORS VELOCITY float\n";
        format_planes(2, parts), flush();
        ofs.close();
        return 0;
    }

    // ---- periodic dumps of the run loops are formatted and written by helper threads while the GPU keeps
    // stepping: at 64^3 one ASCII dump takes as long as ~1000 steps, and the reference dumps every 500, so up
    // to MAX_DUMPS_IN_FLIGHT snapshots are being written at any time
    struct DumpJob {
        std::thread th;
        std::vector<T> rho, ux, uy, uz;  // the snapshot the helper thread reads
        int rc = 0;
        std::string err;
    };
    std::deque<std::unique_ptr<DumpJob>> dump_jobs;
    static constexpr size_t MAX_DUMPS_IN_FLIGHT = 4;
    static constexpr int ASYNC_DUMP_THREADS = 3;  // per dump: 12 formatting threads at most, the launching thread keeps a core
    int join_oldest_dump() {
        auto &j = dump_jobs.front();
        if (j->th.joinable()) j->th.join();
        const int rc = j->rc;
        if (rc) err = j->err;
        dump_jobs.pop_front();
        return rc;
    }
    int join_writer() {
        int rc = 0;
        while (!dump_jobs.empty()) {
            const int r = join_oldest_dump();
            if (r && !rc) rc = r;
        }
        return rc;
    }
    // w_rho .. w_uz were just fetched (fetch_for_output)
    int save_fetched_async(int t) {
        if (out_format != LBM_OUT_ASCII_VTK) return output_save_binary(t);
        while (dump_jobs.size() >= MAX_DUMPS_IN_FLIGHT) {
            int r = join_oldest_dump();
            if (r) return r;
        }
        dump_jobs.emplace_back(new DumpJob());
        DumpJob *j = dump_jobs.back().get();
        j->rho = w_rho, j->ux = w_ux, j->uy = w_uy, j->uz = w_uz;
        j->th = std::thread([this, j, t]() { j->rc = write_ascii_from(t, j->rho.data(), j->ux.data(), j->uy.data(), j->uz.data(), j->err, ASYNC_DUMP_THREADS); });
        return 0;
    }
    // write_once(): cor.cu:1033-1051 -- "x,y,z,ux,uy,uz" of every inlet / outlet node (labels 2,3,5,6,7), %f.
    // (coronary.cu defines it but never calls it; the reference's h_u* of those nodes are whatever the
    // device buffers held, here they are 0: nothing ever writes moments of non-fluid nodes.)
    int write_bc_csv(const char *path) override {
        if (lo_halo || hi_halo) FAIL(LBM_ERR_STATE, "lbm_write_bc_csv needs a single-domain handle");
        int r = fetch_for_output();
        if (r) return r;
        std::vector<int32_t> geo((size_t)d.nx * d.ny * d.nz);
        if ((r = get_geo(geo.data()))) return r;
        FILE *f = fopen(path, "w+");
        if (!f) FAIL(LBM_ERR_IO, "cannot write '%s'", path);
        for (int z = 0; z < d.nz; z++)
            for (int y = 0; y < d.ny; y++)
                for (int x = 0; x < d.nx; x++) {
                    const size_t c = (size_t)x + (size_t)d.nx * ((size_t)y + (size_t)d.ny * z);
                    const int type = geo[c], i = w_index[c];
                    if ((type == 2 || type == 3 || type == 5 || type == 6 || type == 7) && i >= 0)
                        fprintf(f, "%d,%d,%d,%f,%f,%f\n", x, y, z, (double)(float)w_ux[i], (double)(float)w_uy[i], (double)(float)w_uz[i]);
                }
        fclose(f);
        return 0;
    }

    // calc_res(): bif.cu:1158-1175 on the host copy, long double like the reference
    long double host_u2sum() {
        long double sum = 0.0L;
        if (w_index.empty() || w_ux.empty()) return sum;
        std::vector<int32_t> geo((size_t)d.nx * d.ny * d.nz);
        if (get_geo(geo.data())) return sum;
        for (int z = 1; z < d.nz - 1; z++)
            for (int y = 2; y < d.ny - 2; y++)
                for (int x = 1; x < d.nx - 1; x++) {
                    size_t c = (size_t)x + (size_t)d.nx * ((size_t)y + (size_t)d.ny * z);
                    int g = geo[c];
                    bool ok = d.case_rule == LBM_CASE_GEO_OPENINGS ? g == 4 : g >= 4;
                    if (!ok) continue;
                    int i = w_index[c];
                    float v = (float)w_ux[i] * (float)w_ux[i] + (float)w_uy[i] * (float)w_uy[i] +
                              (float)w_uz[i] * (float)w_uz[i];
                    sum += v;
                }
        return sum;
    }

    // bif.cu:1246-1274 / cor.cu:1100-1132
    int run_fixed(int repeat, int time_save, int write_files) override {
        if (!have_init) FAIL(LBM_ERR_STATE, "run before initialize");
        if (time_save <= 0) FAIL(LBM_ERR_ARG, "time_save must be positive");
        std::ofstream logfile;
        if (write_files) logfile.open(std::string(d.out_dir) + "/CONVERGENCE.log");
        {
            int r = preload_kernels(false);
            if (r) return r;
        }
        auto t0 = std::chrono::steady_clock::now();
        float residual = 0.f;
        int done = 0;  // iterations executed so far (loop index i runs 0..repeat inclusive)
        long double sum1 = 0.0L;
        while (done <= repeat) {
            // next save happens at loop index i with i % time_save == 0
            int i_save = ((done + time_save - 1) / time_save) * time_save;
            int upto = std::min(i_save, repeat);
            int r = step(upto - done + 1, nullptr);
            if (r) return r;
            done = upto + 1;
            if (upto % time_save == 0) {
                sum1 = host_u2sum();  // fields of the previous save (0 at first)
                r = fetch_for_output();
                if (r) return r;
                long double sum2 = host_u2sum();
                residual = (float)(fabsl(sum1 - sum2) / sum2);
                float milli = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
                if (write_files) {
                    logfile << residual << std::endl;
                    std::cout << "ITERATION # " << upto << ", collapse time: " << milli << " ms, residual:" << residual
                              << std::endl;
                    r = save_fetched_async(upto);  // the fields were fetched just above
                    if (r) return r;
                }
            }
        }
        {
            int r = join_writer();
            if (r) return r;
        }
        float milli = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (write_files) {
            std::cout << "TOTAL RUNNING TIME: " << milli << " MILLI SECONDS" << "#LATTICE" << compact_total << std::endl;
            logfile << "TOTAL RUNNING TIME: " << milli << " MILLI SECONDS" << "#LATTICE" << compact_total << " ERROR IS"
                    << residual << std::endl;
        }
        return 0;
    }

    // ldc.cu:653-685 / pos.cu:986-1019: residual every step, cumulative tol_count.
    // Steps run in batches that end on save iterations; S_k of each step lands in
    // its own device slot, so the host applies the reference's stopping rule
    // exactly without a sync per step; batch sizes shrink as tol_count approaches
    // stag_max so that the loop stops on exactly the same k.
    int run_converge(int max_it, double tol_d, int stag_max, int time_save, int write_files, int *its,
                     double *res) override {
        if (!have_init) FAIL(LBM_ERR_STATE, "run before initialize");
        if (lo_halo || hi_halo) FAIL(LBM_ERR_STATE, "run_converge needs a single-domain handle");
        if (time_save <= 0) FAIL(LBM_ERR_ARG, "time_save must be positive");
        CK(cudaSetDevice(d.device));
        std::ofstream logfile;
        if (write_files) logfile.open(std::string(d.out_dir) + "/CONVERGENCE.log");
        {
            int r = preload_kernels(true);
            if (r) return r;
        }
        auto t0 = std::chrono::steady_clock::now();
        const float tol = (float)tol_d;
        float residual = 0.f, sum_current = 0.f;
        int k = 0, tol_count = 0;
        const int max_batch = std::max(1, std::min(ACC_SLOTS - 2, 48));
        std::vector<double> S(ACC_SLOTS);
        static const bool trace = getenv("LBM_TRACE") != nullptr;
        double tr_step = 0, tr_fetch = 0, tr_save = 0;
        auto now = []() { return std::chrono::steady_clock::now(); };
        auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
        while (k <= max_it && tol_count <= stag_max) {
            // the loop cannot end by the tolerance rule in fewer than stag_max + 1 - tol_count more steps
            // (at most one hit per step), so a batch of that many never overshoots the stopping iteration
            int nb = std::min(max_batch, std::max(1, stag_max + 1 - tol_count));
            nb = std::min(nb, max_it - k + 1);
            // the batch covers iterations k .. k+nb-1; a save iteration inside must be the last one
            for (int j = 0; j < nb; j++)
                if ((k + j) % time_save == 0) {
                    nb = j + 1;
                    break;
                }
            const auto tb0 = now();
            CK(cudaMemsetAsync(d_acc + 2, 0, sizeof(double) * nb, st));
            if (use_persist()) {  // the whole batch in one cooperative launch; moments of its last step (a save iteration, if any)
                int r = persist_steps(nb, true, d_acc + 2);
                if (r) return r;
            } else {
                for (int j = 0; j < nb; j++) {  // moments are needed from the last step of a batch only (a save iteration, if any)
                    int r = launch_range(plane_c(own_z0), plane_c(own_z1), j == nb - 1, true, d_acc + 2 + j);
                    if (r) return r;
                    std::swap(d_cur, d_nxt);
                    steps++;
                }
            }
            have_moments = true;
            CK(cudaMemcpyAsync(S.data(), d_acc + 2, sizeof(double) * nb, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            tr_step += secs(tb0, now());
            for (int j = 0; j < nb; j++) {
                float sum_next = (float)S[j];
                residual = std::fabs(sum_next - sum_current) / sum_next;
                if (k % time_save == 0 && write_files) {
                    float milli = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
                    std::cout << "ITERATION # " << k << ", collapse time: " << milli << " ms, residual:" << residual
                              << std::endl;
                    logfile << residual << std::endl;
                    const auto tf0 = now();
                    int r = fetch_for_output();
                    const auto tf1 = now();
                    if (!r) r = save_fetched_async(k);
                    tr_fetch += secs(tf0, tf1), tr_save += secs(tf1, now());
                    if (r) return r;
                }
                k++;
                sum_current = sum_next;
                if (residual <= tol) tol_count++;
                if (!(k <= max_it && tol_count <= stag_max)) break;
            }
        }
        float milli = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (write_files) {
            const auto tj0 = now();
            int r = output_save(k);  // joins the dumps in flight first
            if (trace) fprintf(stderr, "[lbm trace] run_converge: %d iterations, stepping %.1f ms, fetches %.1f ms, handing dumps over %.1f ms, final dump + joins %.1f ms\n", k, tr_step * 1e3, tr_fetch * 1e3, tr_save * 1e3, secs(tj0, now()) * 1e3);
            if (r) return r;
            std::cout << "TOTAL RUNNING TIME: " << milli << " MILLI SECONDS" << "#LATTICE" << compact_total << std::endl;
            std::cout << "Residual is " << residual << std::endl;
            logfile << "TOTAL RUNNING TIME: " << milli << " MILLI SECONDS" << "#LATTICE" << compact_total << " ERROR IS"
                    << residual << std::endl;
        }
        if (its) *its = k;
        if (res) *res = residual;
        return 0;
    }

    int sync() override {
        CK(cudaSetDevice(d.device));
        CK(cudaStreamSynchronize(st));
        return check_sync_error();
    }
    // ---- self-checking build (tools/selfcheck.py)
    unsigned long long *d_chk_shadow[2] = {nullptr, nullptr}, *d_chk_count = nullptr;
    size_t chk_elems = 0;
    unsigned int chk_launch_id = 0;
    int chk_prepare() {
        const size_t elems = sparse ? (size_t)qstride * Q + 64 : (size_t)qstride * Q + (size_t)box.plane + box.px + 64;
        if (d_chk_count && elems == chk_elems) return 0;
        for (auto &p : d_chk_shadow)
            if (p) cudaFree(p), p = nullptr;
        if (!d_chk_count) {
            CK(cudaMalloc((void **)&d_chk_count, 2 * sizeof(unsigned long long)));
            CK(cudaMemset(d_chk_count, 0, 2 * sizeof(unsigned long long)));
        }
        for (int b = 0; b < (d_fb == d_fa ? 1 : 2); b++) {
            CK(cudaMalloc((void **)&d_chk_shadow[b], elems * sizeof(unsigned long long)));
            CK(cudaMemset(d_chk_shadow[b], 0, elems * sizeof(unsigned long long)));
        }
        chk_elems = elems;
        return 0;
    }
    int set_collision(int model, double lambda) override {
        if (in_step) FAIL(LBM_ERR_STATE, "lbm_set_collision inside lbm_step_begin / lbm_step_end");
        const std::string why = collision_refusal(d, model, lambda);
        if (!why.empty()) FAIL(LBM_ERR_ARG, "lbm_set_collision: %s", why.c_str());
        collision = model, trt_magic = model == LBM_COLL_TRT ? lambda : 0.0;
        return 0;
    }
    int set_option(const char *name, double value) override {
        if (!strcmp(name, "persistent")) opt_persist = value < 0 ? -1 : (value != 0.0);
        else if (!strcmp(name, "overlap_launches")) opt_pdl = value != 0.0;
        else FAIL(LBM_ERR_ARG, "unknown option '%s'", name);
        return 0;
    }
    int selfcheck(uint64_t *out2) override {
#ifdef LBM_SELFCHECK
        CK(cudaSetDevice(d.device));
        CK(cudaStreamSynchronize(st));
        out2[0] = out2[1] = 0;
        if (d_chk_count) {
            unsigned long long v[2];
            CK(cudaMemcpy(v, d_chk_count, sizeof v, cudaMemcpyDeviceToHost));
            out2[0] = v[0], out2[1] = v[1];
        }
        out2[2] = chk_launch_id;
        return 0;
#else
        (void)out2;
        FAIL(LBM_ERR_STATE, "not a self-checking build (compile with -DLBM_SELFCHECK, tools/selfcheck.py)");
#endif
    }
    void *stream_ptr() override { return (void *)st; }
};

}  // namespace lbm

// ============================================================================
// C ABI
// ============================================================================
using lbm::SolverBase;
struct lbm_solver_s {
    SolverBase *s;
};

static void set_bc(lbm_case_desc *d, int label, int kind, int naxis, int nsign, int vaxis, int source, double value,
                   double init_value) {
    lbm_bc_desc &b = d->bc[d->n_bc++];
    b.label = label, b.kind = kind, b.normal_axis = naxis, b.normal_sign = nsign, b.vel_axis = vaxis;
    b.source = source, b.pulsatile = 0, b.reserved = 0, b.value = value, b.init_value = init_value;
}
static void set_open(lbm_case_desc *d, int axis, int coord, int lo_a, int hi_a, int lo_b, int hi_b, int reps) {
    lbm_opening_rule &o = d->openings[d->n_openings++];
    o.axis = axis, o.coord = coord, o.lo_a = lo_a, o.hi_a = hi_a, o.lo_b = lo_b, o.hi_b = hi_b, o.reps = reps;
    o.reserved = 0;
}

extern "C" {

int lbm_case_defaults(int32_t rule, lbm_case_desc *d) {
    if (!d) return LBM_ERR_ARG;
    memset(d, 0, sizeof *d);
    d->struct_size = (int32_t)sizeof *d;
    d->case_rule = rule;
    d->precision = LBM_F32;  // the reference's precision (thesis section 4.4)
    d->storage = LBM_STORE_DENSE_AB;
    d->math = LBM_MATH_FAST;
    snprintf(d->geo_path, sizeof d->geo_path, "./geo.txt");
    snprintf(d->bc_path, sizeof d->bc_path, "./bc.txt");
    snprintf(d->out_dir, sizeof d->out_dir, "./out");
    // constants are the reference's float literals, widened
    switch (rule) {
    case LBM_CASE_LDC: {  // ldc.cu:48-55
        d->nx = d->ny = d->nz = 64;
        const float C_U = 2.4705f;
        d->tau = 0.55f, d->C_U = C_U, d->C_rho = 1060.f, d->CH = 0.0000655737f;
        d->u_max = 0.15f / C_U;
        set_bc(d, 2, LBM_BC_V, 1, -1, 2, LBM_SRC_CONST, 0.15f / C_U, 0.15f / C_U);  // lid, ldc.cu:378,391-456
        snprintf(d->out_name, sizeof d->out_name, "lid");
        break;
    }
    case LBM_CASE_POISEUILLE: {  // pos.cu:38-44,590
        d->nx = d->ny = d->nz = 64;
        const float C_U = 1.5441f;
        d->tau = 0.58f, d->C_U = C_U, d->C_rho = 1060.f, d->CH = 0.0000655737f;
        d->u_max = 0.15f / C_U;
        set_bc(d, 2, LBM_BC_V, 1, +1, 1, LBM_SRC_PARABOLA, 0.09714700668f, 0.15f / C_U);
        set_bc(d, 3, LBM_BC_V, 1, -1, 1, LBM_SRC_PARABOLA, 0.09714700668f, 0.15f / C_U);
        snprintf(d->out_name, sizeof d->out_name, "pos");
        break;
    }
    case LBM_CASE_GEO_Y_INOUT: {  // bif.cu:19-20,434
        d->nx = 64, d->ny = 83, d->nz = 32;
        d->tau = 0.55f, d->C_U = 0.24159041f, d->C_rho = 998.2f, d->CH = 0.000248925f;
        set_bc(d, 2, LBM_BC_V, 1, +1, 1, LBM_SRC_PLANE_INLET, 0.0, 0.0);  // bif.cu:950-1021
        set_bc(d, 3, LBM_BC_P, 1, -1, 1, LBM_SRC_CONST, 0.0, 0.0);         // bif.cu:877-948
        snprintf(d->out_name, sizeof d->out_name, "bif");
        break;
    }
    case LBM_CASE_GEO_OPENINGS: {  // cor.cu:19-20,302-306,717,796,871
        d->nx = 291, d->ny = 291, d->nz = 372;
        const float C_U = 2.74909090909091f;
        d->tau = 0.55f, d->C_U = C_U, d->C_rho = 1060.f, d->CH = 6.1111e-05f;
        d->geo_yfast = 1;
        set_bc(d, 2, LBM_BC_VP, 0, +1, 0, LBM_SRC_CONST, (float)(0.1745 / C_U), 0.1745f / C_U);
        set_bc(d, 3, LBM_BC_V, 0, -1, 0, LBM_SRC_CONST, (float)(0.1 / C_U), 0.1f / C_U);
        for (int l = 5; l <= 7; l++) set_bc(d, l, LBM_BC_V, 2, -1, 2, LBM_SRC_CONST, (float)(0.02 / C_U), 0.02f / C_U);
        set_open(d, 0, 3, 1, d->ny - 2, 1, d->nz - 2, 1);      // cor.cu:77-87
        set_open(d, 0, 272, 1, d->ny - 2, 1, d->nz - 2, 2);    // cor.cu:89-101
        set_open(d, 2, 185, 217, 236, 113, 137, 4);            // cor.cu:103-115
        set_open(d, 2, 191, 160, 205, 159, 199, 5);            // cor.cu:117-129
        set_open(d, 2, 204, 1, d->nx - 2, 1, d->ny - 2, 6);    // cor.cu:131-141
        snprintf(d->out_name, sizeof d->out_name, "coronary");
        break;
    }
    default:
        return LBM_ERR_ARG;
    }
    d->z_begin = 0, d->z_end = d->nz;
    return LBM_OK;
}

int lbm_create(const lbm_case_desc *desc, lbm_handle *out) {
    using namespace lbm;
    if (!desc || !out) {
        g_create_error = "null argument";
        return LBM_ERR_ARG;
    }
    *out = nullptr;
    if (desc->struct_size != (int32_t)sizeof(lbm_case_desc)) {
        g_create_error = fmt("lbm_case_desc size mismatch: caller %d, library %zu", desc->struct_size, sizeof(lbm_case_desc));
        return LBM_ERR_ARG;
    }
    if (desc->nx < 5 || desc->ny < 6 || desc->nz < 5 || desc->case_rule < 0 || desc->case_rule > 3 ||
        desc->z_begin < 0 || desc->z_end > desc->nz || desc->z_begin >= desc->z_end || desc->tau <= 0.5 ||
        desc->n_bc < 0 || desc->n_bc > LBM_MAX_BC || desc->n_openings < 0 || desc->n_openings > LBM_MAX_OPENINGS ||
        (desc->precision != LBM_F32 && desc->precision != LBM_F64)) {
        g_create_error = "invalid case descriptor (dims >= 5, tau > 0.5, 0 <= z_begin < z_end <= nz)";
        return LBM_ERR_ARG;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || desc->device >= ndev || desc->device < 0) {
        cudaGetLastError();
        g_create_error = "no usable CUDA device: liblbm_b200 has no CPU path";
        return LBM_ERR_NO_DEVICE;
    }
    SolverBase *s = nullptr;
    int r;
    if (desc->precision == LBM_F32) {
        auto *p = new (std::nothrow) Solver<float>();
        if (!p) return LBM_ERR_NOMEM;
        p->d = *desc;
        r = p->setup();
        s = p;
    } else {
        auto *p = new (std::nothrow) Solver<double>();
        if (!p) return LBM_ERR_NOMEM;
        p->d = *desc;
        r = p->setup();
        s = p;
    }
    if (r) {
        g_create_error = s->err;
        delete s;
        return r;
    }
    *out = new lbm_solver_s{s};
    return LBM_OK;
}

int lbm_destroy(lbm_handle h) {
    if (!h) return LBM_ERR_ARG;
    delete h->s;
    delete h;
    return LBM_OK;
}
const char *lbm_last_error(lbm_handle h) { return h ? h->s->err.c_str() : lbm::g_create_error.c_str(); }

#define H_OR_FAIL \
    if (!h) return LBM_ERR_ARG

int lbm_set_flag(lbm_handle h, const int32_t *f) { H_OR_FAIL; return h->s->set_flag(f); }
int lbm_set_flag_slab(lbm_handle h, const uint8_t *f, int32_t z0, int32_t nz) { H_OR_FAIL; return h->s->set_flag_slab(f, z0, nz); }
int lbm_geo_pre(lbm_handle h) { H_OR_FAIL; return h->s->geo_pre(); }
int lbm_index_transform(lbm_handle h, int64_t *n) { H_OR_FAIL; return h->s->index_transform(n); }
int lbm_local_stored_count(lbm_handle h, int64_t *n) { H_OR_FAIL; return n ? h->s->local_stored_count(n) : LBM_ERR_ARG; }
int lbm_set_compact_offset(lbm_handle h, int64_t off, int64_t total) { H_OR_FAIL; return h->s->set_compact_offset(off, total); }
int lbm_read_vel(lbm_handle h) { H_OR_FAIL; return h->s->read_vel(); }
int lbm_set_bc_planes(lbm_handle h, const float *a, const float *b) { H_OR_FAIL; return h->s->set_bc_planes(a, b); }
int lbm_initialize(lbm_handle h) { H_OR_FAIL; return h->s->initialize(); }
int lbm_step(lbm_handle h, int32_t n) { H_OR_FAIL; return h->s->step(n, nullptr); }
int lbm_step_timed(lbm_handle h, int32_t n, float *ms) { H_OR_FAIL; return ms ? h->s->step(n, ms) : LBM_ERR_ARG; }
int64_t lbm_step_count(lbm_handle h) { return h ? h->s->steps : -1; }
int64_t lbm_launch_count(lbm_handle h) { return h ? h->s->launches : -1; }
int lbm_residual(lbm_handle h, int32_t kind, double *v) { H_OR_FAIL; return v ? h->s->residual(kind, v) : LBM_ERR_ARG; }
int lbm_get_geo(lbm_handle h, int32_t *g) { H_OR_FAIL; return g ? h->s->get_geo(g) : LBM_ERR_ARG; }
int lbm_get_index(lbm_handle h, int32_t *g) { H_OR_FAIL; return g ? h->s->get_index(g) : LBM_ERR_ARG; }
int lbm_get_fields(lbm_handle h, void *rho, void *ux, void *uy, void *uz, int64_t *first, int64_t *count) {
    H_OR_FAIL;
    return h->s->get_fields(rho, ux, uy, uz, first, count);
}
int lbm_debug_get_populations(lbm_handle h, void *f) { H_OR_FAIL; return f ? h->s->get_populations(f) : LBM_ERR_ARG; }
int64_t lbm_num_fluid(lbm_handle h) { return h ? h->s->nfluid : -1; }
int64_t lbm_device_bytes(lbm_handle h) { return h ? h->s->dev_bytes : -1; }
int lbm_output_save(lbm_handle h, int32_t t) { H_OR_FAIL; return h->s->output_save(t); }
int lbm_set_output_format(lbm_handle h, int32_t format) {
    H_OR_FAIL;
    if (format != LBM_OUT_ASCII_VTK && format != LBM_OUT_BINARY_VTK) {
        h->s->err = "unknown output format";
        return LBM_ERR_ARG;
    }
    h->s->out_format = format;
    return 0;
}
int lbm_run_fixed(lbm_handle h, int32_t repeat, int32_t time_save, int32_t wf) { H_OR_FAIL; return h->s->run_fixed(repeat, time_save, wf); }
int lbm_run_converge(lbm_handle h, int32_t max_it, double tol, int32_t stag_max, int32_t time_save, int32_t wf,
                     int32_t *its, double *res) {
    H_OR_FAIL;
    return h->s->run_converge(max_it, tol, stag_max, time_save, wf, its, res);
}
int lbm_halo_buffers(lbm_handle h, int32_t side, void **send, void **recv, size_t *send_bytes, size_t *recv_bytes) {
    H_OR_FAIL;
    return h->s->halo_buffers(side, send, recv, send_bytes, recv_bytes);
}
int lbm_p2p_export(lbm_handle h, lbm_ipc_handle handles[2], void *ptrs[2], int64_t byte_offset[2], int64_t *qstride,
                   int64_t halo_c0[2], int64_t face_c0[2]) {
    H_OR_FAIL;
    return h->s->p2p_export(handles, ptrs, byte_offset, qstride, halo_c0, face_c0);
}
int lbm_p2p_open(const lbm_ipc_handle *handle, void **dev_ptr) {
    if (!handle || !dev_ptr) return LBM_ERR_ARG;
    cudaIpcMemHandle_t ih;
    memcpy(&ih, handle, sizeof ih);
    cudaError_t e = cudaIpcOpenMemHandle(dev_ptr, ih, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        lbm::g_create_error = std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e);
        return LBM_ERR_CUDA;
    }
    return LBM_OK;
}
int lbm_p2p_close(void *dev_ptr) { return cudaIpcCloseMemHandle(dev_ptr) == cudaSuccess ? LBM_OK : LBM_ERR_CUDA; }
int lbm_p2p_attach(lbm_handle h, int32_t side, void *pa, void *pb, int64_t pqs, int64_t pc0, int64_t pown) {
    H_OR_FAIL;
    return h->s->p2p_attach(side, pa, pb, pqs, pc0, pown);
}
int lbm_checkpoint_save(lbm_handle h, const char *path) { H_OR_FAIL; return h->s->checkpoint(path, true); }
int lbm_checkpoint_load(lbm_handle h, const char *path) { H_OR_FAIL; return h->s->checkpoint(path, false); }
int lbm_step_begin(lbm_handle h, int32_t flags) { H_OR_FAIL; return h->s->step_begin(flags); }
int lbm_step_interior(lbm_handle h) { H_OR_FAIL; return h->s->step_interior(); }
int lbm_step_end(lbm_handle h) { H_OR_FAIL; return h->s->step_end(); }
int lbm_last_velsum(lbm_handle h, double *v) { H_OR_FAIL; return v ? h->s->last_velsum(v) : LBM_ERR_ARG; }
void *lbm_stream(lbm_handle h) { return h ? h->s->stream_ptr() : nullptr; }
int lbm_sync(lbm_handle h) { H_OR_FAIL; return h->s->sync(); }
int lbm_slab_step(lbm_handle h, int32_t n, int32_t flags_last, double *S_out, float *elapsed_ms) {
    H_OR_FAIL;
    return h->s->slab_steps(n, flags_last, S_out, elapsed_ms);
}
int lbm_sync_export(lbm_handle h, lbm_ipc_handle *handle, void **ptr, int64_t *byte_offset) {
    H_OR_FAIL;
    return h->s->sync_export(handle, ptr, byte_offset);
}
int lbm_mail_export(lbm_handle h, int32_t side, lbm_ipc_handle *handle, void **ptr, int64_t *byte_offset, int64_t *stride,
                    int64_t *guard) {
    H_OR_FAIL;
    return h->s->mail_export(side, handle, ptr, byte_offset, stride, guard);
}
int lbm_mail_attach(lbm_handle h, int32_t side, void *peer_mail) { H_OR_FAIL; return h->s->mail_attach(side, peer_mail); }
int lbm_mail_stage(lbm_handle h, int32_t side) { H_OR_FAIL; return h->s->mail_stage(side); }
int lbm_sync_attach(lbm_handle h, int32_t side, void *peer_sync) { H_OR_FAIL; return h->s->sync_attach(side, peer_sync); }
int lbm_set_option(lbm_handle h, const char *name, double value) { H_OR_FAIL; return name ? h->s->set_option(name, value) : LBM_ERR_ARG; }
int lbm_set_collision(lbm_handle h, int32_t model, double magic) { H_OR_FAIL; return h->s->set_collision(model, magic); }
int lbm_debug_selfcheck(lbm_handle h, uint64_t out[3]) { H_OR_FAIL; return out ? h->s->selfcheck(out) : LBM_ERR_ARG; }
int lbm_write_bc_csv(lbm_handle h, const char *path) { H_OR_FAIL; return path ? h->s->write_bc_csv(path) : LBM_ERR_ARG; }

// ============================================================================
// several z-slabs driven from ONE process (SURVEY 8b: lbm_create_distributed)
// ============================================================================
struct lbm_group_s {
    lbm_case_desc d;
    std::vector<lbm_handle> h;
    std::vector<int> dev;
    std::string err;
    int64_t nlattice = 0;
    bool ready = false;
    int fail(int code, const std::string &m) {
        err = m;
        return code;
    }
    int from(int r, int code) {  // propagate a slab's error
        if (code) err = lbm::fmt("slab %d: %s", r, lbm_last_error(h[(size_t)r]));
        return code;
    }
};
static thread_local std::string g_group_error;
#define G_OR_FAIL \
    if (!g) return LBM_ERR_ARG

int lbm_create_distributed(const lbm_case_desc *desc, int32_t nslabs, const int32_t *devices, lbm_group *out) {
    if (!desc || !out || nslabs < 1 || nslabs > desc->nz) {
        g_group_error = "lbm_create_distributed: bad arguments (1 <= nslabs <= nz)";
        return LBM_ERR_ARG;
    }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        g_group_error = "no usable CUDA device: liblbm_b200 has no CPU path";
        return LBM_ERR_NO_DEVICE;
    }
    auto *g = new lbm_group_s();
    g->d = *desc;
    const int base = desc->nz / nslabs, rem = desc->nz % nslabs;  // contiguous, near-equal z ranges
    int z = 0;
    for (int r = 0; r < nslabs; r++) {
        lbm_case_desc dr = *desc;
        const int n = base + (r < rem ? 1 : 0);
        dr.z_begin = z, dr.z_end = z + n, z += n;
        dr.device = devices ? devices[r] : r % ndev;
        lbm_handle hr = nullptr;
        int rc = lbm_create(&dr, &hr);
        if (rc) {
            g_group_error = lbm::fmt("slab %d: %s", r, lbm_last_error(nullptr));
            for (auto x : g->h) lbm_destroy(x);
            delete g;
            return rc;
        }
        g->h.push_back(hr), g->dev.push_back(dr.device);
    }
    *out = g;
    return LBM_OK;
}
int lbm_group_destroy(lbm_group g) {
    G_OR_FAIL;
    for (auto x : g->h) lbm_sync(x);
    for (auto x : g->h) lbm_destroy(x);
    delete g;
    return LBM_OK;
}
const char *lbm_group_last_error(lbm_group g) { return g ? g->err.c_str() : g_group_error.c_str(); }
int32_t lbm_group_size(lbm_group g) { return g ? (int32_t)g->h.size() : -1; }
lbm_handle lbm_group_slab(lbm_group g, int32_t r) { return g && r >= 0 && r < (int)g->h.size() ? g->h[(size_t)r] : nullptr; }

// geo_pre .. initialize on every slab, compact numbering continued across slabs (bif:241-252), then the
// slabs are wired to each other: peer stores for the crossing populations, events for the ordering
int lbm_group_setup(lbm_group g, const int32_t *flag_cartesian, const float *inlet_uy, const float *outlet_uy,
                    int64_t *nlattice) {
    G_OR_FAIL;
    const int P = (int)g->h.size();
    int rc;
    for (int r = 0; r < P; r++) {
        if (flag_cartesian && (rc = g->from(r, lbm_set_flag(g->h[(size_t)r], flag_cartesian)))) return rc;
        if ((rc = g->from(r, lbm_geo_pre(g->h[(size_t)r])))) return rc;
    }
    std::vector<int64_t> cnt((size_t)P), off((size_t)P);
    int64_t total = 0;
    for (int r = 0; r < P; r++) {
        if ((rc = g->from(r, lbm_local_stored_count(g->h[(size_t)r], &cnt[(size_t)r])))) return rc;
        off[(size_t)r] = total, total += cnt[(size_t)r];
    }
    const bool want_planes = g->d.case_rule == LBM_CASE_GEO_Y_INOUT;
    for (int r = 0; r < P; r++) {
        lbm_handle h = g->h[(size_t)r];
        if ((rc = g->from(r, lbm_set_compact_offset(h, off[(size_t)r], total)))) return rc;
        if ((rc = g->from(r, lbm_index_transform(h, nullptr)))) return rc;
        if (want_planes) {
            if (inlet_uy && outlet_uy) rc = lbm_set_bc_planes(h, inlet_uy, outlet_uy);
            else rc = lbm_read_vel(h);  // bif:255-327
            if ((rc = g->from(r, rc))) return rc;
        }
        if ((rc = g->from(r, lbm_initialize(h)))) return rc;
    }
    // wiring
    for (int r = 0; r + 1 < P; r++) {
        const int da = g->dev[(size_t)r], db = g->dev[(size_t)r + 1];
        if (da != db) {
            int ok_ab = 0, ok_ba = 0;
            cudaDeviceCanAccessPeer(&ok_ab, da, db), cudaDeviceCanAccessPeer(&ok_ba, db, da);
            if (!ok_ab || !ok_ba) return g->fail(LBM_ERR_CUDA, lbm::fmt("devices %d and %d cannot access each other's memory", da, db));
            cudaSetDevice(da);
            cudaError_t e = cudaDeviceEnablePeerAccess(db, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return g->fail(LBM_ERR_CUDA, cudaGetErrorString(e));
            cudaSetDevice(db);
            e = cudaDeviceEnablePeerAccess(da, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return g->fail(LBM_ERR_CUDA, cudaGetErrorString(e));
            cudaGetLastError();
        }
    }
    struct Exp {
        void *ptrs[2];
        int64_t qs, halo[2], face[2];
    };
    std::vector<Exp> ex((size_t)P);
    for (int r = 0; r < P; r++)
        if ((rc = g->from(r, lbm_p2p_export(g->h[(size_t)r], nullptr, ex[(size_t)r].ptrs, nullptr, &ex[(size_t)r].qs, ex[(size_t)r].halo,
                                            ex[(size_t)r].face))))
            return rc;
    for (int r = 0; r < P; r++)
        for (int side = 0; side < 2; side++) {
            const int nb = side == 0 ? r - 1 : r + 1;
            if (nb < 0 || nb >= P) continue;
            const Exp &e = ex[(size_t)nb];
            // my low face feeds the neighbour's HIGH halo plane and vice versa
            if ((rc = g->from(r, lbm_p2p_attach(g->h[(size_t)r], side, e.ptrs[0], e.ptrs[1], e.qs, e.halo[1 - side], e.face[1 - side]))))
                return rc;
            g->h[(size_t)r]->s->set_inproc_neighbour(side, g->h[(size_t)nb]->s);
        }
    g->nlattice = total, g->ready = true;
    if (nlattice) *nlattice = total;
    return LBM_OK;
}

// one time step on every slab: launches only; slab r+1 is enqueued right after slab r so that no stream
// runs ahead of its neighbours by more than the launch queue allows
static int group_enqueue(lbm_group g, int flags, int slot) {
    for (size_t r = 0; r < g->h.size(); r++) {
        SolverBase *s = g->h[r]->s;
        int rc = s->enqueue_step(flags, slot >= 0 ? s->acc_slot(slot) : s->acc_slot(0));
        if (rc) return g->from((int)r, rc);
    }
    return 0;
}
static int group_sync(lbm_group g) {
    for (size_t r = 0; r < g->h.size(); r++) {
        int rc = lbm_sync(g->h[r]);
        if (rc) return g->from((int)r, rc);
    }
    return 0;
}
int lbm_group_step(lbm_group g, int32_t n, float *elapsed_ms) {
    G_OR_FAIL;
    if (!g->ready) return g->fail(LBM_ERR_STATE, "lbm_group_step before lbm_group_setup");
    if (n < 0) return g->fail(LBM_ERR_ARG, "negative step count");
    int rc = group_sync(g);
    if (rc) return rc;
    const auto t0 = std::chrono::steady_clock::now();
    for (int i = 0; i < n; i++)
        if ((rc = group_enqueue(g, i == n - 1 ? LBM_STEP_MOMENTS : 0, -1))) return rc;
    if ((rc = group_sync(g))) return rc;
    if (elapsed_ms) *elapsed_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return LBM_OK;
}
int lbm_group_set_collision(lbm_group g, int32_t model, double magic) {
    G_OR_FAIL;
    const std::string why = lbm::collision_refusal(g->d, model, magic);  // every slab has the group's tau and math
    if (!why.empty()) return g->fail(LBM_ERR_ARG, "lbm_group_set_collision: " + why);
    for (size_t r = 0; r < g->h.size(); r++) {
        const int rc = lbm_set_collision(g->h[r], model, magic);
        if (rc) return g->from((int)r, rc);
    }
    return LBM_OK;
}
int64_t lbm_group_num_fluid(lbm_group g) {
    if (!g) return -1;
    int64_t n = 0;
    for (auto x : g->h) n += lbm_num_fluid(x);
    return n;
}
// "all-reduced" reductions: the sum of the slabs' shares
int lbm_group_residual(lbm_group g, int32_t kind, double *value) {
    G_OR_FAIL;
    if (!value) return LBM_ERR_ARG;
    double acc = 0.0;
    for (size_t r = 0; r < g->h.size(); r++) {
        double v = 0.0;
        int rc = lbm_residual(g->h[r], kind, &v);
        if (rc) return g->from((int)r, rc);
        acc += v;
    }
    *value = acc;
    return LBM_OK;
}
// fields of the whole domain in the reference's compact order (NLATTICE entries each)
int lbm_group_get_fields(lbm_group g, void *rho, void *ux, void *uy, void *uz) {
    G_OR_FAIL;
    if (!g->ready) return g->fail(LBM_ERR_STATE, "lbm_group_get_fields before lbm_group_setup");
    const size_t es = g->d.precision == LBM_F64 ? 8 : 4;
    int64_t first = 0;
    for (size_t r = 0; r < g->h.size(); r++) {
        int64_t cnt = 0;
        if ((lbm_local_stored_count(g->h[r], &cnt))) return g->from((int)r, LBM_ERR_STATE);
        auto at = [&](void *p) { return p ? (void *)((char *)p + (size_t)first * es) : nullptr; };
        int rc = lbm_get_fields(g->h[r], at(rho), at(ux), at(uy), at(uz), nullptr, nullptr);
        if (rc) return g->from((int)r, rc);
        first += cnt;
    }
    return LBM_OK;
}
int lbm_group_get_index(lbm_group g, int32_t *index_cartesian) {
    G_OR_FAIL;
    size_t at = 0;
    for (size_t r = 0; r < g->h.size(); r++) {
        int rc = lbm_get_index(g->h[r], index_cartesian + at);
        if (rc) return g->from((int)r, rc);
        at += (size_t)g->d.nx * g->d.ny * (size_t)(g->h[r]->s->d.z_end - g->h[r]->s->d.z_begin);
    }
    return LBM_OK;
}
int lbm_group_set_output_format(lbm_group g, int32_t format) {
    G_OR_FAIL;
    for (size_t r = 0; r < g->h.size(); r++) {
        int rc = lbm_set_output_format(g->h[r], format);
        if (rc) return g->from((int)r, rc);
    }
    return LBM_OK;
}
// outputSave(t) for a sharded run: ASCII -> ONE file, byte-compatible with the single-domain writer (the
// slabs' fields are gathered on the host); binary -> every slab writes its own piece
int lbm_group_output_save(lbm_group g, int32_t t) {
    G_OR_FAIL;
    if (!g->ready) return g->fail(LBM_ERR_STATE, "lbm_group_output_save before lbm_group_setup");
    if (g->h[0]->s->out_format == LBM_OUT_BINARY_VTK) {
        for (size_t r = 0; r < g->h.size(); r++) {
            int rc = lbm_output_save(g->h[r], t);
            if (rc) return g->from((int)r, rc);
        }
        return LBM_OK;
    }
    const size_t es = g->d.precision == LBM_F64 ? 8 : 4, n = (size_t)g->nlattice;
    std::vector<int32_t> idx((size_t)g->d.nx * g->d.ny * g->d.nz);
    std::vector<char> f(4 * n * es);
    int rc = lbm_group_get_index(g, idx.data());
    if (rc) return rc;
    if ((rc = lbm_group_get_fields(g, f.data(), f.data() + n * es, f.data() + 2 * n * es, f.data() + 3 * n * es))) return rc;
    return g->from(0, g->h[0]->s->write_global(t, idx.data(), f.data(), f.data() + n * es, f.data() + 2 * n * es,
                                                f.data() + 3 * n * es, g->nlattice));
}

// ldc.cu:653-685 / pos.cu:986-1019 on several slabs: S_k = sum over slabs of each slab's share, the
// stopping rule applied on the host exactly as in the single-domain loop (Solver::run_converge)
int lbm_group_run_converge(lbm_group g, int32_t max_it, double tol_d, int32_t stag_max, int32_t time_save, int32_t write_files,
                           int32_t *iterations, double *residual_out) {
    G_OR_FAIL;
    if (!g->ready) return g->fail(LBM_ERR_STATE, "run before lbm_group_setup");
    if (time_save <= 0) return g->fail(LBM_ERR_ARG, "time_save must be positive");
    const int P = (int)g->h.size();
    std::ofstream logfile;
    if (write_files) logfile.open(std::string(g->d.out_dir) + "/CONVERGENCE.log");
    const auto t0 = std::chrono::steady_clock::now();
    const float tol = (float)tol_d;
    float residual = 0.f, sum_current = 0.f;
    int k = 0, tol_count = 0, rc;
    const int max_batch = 48;
    std::vector<double> S((size_t)max_batch), part((size_t)max_batch);
    while (k <= max_it && tol_count <= stag_max) {
        int nb = std::min(max_batch, std::max(1, stag_max + 1 - tol_count));
        nb = std::min(nb, max_it - k + 1);
        for (int j = 0; j < nb; j++)
            if ((k + j) % time_save == 0) {
                nb = j + 1;
                break;
            }
        for (int r = 0; r < P; r++)
            if ((rc = g->from(r, g->h[(size_t)r]->s->zero_acc(0, nb)))) return rc;
        for (int j = 0; j < nb; j++)
            if ((rc = group_enqueue(g, LBM_STEP_MOMENTS | LBM_STEP_VELSUM, j))) return rc;
        std::fill(S.begin(), S.end(), 0.0);
        for (int r = 0; r < P; r++) {
            if ((rc = g->from(r, g->h[(size_t)r]->s->fetch_acc(0, nb, part.data())))) return rc;
            for (int j = 0; j < nb; j++) S[(size_t)j] += part[(size_t)j];
        }
        for (int j = 0; j < nb; j++) {
            const float sum_next = (float)S[(size_t)j];
            residual = std::fabs(sum_next - sum_current) / sum_next;
            if (k % time_save == 0 && write_files) {
                const float milli = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
                std::cout << "ITERATION # " << k << ", collapse time: " << milli << " ms, residual:" << residual << std::endl;
                logfile << residual << std::endl;
                if ((rc = lbm_group_output_save(g, k))) return rc;
            }
            k++;
            sum_current = sum_next;
            if (residual <= tol) tol_count++;
            if (!(k <= max_it && tol_count <= stag_max)) break;
        }
    }
    const float milli = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (write_files) {
        if ((rc = lbm_group_output_save(g, k))) return rc;
        std::cout << "TOTAL RUNNING TIME: " << milli << " MILLI SECONDS" << "#LATTICE" << g->nlattice << std::endl;
        std::cout << "Residual is " << residual << std::endl;
        logfile << "TOTAL RUNNING TIME: " << milli << " MILLI SECONDS" << "#LATTICE" << g->nlattice << " ERROR IS" << residual
                << std::endl;
    }
    if (iterations) *iterations = k;
    if (residual_out) *residual_out = residual;
    return LBM_OK;
}
// bif.cu:1246-1274 / cor.cu:1100-1132 on several slabs; the residual between saves is the device reduction
// sum(u^2) over the slabs (the single-domain loop sums the same terms on the host in long double)
int lbm_group_run_fixed(lbm_group g, int32_t repeat, int32_t time_save, int32_t write_files) {
    G_OR_FAIL;
    if (!g->ready) return g->fail(LBM_ERR_STATE, "run before lbm_group_setup");
    if (time_save <= 0) return g->fail(LBM_ERR_ARG, "time_save must be positive");
    std::ofstream logfile;
    if (write_files) logfile.open(std::string(g->d.out_dir) + "/CONVERGENCE.log");
    const auto t0 = std::chrono::steady_clock::now();
    float residual = 0.f;
    int done = 0, rc;
    double sum1 = 0.0, sum2 = 0.0;
    while (done <= repeat) {
        const int i_save = ((done + time_save - 1) / time_save) * time_save;
        const int upto = std::min(i_save, repeat);
        if ((rc = lbm_group_step(g, upto - done + 1, nullptr))) return rc;
        done = upto + 1;
        if (upto % time_save == 0) {
            sum1 = sum2;  // fields of the previous save (0 at first)
            if ((rc = lbm_group_residual(g, LBM_RES_U2SUM, &sum2))) return rc;
            residual = (float)(std::fabs(sum1 - sum2) / sum2);
            const float milli = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
            if (write_files) {
                logfile << residual << std::endl;
                std::cout << "ITERATION # " << upto << ", collapse time: " << milli << " ms, residual:" << residual << std::endl;
                if ((rc = lbm_group_output_save(g, upto))) return rc;
            }
        }
    }
    const float milli = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (write_files) {
        std::cout << "TOTAL RUNNING TIME: " << milli << " MILLI SECONDS" << "#LATTICE" << g->nlattice << std::endl;
        logfile << "TOTAL RUNNING TIME: " << milli << " MILLI SECONDS" << "#LATTICE" << g->nlattice << " ERROR IS" << residual
                << std::endl;
    }
    return LBM_OK;
}

}  // extern "C"
