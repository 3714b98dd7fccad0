"""ctypes binding of liblbm_b200.so and a host-side mirror of the reference's case interface.

The reference (Xinhuan-Imperial/Lattice-Boltzmann-Method-GPU) has no library API: each of its
four programs calls, from main(), the file-scope functions

    geo_pre(); index_transform(); read_vel(); initialize();
    loop { update<<<>>>; boundary_stream<<<>>>; swap }   calc_res(); outputSave(t);

(bifurcation/bifurcation.cu:1177-1326).  :class:`Case` keeps those names and that order, so a
driver or a test written against it reads like the reference's main().  All compute happens in
the CUDA library; there is no CPU fallback -- if the shared library is missing or no GPU is
visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
# LBM_B200_LIB selects another build of the same library (the self-checking one, tools/selfcheck.py)
LIB_PATH = Path(os.environ["LBM_B200_LIB"]) if os.environ.get("LBM_B200_LIB") else PKG / "liblbm_b200.so"

# enums of include/lbm_b200.h
CASE_LDC, CASE_POISEUILLE, CASE_GEO_Y_INOUT, CASE_GEO_OPENINGS = 0, 1, 2, 3
F32, F64 = 0, 1
STORE_DENSE_AB, STORE_DENSE_AA, STORE_SPARSE_AB, STORE_SPARSE_AA = 0, 1, 2, 3
MATH_FAST, MATH_STRICT = 0, 1
COLL_BGK, COLL_TRT = 0, 1
BC_NONE, BC_V, BC_P, BC_VP = 0, 1, 2, 3
SRC_CONST, SRC_PARABOLA, SRC_PLANE_INLET, SRC_PLANE_OUTLET = 0, 1, 2, 3
RES_VELSUM, RES_U2SUM = 0, 1
OUT_ASCII_VTK, OUT_BINARY_VTK = 0, 1
STEP_MOMENTS, STEP_VELSUM = 1, 2
MAX_BC, MAX_OPENINGS = 8, 8


class BcDesc(C.Structure):
    _fields_ = [
        ("label", C.c_int32), ("kind", C.c_int32), ("normal_axis", C.c_int32), ("normal_sign", C.c_int32),
        ("vel_axis", C.c_int32), ("source", C.c_int32), ("pulsatile", C.c_int32), ("reserved", C.c_int32),
        ("value", C.c_double), ("init_value", C.c_double),
    ]


class OpeningRule(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("axis", "coord", "lo_a", "hi_a", "lo_b", "hi_b", "reps", "reserved")]


class CaseDesc(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("case_rule", C.c_int32),
        ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32),
        ("precision", C.c_int32), ("storage", C.c_int32), ("math", C.c_int32), ("device", C.c_int32),
        ("geo_yfast", C.c_int32), ("z_begin", C.c_int32), ("z_end", C.c_int32),
        ("n_bc", C.c_int32), ("n_openings", C.c_int32),
        ("tau", C.c_double), ("u_max", C.c_double),
        ("C_U", C.c_double), ("C_rho", C.c_double), ("CH", C.c_double),
        ("pulse_amp", C.c_double), ("pulse_period", C.c_double),
        ("bc", BcDesc * MAX_BC), ("openings", OpeningRule * MAX_OPENINGS),
        ("geo_path", C.c_char * 256), ("bc_path", C.c_char * 256), ("out_dir", C.c_char * 256),
        ("out_name", C.c_char * 32),
    ]


class LbmError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"liblbm_b200 status {status}: {msg}")
        self.status = status


# every symbol include/lbm_b200.h declares (tests check the library exports all of them)
ABI_SYMBOLS = [
    "lbm_case_defaults", "lbm_create", "lbm_destroy", "lbm_last_error", "lbm_set_flag", "lbm_set_flag_slab", "lbm_geo_pre",
    "lbm_index_transform", "lbm_local_stored_count", "lbm_set_compact_offset", "lbm_read_vel", "lbm_set_bc_planes",
    "lbm_initialize", "lbm_step", "lbm_step_timed", "lbm_step_count", "lbm_launch_count", "lbm_residual",
    "lbm_get_geo", "lbm_get_index", "lbm_get_fields", "lbm_debug_get_populations", "lbm_num_fluid",
    "lbm_device_bytes", "lbm_output_save", "lbm_set_output_format", "lbm_voxelize_stl", "lbm_voxelize_triangles", "lbm_voxel_last_error", "lbm_run_fixed", "lbm_run_converge", "lbm_halo_buffers",
    "lbm_step_begin", "lbm_step_interior", "lbm_step_end", "lbm_last_velsum", "lbm_stream", "lbm_sync",
    "lbm_p2p_export", "lbm_p2p_open", "lbm_p2p_close", "lbm_p2p_attach", "lbm_checkpoint_save", "lbm_checkpoint_load",
    "lbm_slab_step", "lbm_sync_export", "lbm_sync_attach", "lbm_mail_export", "lbm_mail_attach", "lbm_mail_stage", "lbm_write_bc_csv", "lbm_debug_selfcheck", "lbm_set_option",
    "lbm_set_collision",
    "lbm_create_distributed", "lbm_group_destroy", "lbm_group_last_error", "lbm_group_size", "lbm_group_slab",
    "lbm_group_setup", "lbm_group_step", "lbm_group_num_fluid", "lbm_group_residual", "lbm_group_get_fields",
    "lbm_group_get_index", "lbm_group_set_output_format", "lbm_group_output_save", "lbm_group_run_fixed",
    "lbm_group_run_converge", "lbm_group_set_collision",
]

_lib = None


class VoxelGrid(C.Structure):
    """lbm_voxel_grid (include/lbm_b200.h)"""
    _fields_ = [("origin", C.c_double * 3), ("spacing", C.c_double), ("nx", C.c_int32), ("ny", C.c_int32),
                ("nz", C.c_int32), ("reserved", C.c_int32)]


def load_library() -> C.CDLL:
    """dlopen the in-tree CUDA library.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"or `make -C {PKG / 'csrc'}`.  There is no CPU fallback.")
    L = C.CDLL(str(LIB_PATH))
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    P = C.POINTER
    sig = {
        "lbm_case_defaults": ([i32, P(CaseDesc)], C.c_int),
        "lbm_create": ([P(CaseDesc), P(vp)], C.c_int),
        "lbm_destroy": ([vp], C.c_int),
        "lbm_last_error": ([vp], C.c_char_p),
        "lbm_set_flag": ([vp, vp], C.c_int),
        "lbm_set_flag_slab": ([vp, vp, i32, i32], C.c_int),
        "lbm_geo_pre": ([vp], C.c_int),
        "lbm_index_transform": ([vp, P(i64)], C.c_int),
        "lbm_local_stored_count": ([vp, P(i64)], C.c_int),
        "lbm_set_compact_offset": ([vp, i64, i64], C.c_int),
        "lbm_read_vel": ([vp], C.c_int),
        "lbm_set_bc_planes": ([vp, vp, vp], C.c_int),
        "lbm_initialize": ([vp], C.c_int),
        "lbm_step": ([vp, i32], C.c_int),
        "lbm_step_timed": ([vp, i32, P(C.c_float)], C.c_int),
        "lbm_step_count": ([vp], i64),
        "lbm_launch_count": ([vp], i64),
        "lbm_residual": ([vp, i32, P(dbl)], C.c_int),
        "lbm_get_geo": ([vp, vp], C.c_int),
        "lbm_get_index": ([vp, vp], C.c_int),
        "lbm_get_fields": ([vp, vp, vp, vp, vp, P(i64), P(i64)], C.c_int),
        "lbm_debug_get_populations": ([vp, vp], C.c_int),
        "lbm_num_fluid": ([vp], i64),
        "lbm_device_bytes": ([vp], i64),
        "lbm_output_save": ([vp, i32], C.c_int),
        "lbm_set_output_format": ([vp, i32], C.c_int),
        "lbm_voxelize_stl": ([C.c_char_p, P(VoxelGrid), i32, i32, i32, vp], C.c_int),
        "lbm_voxelize_triangles": ([vp, i64, P(VoxelGrid), i32, i32, i32, vp], C.c_int),
        "lbm_voxel_last_error": ([], C.c_char_p),
        "lbm_run_fixed": ([vp, i32, i32, i32], C.c_int),
        "lbm_run_converge": ([vp, i32, dbl, i32, i32, i32, P(i32), P(dbl)], C.c_int),
        "lbm_halo_buffers": ([vp, i32, P(vp), P(vp), P(C.c_size_t), P(C.c_size_t)], C.c_int),
        "lbm_step_begin": ([vp, i32], C.c_int),
        "lbm_step_interior": ([vp], C.c_int),
        "lbm_step_end": ([vp], C.c_int),
        "lbm_last_velsum": ([vp, P(dbl)], C.c_int),
        "lbm_p2p_export": ([vp, vp, P(vp), P(i64), P(i64), P(i64), P(i64)], C.c_int),
        "lbm_p2p_open": ([vp, P(vp)], C.c_int),
        "lbm_p2p_close": ([vp], C.c_int),
        "lbm_p2p_attach": ([vp, i32, vp, vp, i64, i64, i64], C.c_int),
        "lbm_checkpoint_save": ([vp, C.c_char_p], C.c_int),
        "lbm_checkpoint_load": ([vp, C.c_char_p], C.c_int),
        "lbm_stream": ([vp], vp),
        "lbm_sync": ([vp], C.c_int),
        "lbm_slab_step": ([vp, i32, i32, vp, P(C.c_float)], C.c_int),
        "lbm_sync_export": ([vp, vp, P(vp), P(i64)], C.c_int),
        "lbm_sync_attach": ([vp, i32, vp], C.c_int),
        "lbm_mail_export": ([vp, i32, vp, P(vp), P(i64), P(i64), P(i64)], C.c_int),
        "lbm_mail_attach": ([vp, i32, vp], C.c_int),
        "lbm_mail_stage": ([vp, i32], C.c_int),
        "lbm_write_bc_csv": ([vp, C.c_char_p], C.c_int),
        "lbm_debug_selfcheck": ([vp, vp], C.c_int),
        "lbm_set_option": ([vp, C.c_char_p, dbl], C.c_int),
        "lbm_set_collision": ([vp, i32, dbl], C.c_int),
        "lbm_create_distributed": ([P(CaseDesc), i32, vp, P(vp)], C.c_int),
        "lbm_group_destroy": ([vp], C.c_int),
        "lbm_group_last_error": ([vp], C.c_char_p),
        "lbm_group_size": ([vp], i32),
        "lbm_group_slab": ([vp, i32], vp),
        "lbm_group_setup": ([vp, vp, vp, vp, P(i64)], C.c_int),
        "lbm_group_step": ([vp, i32, P(C.c_float)], C.c_int),
        "lbm_group_num_fluid": ([vp], i64),
        "lbm_group_residual": ([vp, i32, P(dbl)], C.c_int),
        "lbm_group_get_fields": ([vp, vp, vp, vp, vp], C.c_int),
        "lbm_group_get_index": ([vp, vp], C.c_int),
        "lbm_group_set_output_format": ([vp, i32], C.c_int),
        "lbm_group_output_save": ([vp, i32], C.c_int),
        "lbm_group_run_fixed": ([vp, i32, i32, i32], C.c_int),
        "lbm_group_run_converge": ([vp, i32, dbl, i32, i32, i32, P(i32), P(dbl)], C.c_int),
        "lbm_group_set_collision": ([vp, i32, dbl], C.c_int),
    }
    for name, (args, res) in sig.items():
        fn = getattr(L, name)
        fn.argtypes, fn.restype = args, res
    _lib = L
    return L


def case_defaults(case_rule: int) -> CaseDesc:
    d = CaseDesc()
    rc = load_library().lbm_case_defaults(case_rule, C.byref(d))
    if rc:
        raise LbmError(rc, "unknown case rule")
    return d


class Case:
    """One simulation.  Methods carry the reference's function names."""

    def __init__(self, desc: CaseDesc):
        self._L = load_library()
        self.desc = desc
        self.dtype = np.dtype(np.float32 if desc.precision == F32 else np.float64)
        self._h = C.c_void_p()
        rc = self._L.lbm_create(C.byref(desc), C.byref(self._h))
        if rc:
            raise LbmError(rc, self._L.lbm_last_error(None).decode())
        self.nlattice = None
        self._keep = []

    # -- plumbing
    def _ck(self, rc):
        if rc:
            raise LbmError(rc, self._L.lbm_last_error(self._h).decode())

    @property
    def handle(self):
        return self._h

    @property
    def owned_shape(self):
        d = self.desc
        return (d.z_end - d.z_begin, d.ny, d.nx)

    def close(self):
        if self._h:
            self._L.lbm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- the reference's call sequence
    def set_flag(self, flag: np.ndarray):
        """binary voxel field [nz][ny][nx] from memory instead of ./geo.txt"""
        d = self.desc
        flag = np.ascontiguousarray(flag, dtype=np.int32)
        if flag.shape != (d.nz, d.ny, d.nx):
            raise ValueError(f"flag shape {flag.shape} != {(d.nz, d.ny, d.nx)}")
        self._ck(self._L.lbm_set_flag(self._h, flag.ctypes.data))

    def set_flag_slab(self, flag: np.ndarray, z_first: int):
        """planes [z_first, z_first + len(flag)) of the voxel field, uint8 [z][y][x]"""
        d = self.desc
        flag = np.ascontiguousarray(flag, dtype=np.uint8)
        if flag.shape[1:] != (d.ny, d.nx):
            raise ValueError(f"flag slab shape {flag.shape} does not match ny, nx = {(d.ny, d.nx)}")
        self._ck(self._L.lbm_set_flag_slab(self._h, flag.ctypes.data, int(z_first), int(flag.shape[0])))

    def needed_flag_planes(self):
        """z range of the voxel field this (slab) handle reads in geo_pre"""
        d = self.desc
        return max(0, d.z_begin - 3), min(d.nz, d.z_end + 3)

    def geo_pre(self):
        self._ck(self._L.lbm_geo_pre(self._h))

    def local_stored_count(self) -> int:
        n = C.c_int64()
        self._ck(self._L.lbm_local_stored_count(self._h, C.byref(n)))
        return n.value

    def set_compact_offset(self, offset: int, total: int):
        self._ck(self._L.lbm_set_compact_offset(self._h, offset, total))

    def index_transform(self) -> int:
        n = C.c_int64()
        self._ck(self._L.lbm_index_transform(self._h, C.byref(n)))
        self.nlattice = n.value
        return n.value

    def read_vel(self):
        self._ck(self._L.lbm_read_vel(self._h))

    def set_bc_planes(self, inlet_uy: np.ndarray, outlet_uy: np.ndarray):
        a = np.ascontiguousarray(inlet_uy, dtype=np.float32)
        b = np.ascontiguousarray(outlet_uy, dtype=np.float32)
        n = self.desc.nx * self.desc.nz
        if a.size != n or b.size != n:
            raise ValueError("BC planes must hold nx*nz floats")
        self._ck(self._L.lbm_set_bc_planes(self._h, a.ctypes.data, b.ctypes.data))

    def initialize(self):
        self._ck(self._L.lbm_initialize(self._h))

    def step(self, n: int = 1):
        """n iterations of update + boundary_stream + swap"""
        self._ck(self._L.lbm_step(self._h, int(n)))

    update = step

    def step_timed(self, n: int) -> float:
        ms = C.c_float()
        self._ck(self._L.lbm_step_timed(self._h, int(n), C.byref(ms)))
        return ms.value

    def step_begin(self, flags: int = 0):
        self._ck(self._L.lbm_step_begin(self._h, flags))

    def step_interior(self):
        self._ck(self._L.lbm_step_interior(self._h))

    def step_end(self):
        self._ck(self._L.lbm_step_end(self._h))

    def last_velsum(self) -> float:
        v = C.c_double()
        self._ck(self._L.lbm_last_velsum(self._h, C.byref(v)))
        return v.value

    def halo_buffers(self, side: int):
        s, r, ns, nr = C.c_void_p(), C.c_void_p(), C.c_size_t(), C.c_size_t()
        self._ck(self._L.lbm_halo_buffers(self._h, side, C.byref(s), C.byref(r), C.byref(ns), C.byref(nr)))
        return s.value, r.value, ns.value, nr.value

    # -- fused peer-to-peer halo exchange
    def p2p_export(self):
        """dict: two 64-byte IPC handles, two raw device pointers, q stride, [low, high] halo-plane offsets,
        [low, high] outermost-owned-plane offsets, byte offsets of the buffers inside their allocations"""
        handles = (C.c_ubyte * 128)()
        ptrs = (C.c_void_p * 2)()
        boff = (C.c_int64 * 2)()
        qs = C.c_int64()
        c0 = (C.c_int64 * 2)()
        f0 = (C.c_int64 * 2)()
        self._ck(self._L.lbm_p2p_export(self._h, handles, ptrs, boff, C.byref(qs), c0, f0))
        raw = bytes(handles)
        return {"handles": [raw[:64], raw[64:]], "ptrs": [ptrs[0], ptrs[1]], "qs": qs.value, "halo_c0": [c0[0], c0[1]],
                "face_c0": [f0[0], f0[1]], "boff": [boff[0], boff[1]]}

    def p2p_attach(self, side: int, peer_a, peer_b, peer_qstride: int = 0, peer_halo_c0: int = 0, peer_face_c0: int = 0):
        self._ck(self._L.lbm_p2p_attach(self._h, side, peer_a, peer_b, peer_qstride, peer_halo_c0, peer_face_c0))

    # -- the slab's time loop inside the library (neighbours ordered on the device)
    def sync_export(self):
        """dict: IPC handle of this slab's sync block, its raw pointer and byte offset inside its allocation"""
        handle = (C.c_ubyte * 64)()
        ptr, boff = C.c_void_p(), C.c_int64()
        self._ck(self._L.lbm_sync_export(self._h, handle, C.byref(ptr), C.byref(boff)))
        return {"handle": bytes(handle), "ptr": ptr.value, "boff": boff.value}

    def mail_export(self, side: int):
        """this slab's mailbox of `side` (dense in-place storage): IPC handle, raw pointer, byte offset, stride, guard"""
        handle = (C.c_ubyte * 64)()
        ptr, boff, ms, g = C.c_void_p(), C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self._L.lbm_mail_export(self._h, side, handle, C.byref(ptr), C.byref(boff), C.byref(ms), C.byref(g)))
        return {"handle": bytes(handle), "ptr": ptr.value, "boff": boff.value, "stride": ms.value, "guard": g.value}

    def mail_attach(self, side: int, peer_mail):
        self._ck(self._L.lbm_mail_attach(self._h, side, peer_mail))

    def mail_stage(self, side: int):
        """mailbox exchange of `side` through local staging buffers (transport without peer mapping)"""
        self._ck(self._L.lbm_mail_stage(self._h, side))

    def sync_attach(self, side: int, peer_sync):
        self._ck(self._L.lbm_sync_attach(self._h, side, peer_sync))

    def slab_step(self, n: int, moments_last: bool = True, velsum: bool = False):
        """n steps; returns (elapsed ms measured with CUDA events on the slab's stream, S per step or None)"""
        S = np.zeros(int(n), dtype=np.float64) if velsum else None
        ms = C.c_float()
        self._ck(self._L.lbm_slab_step(self._h, int(n), STEP_MOMENTS if moments_last else 0,
                                       S.ctypes.data if velsum else None, C.byref(ms)))
        return ms.value, S

    def set_option(self, name: str, value: float):
        self._ck(self._L.lbm_set_option(self._h, name.encode(), float(value)))

    def set_collision(self, model: int, magic: float = 3 / 16):
        """COLL_BGK (default) or COLL_TRT with the magic parameter Lambda (3/16: a straight bounce-back wall lies
        exactly half-way; 1/4: the usual choice for stability).  FAST arithmetic only; from the next step on."""
        self._ck(self._L.lbm_set_collision(self._h, int(model), float(magic)))

    def selfcheck(self):
        """(out-of-range accesses, elements touched by two threads in one launch, launches checked) of a
        self-checking build; raises LbmError on a normal build"""
        out = (C.c_uint64 * 3)()
        self._ck(self._L.lbm_debug_selfcheck(self._h, out))
        return int(out[0]), int(out[1]), int(out[2])

    def write_bc_csv(self, path):
        self._ck(self._L.lbm_write_bc_csv(self._h, os.fsencode(str(path))))

    def residual(self, kind: int = RES_VELSUM) -> float:
        v = C.c_double()
        self._ck(self._L.lbm_residual(self._h, kind, C.byref(v)))
        return v.value

    def calc_res(self) -> float:
        return self.residual(RES_U2SUM)

    def get_geo(self) -> np.ndarray:
        g = np.empty(self.owned_shape, dtype=np.int32)
        self._ck(self._L.lbm_get_geo(self._h, g.ctypes.data))
        return g

    def get_index(self) -> np.ndarray:
        g = np.empty(self.owned_shape, dtype=np.int32)
        self._ck(self._L.lbm_get_index(self._h, g.ctypes.data))
        return g

    def get_fields(self, out=None):
        """(rho, ux, uy, uz) in the reference's compact order (entries of the owned planes)"""
        n = self.local_stored_count()
        if out is None:
            out = [np.empty(n, dtype=self.dtype) for _ in range(4)]
        first, count = C.c_int64(), C.c_int64()
        self._ck(self._L.lbm_get_fields(self._h, *[o.ctypes.data for o in out], C.byref(first), C.byref(count)))
        self.compact_first, self.compact_count = first.value, count.value
        return out

    def get_populations(self) -> np.ndarray:
        n = self.local_stored_count()
        f = np.empty((19, n), dtype=self.dtype)
        self._ck(self._L.lbm_debug_get_populations(self._h, f.ctypes.data))
        return f

    def outputSave(self, t: int):
        self._ck(self._L.lbm_output_save(self._h, int(t)))

    def set_output_format(self, fmt: int):
        """OUT_ASCII_VTK (the reference's files, default) or OUT_BINARY_VTK (legacy-VTK BINARY; also for slabs)"""
        self._ck(self._L.lbm_set_output_format(self._h, int(fmt)))

    def run_fixed(self, repeat: int, time_save: int, write_files: bool = True):
        self._ck(self._L.lbm_run_fixed(self._h, repeat, time_save, int(write_files)))

    def run_converge(self, max_it=10000, tol=1e-6, stag_max=50, time_save=500, write_files=True):
        its, res = C.c_int32(), C.c_double()
        self._ck(self._L.lbm_run_converge(self._h, max_it, tol, stag_max, time_save, int(write_files),
                                          C.byref(its), C.byref(res)))
        return its.value, res.value

    def checkpoint_save(self, path):
        self._ck(self._L.lbm_checkpoint_save(self._h, os.fsencode(str(path))))

    def checkpoint_load(self, path):
        self._ck(self._L.lbm_checkpoint_load(self._h, os.fsencode(str(path))))

    def sync(self):
        self._ck(self._L.lbm_sync(self._h))

    @property
    def num_fluid(self) -> int:
        return self._L.lbm_num_fluid(self._h)

    @property
    def launch_count(self) -> int:
        return self._L.lbm_launch_count(self._h)

    @property
    def step_count(self) -> int:
        return self._L.lbm_step_count(self._h)

    @property
    def device_bytes(self) -> int:
        return self._L.lbm_device_bytes(self._h)

    @property
    def stream(self) -> int:
        return self._L.lbm_stream(self._h)


class Group:
    """Several z-slabs of one case driven from this process (`lbm_create_distributed`): the multi-GPU
    form of the reference's main().  devices=None puts slab r on device r modulo the device count;
    repeating a device gives several slabs on one GPU."""

    def __init__(self, desc: CaseDesc, nslabs: int, devices=None):
        self._L = load_library()
        desc.struct_size = C.sizeof(CaseDesc)
        self.desc = desc
        self.dtype = np.dtype(np.float64 if desc.precision == F64 else np.float32)
        self._g = C.c_void_p()
        dev = None if devices is None else (C.c_int32 * nslabs)(*[int(v) for v in devices])
        rc = self._L.lbm_create_distributed(C.byref(desc), int(nslabs), dev, C.byref(self._g))
        if rc:
            raise LbmError(rc, self._L.lbm_group_last_error(None).decode())
        self.nlattice = None

    def _ck(self, rc):
        if rc:
            raise LbmError(rc, self._L.lbm_group_last_error(self._g).decode())

    def close(self):
        if getattr(self, "_g", None) and self._g.value:
            self._L.lbm_group_destroy(self._g)
            self._g = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def size(self) -> int:
        return self._L.lbm_group_size(self._g)

    def setup(self, flag=None, bc_planes=None) -> int:
        n = C.c_int64()
        f = None if flag is None else np.ascontiguousarray(flag, dtype=np.int32)
        a = b = None
        if bc_planes is not None:
            a = np.ascontiguousarray(bc_planes[0], dtype=np.float32)
            b = np.ascontiguousarray(bc_planes[1], dtype=np.float32)
        self._ck(self._L.lbm_group_setup(self._g, None if f is None else f.ctypes.data, None if a is None else a.ctypes.data,
                                         None if b is None else b.ctypes.data, C.byref(n)))
        self.nlattice = n.value
        return n.value

    def step(self, n: int = 1) -> float:
        ms = C.c_float()
        self._ck(self._L.lbm_group_step(self._g, int(n), C.byref(ms)))
        return ms.value

    @property
    def num_fluid(self) -> int:
        return self._L.lbm_group_num_fluid(self._g)

    def residual(self, kind: int = RES_VELSUM) -> float:
        v = C.c_double()
        self._ck(self._L.lbm_group_residual(self._g, kind, C.byref(v)))
        return v.value

    def get_fields(self):
        out = [np.empty(self.nlattice, dtype=self.dtype) for _ in range(4)]
        self._ck(self._L.lbm_group_get_fields(self._g, *[o.ctypes.data for o in out]))
        return out

    def get_index(self) -> np.ndarray:
        g = np.empty((self.desc.nz, self.desc.ny, self.desc.nx), dtype=np.int32)
        self._ck(self._L.lbm_group_get_index(self._g, g.ctypes.data))
        return g

    def set_output_format(self, fmt: int):
        self._ck(self._L.lbm_group_set_output_format(self._g, fmt))

    def set_collision(self, model: int, magic: float = 3 / 16):
        """Case.set_collision on every slab"""
        self._ck(self._L.lbm_group_set_collision(self._g, int(model), float(magic)))

    def outputSave(self, t: int):
        self._ck(self._L.lbm_group_output_save(self._g, int(t)))

    def run_fixed(self, repeat: int, time_save: int, write_files: bool = True):
        self._ck(self._L.lbm_group_run_fixed(self._g, repeat, time_save, int(write_files)))

    def run_converge(self, max_it=10000, tol=1e-6, stag_max=50, time_save=500, write_files=True):
        its, res = C.c_int32(), C.c_double()
        self._ck(self._L.lbm_group_run_converge(self._g, max_it, tol, stag_max, time_save, int(write_files), C.byref(its), C.byref(res)))
        return its.value, res.value


_opened_ipc = {}  # handle bytes -> [mapped pointer, reference count]


def p2p_open(handle_bytes: bytes) -> int:
    """map an allocation exported by another process (cudaIpcOpenMemHandle); an allocation can be
    opened only once per process, so mappings are cached by handle and reference-counted"""
    ent = _opened_ipc.get(handle_bytes)
    if ent is not None:
        ent[1] += 1
        return ent[0]
    L = load_library()
    buf = (C.c_ubyte * 64).from_buffer_copy(handle_bytes)
    ptr = C.c_void_p()
    rc = L.lbm_p2p_open(buf, C.byref(ptr))
    if rc:
        raise LbmError(rc, L.lbm_last_error(None).decode())
    _opened_ipc[handle_bytes] = [ptr.value, 1]
    return ptr.value


def p2p_release(handle_bytes: bytes):
    """drop one reference; the mapping is closed (cudaIpcCloseMemHandle) with the last one.  The
    exporting process must not free the allocation before every importer has released it."""
    ent = _opened_ipc.get(handle_bytes)
    if ent is None:
        return
    ent[1] -= 1
    if ent[1] <= 0:
        del _opened_ipc[handle_bytes]
        load_library().lbm_p2p_close(C.c_void_p(ent[0]))


def voxelize(surface, origin, spacing: float, dims, z_range=None, device: int = 0) -> np.ndarray:
    """STL file (path) or triangle array [n][3][3] -> uint8 mask [z1-z0][ny][nx] (1 inside), the binary
    voxel field geo.txt holds; dims = (nx, ny, nz).  Runs on the GPU (csrc/lbm_voxel.cu)."""
    L = load_library()
    g = VoxelGrid()
    g.origin[:] = [float(v) for v in origin]
    g.spacing = float(spacing)
    g.nx, g.ny, g.nz = (int(v) for v in dims)
    z0, z1 = (0, g.nz) if z_range is None else (int(z_range[0]), int(z_range[1]))
    out = np.zeros((max(z1 - z0, 0), g.ny, g.nx), dtype=np.uint8)
    if isinstance(surface, (str, os.PathLike)):
        rc = L.lbm_voxelize_stl(os.fsencode(str(surface)), C.byref(g), z0, z1, device, out.ctypes.data)
    else:
        tri = np.ascontiguousarray(surface, dtype=np.float32).reshape(-1, 9)
        rc = L.lbm_voxelize_triangles(tri.ctypes.data, tri.shape[0], C.byref(g), z0, z1, device, out.ctypes.data)
    if rc:
        raise LbmError(rc, L.lbm_voxel_last_error().decode())
    return out


def make_case(case_rule: int, *, n=None, dims=None, precision=F32, math_mode=MATH_FAST, storage=STORE_DENSE_AB,
              tau=None, device=0, z_range=None, **paths) -> Case:
    """Reference defaults for `case_rule`, optionally resized (cube `n` or `dims=(nx,ny,nz)`)."""
    d = case_defaults(case_rule)
    if n is not None:
        dims = (n, n, n)
    if dims is not None:
        d.nx, d.ny, d.nz = dims
        d.z_begin, d.z_end = 0, d.nz
    if z_range is not None:
        d.z_begin, d.z_end = z_range
    d.precision, d.math, d.storage, d.device = precision, math_mode, storage, device
    if tau is not None:
        d.tau = tau
    for k, v in paths.items():
        setattr(d, k, os.fsencode(str(v)))
    return Case(d)
