"""Shared builders for the parity tests: the same case set up on the CPU oracle and (on a GPU
box) on the CUDA library through its C ABI."""
from __future__ import annotations

from pathlib import Path

import numpy as np

from oracle import oracle as O

GOLDEN = Path(__file__).resolve().parent / "golden"

LDC_UMAX = float(np.float32(0.15) / np.float32(2.4705))          # ldc.cu:52
POS_UMAX = float(np.float32(0.15) / np.float32(1.5441))          # pos.cu:44 (initialize)
POS_UBC = float(np.float32(0.09714700668))                       # pos.cu:590 (boundary kernel literal)
TAU_LDC = float(np.float32(0.55))
TAU_POS = float(np.float32(0.58))


def bif_flag():
    bits = np.load(GOLDEN / "bif_flag_bits.npy")
    return np.unpackbits(bits)[: 64 * 83 * 32].astype(np.int32).reshape(32, 83, 64)


def bif_bc_planes(shipped_order=False):
    """(inlet, outlet) raw planes.  The shipped bc.txt holds the inlet profile in its SECOND plane
    (so code + data as shipped give a zero inlet, SURVEY 8a5); the default fixture moves it first."""
    bc = np.load(GOLDEN / "bif_bc.npy")
    return (bc[0], bc[1]) if shipped_order else (bc[1], bc[2])


def synthetic_openings_mask(nx=40, ny=36, nz=44):
    """A small vessel for the GEO_OPENINGS (coronary) rule: a tube along +x cut at x=3 (inlet) and
    x=nx-5 (main outlet), with a side branch rising in +z that is cut at z=ztop (sub-exit)."""
    z, y, x = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    cy, cz, r = ny / 2 - 0.5, nz / 3.0, 6.3
    x1, ztop = nx - 5, nz - 6
    tube = ((y - cy) ** 2 + (z - cz) ** 2 <= r * r) & (x >= 3) & (x <= x1)
    bx, rb = nx / 2.0, 4.4
    branch = ((x - bx) ** 2 + (y - cy) ** 2 <= rb * rb) & (z >= cz) & (z <= ztop)
    flag = (tube | branch).astype(np.int32)
    rules = np.array(
        [
            [0, 3, 1, ny - 2, 1, nz - 2, 1],
            [0, x1, 1, ny - 2, 1, nz - 2, 2],
            [2, ztop, int(bx - 8), int(bx + 8), int(cy - 8), int(cy + 8), 4],
        ],
        dtype=np.int32,
    )
    return flag, rules


def stepped_duct_mask(nx=40, ny=24, nz=28):
    """GEO_OPENINGS mask in which a boundary node has fluid on a TANGENTIAL side: a rectangular duct along x
    whose ceiling steps up at x = 20; the sub-exit rule labels the low ceiling (z = 14, x <= 19) 5, so the
    fluid node (20, y, 14) pulls direction (+1,0,0) from the label-5 node (19, y, 14) -- a static link whose
    source was initialised with a nonzero velocity (cor.cu:302-306)."""
    z, y, x = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    ztop = np.where(x < 20, 14, 20)
    flag = ((x >= 3) & (x <= nx - 4) & (y >= 4) & (y <= ny - 5) & (z >= 4) & (z <= ztop)).astype(np.int32)
    rules = np.array([[0, 3, 1, ny - 2, 1, nz - 2, 1], [0, nx - 4, 1, ny - 2, 1, nz - 2, 2], [2, 14, 6, 19, 6, ny - 7, 4]],
                     dtype=np.int32)
    return flag, rules


def coronary_like_flag():
    """A binary voxel field for the UNMODIFIED coronary.cu: its box (291 x 291 x 372, cor:18) and the five
    opening planes it hard-codes (cor:77-141) -- inlet x = 3, main outlet x = 272, sub-exits capped at
    z = 185 inside x[217,236] y[113,137], at z = 191 inside x[160,205] y[159,199], and at z = 204.  A main
    tube along x with three branches rising in +z, each ending exactly on its plane and inside its window.
    Deterministic formula, no RNG (SURVEY 8d)."""
    nx, ny, nz = 291, 291, 372
    z, y, x = np.meshgrid(np.arange(nz, dtype=np.float32), np.arange(ny, dtype=np.float32),
                          np.arange(nx, dtype=np.float32), indexing="ij", sparse=True)
    zc = 100.0
    main = ((y - 150.0) ** 2 + (z - zc) ** 2 <= 16.0 ** 2) & (x >= 3) & (x <= 272)
    b1 = ((x - 226.5) ** 2 + (y - 128.0) ** 2 <= 8.0 ** 2) & (z >= zc) & (z <= 185)
    b2 = ((x - 182.0) ** 2 + (y - 170.0) ** 2 <= 9.0 ** 2) & (z >= zc) & (z <= 191)
    b3 = ((x - 100.0) ** 2 + (y - 150.0) ** 2 <= 10.0 ** 2) & (z >= zc) & (z <= 204)
    return (main | b1 | b2 | b3).astype(np.int32)


def write_geo_txt(path, flag, yfast=False):
    """geo.txt as the reference reads it: "%d " tokens, x fastest (bif:50-61) or y fastest (cor:45-56)"""
    a = np.ascontiguousarray(flag.transpose(0, 2, 1) if yfast else flag).astype(np.uint8).ravel()
    out = np.empty((a.size, 2), dtype=np.uint8)
    out[:, 0] = a + ord("0")
    out[:, 1] = ord(" ")
    out.tofile(str(path))


def openings_mask(name):
    return stepped_duct_mask() if name == "corstep" else synthetic_openings_mask()


# the reference's own lattice speeds (cor.cu:302-306): 0.1745, 0.1, 0.02 m/s over C_U = 2.74909
COR_SPEEDS = dict(uin=float(np.float32(0.1745) / np.float32(2.74909090909091)),
                  uout=float(np.float32(0.1) / np.float32(2.74909090909091)),
                  usub=float(np.float32(0.02) / np.float32(2.74909090909091)))


def oracle_case(name, n=None, dtype=np.float32, pulse=None, shipped_bc=False):
    """Returns (Oracle, geo, index, nlat)."""
    if name == "ldc":
        geo = O.geo_pre_ldc(n, n, n)
        idx, nlat = O.index_dense(geo.shape)
        o = O.Oracle(O.CASE_LDC, geo, idx, nlat, TAU_LDC, LDC_UMAX, dtype=dtype)
    elif name == "pos":
        geo = O.geo_pre_pos(n, n, n)
        idx, nlat = O.index_transform(geo)
        o = O.Oracle(O.CASE_POS, geo, idx, nlat, TAU_POS, POS_UMAX, dtype=dtype)
        o.set_u_bc(POS_UBC)
    elif name == "bif":
        geo = O.geo_pre_bif(bif_flag())
        idx, nlat = O.index_transform(geo)
        o = O.Oracle(O.CASE_BIF, geo, idx, nlat, TAU_LDC, 0.0, dtype=dtype)
        inl, out = bif_bc_planes(shipped_bc)
        nz, ny, nx = geo.shape
        inl = np.where(geo[:, 1, :] == 2, inl, 0).astype(np.float32)
        out = np.where(geo[:, ny - 2, :] == 3, out, 0).astype(np.float32)
        o.set_bc_planes(inl, out)
        if pulse:
            o.set_pulse(*pulse)
    elif name in ("cor", "corstep"):
        flag, rules = openings_mask(name)
        geo = O.geo_pre_cor(flag, rules)
        idx, nlat = O.index_transform(geo)
        o = O.Oracle(O.CASE_COR, geo, idx, nlat, TAU_LDC, 0.0, dtype=dtype)
        o.set_cor_speeds(COR_SPEEDS["uin"], COR_SPEEDS["uout"], COR_SPEEDS["usub"])
        if pulse:
            o.set_pulse(*pulse)
    else:
        raise ValueError(name)
    o.initialize()
    return o, geo, idx, nlat


def gpu_case(name, n=None, precision=None, math_mode=None, pulse=None, shipped_bc=False, z_range=None,
             storage=None, out_dir=None):
    """The same case on the CUDA library, driven through the reference-named call sequence."""
    import lattice_boltzmann_method_gpu_b200 as L

    precision = L.F32 if precision is None else precision
    math_mode = L.MATH_FAST if math_mode is None else math_mode
    storage = L.STORE_DENSE_AB if storage is None else storage
    if name == "ldc":
        d = L.case_defaults(L.CASE_LDC)
        d.nx = d.ny = d.nz = n
    elif name == "pos":
        d = L.case_defaults(L.CASE_POISEUILLE)
        d.nx = d.ny = d.nz = n
    elif name == "bif":
        d = L.case_defaults(L.CASE_GEO_Y_INOUT)
    elif name in ("cor", "corstep"):
        flag, rules = openings_mask(name)
        d = L.case_defaults(L.CASE_GEO_OPENINGS)
        d.nz, d.ny, d.nx = flag.shape
        d.n_openings = len(rules)
        for i, r in enumerate(rules):
            o = d.openings[i]
            o.axis, o.coord, o.lo_a, o.hi_a, o.lo_b, o.hi_b, o.reps = (int(v) for v in r)
        vals = {2: COR_SPEEDS["uin"], 3: COR_SPEEDS["uout"], 5: COR_SPEEDS["usub"], 6: COR_SPEEDS["usub"],
                7: COR_SPEEDS["usub"]}
        for i in range(d.n_bc):
            d.bc[i].value = d.bc[i].init_value = vals[d.bc[i].label]
    else:
        raise ValueError(name)
    d.z_begin, d.z_end = (0, d.nz) if z_range is None else z_range
    d.precision, d.math, d.storage = precision, math_mode, storage
    if out_dir is not None:
        d.out_dir = str(out_dir).encode()
    if pulse:
        d.pulse_amp, d.pulse_period = pulse
        for i in range(d.n_bc):
            if d.bc[i].label == 2:
                d.bc[i].pulsatile = 1
    c = L.Case(d)
    if name == "bif":
        c.set_flag(bif_flag())
    if name in ("cor", "corstep"):
        c.set_flag(openings_mask(name)[0])
    return c


def gpu_setup(c, name, shipped_bc=False):
    """geo_pre -> index_transform -> read_vel -> initialize, like the reference's main()."""
    c.geo_pre()
    nlat = c.index_transform()
    if name == "bif":
        c.set_bc_planes(*bif_bc_planes(shipped_bc))
    c.initialize()
    return nlat


# TRT parity runs bif with its inlet speeds halved (max 0.10): at the fixture's 0.21 (Mach 0.36) and tau = 0.55 the
# TRT run diverges after ~150 steps, in the CPU reference as well -- a stability limit of that flow, not a difference
BIF_TRT_INLET_SCALE = 0.5


def trt_gpu_setup(c, name):
    """gpu_setup, with the inlet of trt_oracle_case"""
    if name != "bif":
        return gpu_setup(c, name)
    c.geo_pre()
    nlat = c.index_transform()
    inl, out = bif_bc_planes()
    c.set_bc_planes((inl * BIF_TRT_INLET_SCALE).astype(np.float32), out)
    c.initialize()
    return nlat


def trt_oracle_case(name, n, dtype):
    """oracle_case for the TRT parity runs (bif with the halved inlet); step it with trt_reference.step"""
    o, geo, idx, nlat = oracle_case(name, n, dtype)
    if name == "bif":
        inl, out = bif_bc_planes()
        ny = geo.shape[1]
        o.set_bc_planes(np.where(geo[:, 1, :] == 2, inl * BIF_TRT_INLET_SCALE, 0).astype(np.float32),
                        np.where(geo[:, ny - 2, :] == 3, out, 0).astype(np.float32))
        o.initialize()
    return o, geo, idx, nlat


def rel_err(got, ref):
    """max |got-ref| over rho,ux,uy,uz, velocity components relative to max|u|, rho relative to 1"""
    scale = max(float(np.abs(r).max()) for r in ref[1:])
    scale = scale if scale > 0 else 1.0
    e_u = max(float(np.abs(g.astype(np.float64) - r.astype(np.float64)).max()) for g, r in zip(got[1:], ref[1:]))
    e_r = float(np.abs(got[0].astype(np.float64) - ref[0].astype(np.float64)).max())
    return max(e_u / scale, e_r)


def virtual_slabs(name, n, P):
    """P dense in-place slab handles of one case on ONE GPU, initialised, numbered like the single domain"""
    import lattice_boltzmann_method_gpu_b200 as L
    from lattice_boltzmann_method_gpu_b200 import slab

    nz = {"ldc": n, "pos": n, "bif": 32, "cor": 44, "corstep": 28}[name]
    cs = [gpu_case(name, n, L.F64, L.MATH_FAST, z_range=r, storage=L.STORE_DENSE_AA) for r in slab.slab_ranges(nz, P)]
    for c in cs:
        c.geo_pre()
    offs, total = slab.compact_offsets([c.local_stored_count() for c in cs])
    for c, o in zip(cs, offs):
        c.set_compact_offset(o, total)
        c.index_transform()
        if name == "bif":
            c.set_bc_planes(*bif_bc_planes())
        c.initialize()
    return cs


def attach_virtual_slabs(cs, mail=False):
    """several slab handles on ONE GPU: every handle stores its crossing populations straight into its
    neighbours' buffers (lbm_p2p_attach with plain device pointers) or, mail=True, into their mailboxes
    (lbm_mail_export / lbm_mail_attach, dense in-place storage)"""
    if mail:
        boxes = [{s: c.mail_export(s)["ptr"] for s, nb in ((0, r - 1), (1, r + 1)) if 0 <= nb < len(cs)} for r, c in enumerate(cs)]
        for r, c in enumerate(cs):
            for side, nb in ((0, r - 1), (1, r + 1)):
                if 0 <= nb < len(cs):
                    c.mail_attach(side, boxes[nb][1 - side])
        return
    exp = [c.p2p_export() for c in cs]
    for r, c in enumerate(cs):
        for side, nb in ((0, r - 1), (1, r + 1)):
            if 0 <= nb < len(cs):
                e = exp[nb]
                c.p2p_attach(side, e["ptrs"][0], e["ptrs"][1], e["qs"], e["halo_c0"][1 - side], e["face_c0"][1 - side])


def step_virtual_slabs(cs, steps):
    """lock-step stepping of attached virtual slabs; moments are materialised on the last step"""
    import lattice_boltzmann_method_gpu_b200 as L

    for it in range(steps):
        for c in cs:
            c.step_begin(L.STEP_MOMENTS if it == steps - 1 else 0)
            c.step_interior()
            c.step_end()
        for c in cs:
            c.sync()


# ---------------------------------------------------------------- triangle meshes for the voxeliser tests
def mesh_box(lo, hi):
    """12 triangles; every face is split along a diagonal (rays through voxel centres hit those edges)"""
    lo, hi = np.asarray(lo, dtype=np.float32), np.asarray(hi, dtype=np.float32)
    c = np.array([[lo[0] if not (i & 1) else hi[0], lo[1] if not (i & 2) else hi[1], lo[2] if not (i & 4) else hi[2]]
                  for i in range(8)], dtype=np.float32)
    quads = [(0, 2, 6, 4), (1, 5, 7, 3), (0, 4, 5, 1), (2, 3, 7, 6), (0, 1, 3, 2), (4, 6, 7, 5)]
    tris = []
    for a, b, cc, d in quads:
        tris += [[c[a], c[b], c[cc]], [c[a], c[cc], c[d]]]
    return np.array(tris, dtype=np.float32)


def mesh_sphere(center, r, nu=48, nv=24):
    """closed UV sphere"""
    center = np.asarray(center, dtype=np.float64)
    th = np.linspace(0.0, np.pi, nv + 1)
    ph = np.linspace(0.0, 2 * np.pi, nu + 1)
    P = np.array([[center + r * np.array([np.sin(t) * np.cos(p), np.sin(t) * np.sin(p), np.cos(t)]) for p in ph[:-1]]
                  for t in th])
    P[0, :] = center + [0, 0, r]      # exact, shared poles: the fan triangles meet in one vertex
    P[-1, :] = center + [0, 0, -r]
    tris = []
    for i in range(nv):
        for j in range(nu):
            a, b, c, d = P[i, j], P[i, (j + 1) % nu], P[i + 1, (j + 1) % nu], P[i + 1, j]
            if i > 0:
                tris.append([a, b, c])
            if i < nv - 1:
                tris.append([a, c, d])
    return np.array(tris, dtype=np.float32)


def mesh_tube(length, r, bend=0.0, nu=64, nv=80, x0=0.0, z0=0.0):
    """open-ended tube along y (like a vessel segment): centre line x = x0 + bend*sin(pi*y/length)"""
    ys = np.linspace(0.0, length, nv + 1)
    ph = np.linspace(0.0, 2 * np.pi, nu + 1)[:-1]
    P = np.array([[[x0 + bend * np.sin(np.pi * y / length) + r * np.cos(p), y, z0 + r * np.sin(p)] for p in ph] for y in ys])
    tris = []
    for i in range(nv):
        for j in range(nu):
            a, b, c, d = P[i, j], P[i, (j + 1) % nu], P[i + 1, (j + 1) % nu], P[i + 1, j]
            tris += [[a, b, c], [a, c, d]]
    return np.array(tris, dtype=np.float32)


def write_binary_stl(path, tri):
    tri = np.asarray(tri, dtype=np.float32).reshape(-1, 3, 3)
    rec = np.zeros(len(tri), dtype=np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")]))
    rec["v"] = tri
    with open(path, "wb") as f:
        f.write(b"binary stl written by the tests".ljust(80, b" "))
        f.write(np.uint32(len(tri)).tobytes())
        f.write(rec.tobytes())


def write_ascii_stl(path, tri):
    tri = np.asarray(tri, dtype=np.float32).reshape(-1, 3, 3)
    with open(path, "w") as f:
        f.write("solid t\n")
        for t in tri:
            f.write(" facet normal 0 0 0\n  outer loop\n")
            for v in t:
                f.write(f"   vertex {float(v[0])!r} {float(v[1])!r} {float(v[2])!r}\n")
            f.write("  endloop\n endfacet\n")
        f.write("endsolid t\n")
