"""GPU: the two-relaxation-time (TRT) collision (lbm_set_collision, csrc/lattice.cuh collide_trt).

- FAST TRT against the CPU oracle stepped with the literal TRT collision and boundary rule (trt_reference.c),
  at the tolerances of the FAST BGK kernels;
- with magic = (tau - 1/2)^2 both rates are 1/tau: every storage must reproduce its own BGK run;
- storages, persistent launches, virtual slabs and a two-slab group agree bit for bit, as under BGK;
- checkpoints carry the operator; the refusals of lbm_set_collision leave the handle stepping as before;
- physics: in a straight duct, the normalised velocity profile no longer depends on tau."""
import numpy as np
import pytest

import helpers as H
import trt_reference as TRT

pytestmark = pytest.mark.gpu

MAGIC = 3 / 16


def L():
    import lattice_boltzmann_method_gpu_b200 as lib

    return lib


def tau_of(name):
    return H.TAU_POS if name == "pos" else H.TAU_LDC


def trt_case(name, n, prec, storage=None, magic=MAGIC, **kw):
    lib = L()
    c = H.gpu_case(name, n, prec, lib.MATH_FAST, storage=storage, **kw)
    c.set_collision(lib.COLL_TRT, magic)
    H.gpu_setup(c, name)
    return c


@pytest.mark.parametrize("name,n", [("ldc", 32), ("pos", 24), ("bif", None), ("cor", None)])
@pytest.mark.parametrize("prec,tol,steps,magic", [("f32", 1e-5, 100, MAGIC), ("f64", 1e-12, 400, MAGIC), ("f64", 1e-12, 400, 0.25)])
def test_fast_trt_matches_trt_oracle(name, n, prec, tol, steps, magic):
    lib = L()
    dt = np.float32 if prec == "f32" else np.float64
    p = lib.F32 if prec == "f32" else lib.F64
    o, *_ = H.trt_oracle_case(name, n, dt)
    c = H.gpu_case(name, n, p, lib.MATH_FAST)
    c.set_collision(lib.COLL_TRT, magic)
    H.trt_gpu_setup(c, name)
    TRT.step(o, steps, magic)
    c.step(steps)
    err = H.rel_err(c.get_fields(), o.fields())
    assert err <= tol, f"{name} {prec} magic {magic}: rel err {err:.3e} > {tol}"
    # the operator is not BGK: the same run under BGK is far from the TRT reference
    b = H.gpu_case(name, n, p, lib.MATH_FAST)
    H.trt_gpu_setup(b, name)
    b.step(steps)
    assert H.rel_err(b.get_fields(), o.fields()) > 100 * tol


@pytest.mark.parametrize("name,n", [("ldc", 24), ("bif", None)])
@pytest.mark.parametrize("storage_name", ["dense_ab", "dense_aa", "sparse_ab", "sparse_aa"])
def test_trt_with_equal_rates_reduces_to_bgk(name, n, storage_name):
    lib = L()
    storage = {"dense_ab": lib.STORE_DENSE_AB, "dense_aa": lib.STORE_DENSE_AA, "sparse_ab": lib.STORE_SPARSE_AB,
               "sparse_aa": lib.STORE_SPARSE_AA}[storage_name]
    b = H.gpu_case(name, n, lib.F64, lib.MATH_FAST, storage=storage)
    H.gpu_setup(b, name)
    t = trt_case(name, n, lib.F64, storage, magic=(float(tau_of(name)) - 0.5) ** 2)
    b.step(400)
    t.step(400)
    assert H.rel_err(t.get_fields(), b.get_fields()) <= 1e-12


@pytest.mark.parametrize("name,n", [("ldc", 24), ("pos", 24), ("bif", None), ("cor", None)])
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_trt_storages_agree_bitwise(name, n, prec):
    lib = L()
    p = lib.F32 if prec == "f32" else lib.F64
    cs = [trt_case(name, n, p, s) for s in (lib.STORE_DENSE_AB, lib.STORE_DENSE_AA, lib.STORE_SPARSE_AB, lib.STORE_SPARSE_AA)]
    for steps in (1, 2, 20):  # odd and even totals
        for c in cs:
            c.step(steps)
        ref = cs[0].get_fields()
        for c in cs[1:]:
            for a, b in zip(ref, c.get_fields()):
                assert np.array_equal(a, b), (name, prec, c.desc.storage, cs[0].step_count)


@pytest.mark.parametrize("name,n", [("ldc", 24), ("bif", None), ("corstep", None)])
def test_trt_persistent_launches_equal_single_launches(name, n):
    lib = L()
    runs = []
    for persistent in (1, 0):
        c = trt_case(name, n, lib.F64, lib.STORE_SPARSE_AA, pulse=(0.3, 40.0) if name == "bif" else None)
        c.set_option("persistent", persistent)
        for nsteps in (1, 2, 7, 64, 131):
            c.step(nsteps)
        runs.append(c.get_fields())
    for a, b in zip(*runs):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("name,n,P", [("ldc", 24, 3), ("bif", None, 4), ("cor", None, 3)])
@pytest.mark.parametrize("mail", [False, True])
def test_trt_virtual_slabs_equal_single_domain_bitwise(name, n, P, mail):
    lib = L()
    one = trt_case(name, n, lib.F64, lib.STORE_DENSE_AA)
    cs = H.virtual_slabs(name, n, P)
    for c in cs:
        c.set_collision(lib.COLL_TRT, MAGIC)
    H.attach_virtual_slabs(cs, mail=mail)
    for steps in (1, 1, 19):  # totals 1, 2, 21
        one.step(steps)
        H.step_virtual_slabs(cs, steps)
        ref = one.get_fields()
        for k in range(4):
            assert np.array_equal(np.concatenate([c.get_fields()[k] for c in cs]), ref[k]), (name, k, one.step_count)


@pytest.mark.parametrize("storage_name", ["dense_aa", "sparse_aa"])
def test_trt_group_equals_single_domain_bitwise(storage_name):
    lib = L()
    storage = lib.STORE_DENSE_AA if storage_name == "dense_aa" else lib.STORE_SPARSE_AA
    one = trt_case("bif", None, lib.F64, storage)
    c = H.gpu_case("bif", None, lib.F64, lib.MATH_FAST, storage=storage)
    d = c.desc
    c.close()
    g = lib.Group(d, 2, [0, 0])
    g.setup(flag=H.bif_flag(), bc_planes=H.bif_bc_planes())
    g.set_collision(lib.COLL_TRT, MAGIC)
    for steps in (1, 2, 20):
        one.step(steps)
        g.step(steps)
        for a, b in zip(one.get_fields(), g.get_fields()):
            assert np.array_equal(a, b), (storage_name, steps)
    with pytest.raises(lib.LbmError):
        g.set_collision(lib.COLL_TRT, -1.0)
    g.close()


@pytest.mark.parametrize("at", [7, 10])
def test_trt_restart_continues_bitwise_and_checkpoints_carry_the_operator(at, tmp_path):
    lib = L()
    pulse = (0.3, 40.0)
    a = trt_case("bif", None, lib.F64, lib.STORE_DENSE_AA, pulse=pulse)
    a.step(at)
    a.checkpoint_save(tmp_path / "trt.bin")
    a.step(13)
    ref = a.get_fields()
    b = trt_case("bif", None, lib.F64, lib.STORE_DENSE_AA, pulse=pulse)
    b.step(3)
    b.checkpoint_load(tmp_path / "trt.bin")
    assert b.step_count == at
    b.step(13)
    for x, y in zip(ref, b.get_fields()):
        assert np.array_equal(x, y)
    # a BGK handle and a TRT handle with another magic parameter refuse the TRT checkpoint
    bgk = H.gpu_case("bif", None, lib.F64, lib.MATH_FAST, pulse=pulse, storage=lib.STORE_DENSE_AA)
    H.gpu_setup(bgk, "bif")
    with pytest.raises(lib.LbmError):
        bgk.checkpoint_load(tmp_path / "trt.bin")
    other = trt_case("bif", None, lib.F64, lib.STORE_DENSE_AA, magic=0.25, pulse=pulse)
    with pytest.raises(lib.LbmError):
        other.checkpoint_load(tmp_path / "trt.bin")
    # a BGK checkpoint still loads into a BGK handle, and not into a TRT one
    bgk.step(4)
    bgk.checkpoint_save(tmp_path / "bgk.bin")
    bgk2 = H.gpu_case("bif", None, lib.F64, lib.MATH_FAST, pulse=pulse, storage=lib.STORE_DENSE_AA)
    H.gpu_setup(bgk2, "bif")
    bgk2.checkpoint_load(tmp_path / "bgk.bin")
    with pytest.raises(lib.LbmError):
        other.checkpoint_load(tmp_path / "bgk.bin")


def test_set_collision_refusals_leave_the_handle_stepping_as_bgk():
    lib = L()
    ref = H.gpu_case("bif", None, lib.F64, lib.MATH_FAST)
    H.gpu_setup(ref, "bif")
    ref.step(30)
    c = H.gpu_case("bif", None, lib.F64, lib.MATH_FAST)
    for model, magic in ((2, MAGIC), (-1, MAGIC), (lib.COLL_TRT, 0.0), (lib.COLL_TRT, -0.1), (lib.COLL_TRT, float("nan")),
                         (lib.COLL_TRT, float("inf"))):
        with pytest.raises(lib.LbmError) as e:
            c.set_collision(model, magic)
        assert e.value.status == -1  # LBM_ERR_ARG
    H.gpu_setup(c, "bif")
    c.step(10)
    c.step_begin(0)
    with pytest.raises(lib.LbmError) as e:  # not between lbm_step_begin and lbm_step_end
        c.set_collision(lib.COLL_TRT, MAGIC)
    assert e.value.status == -2  # LBM_ERR_STATE
    c.step_interior()
    c.step_end()
    c.step(19)
    for a, b in zip(ref.get_fields(), c.get_fields()):
        assert np.array_equal(a, b)
    # STRICT arithmetic has no TRT
    s = H.gpu_case("bif", None, lib.F64, lib.MATH_STRICT)
    with pytest.raises(lib.LbmError) as e:
        s.set_collision(lib.COLL_TRT, MAGIC)
    assert e.value.status == -1
    s.set_collision(lib.COLL_BGK, 0.0)  # BGK ignores the magic parameter
    # switching back to BGK restores the BGK step
    t = H.gpu_case("bif", None, lib.F64, lib.MATH_FAST)
    t.set_collision(lib.COLL_TRT, MAGIC)
    t.set_collision(lib.COLL_BGK, MAGIC)
    H.gpu_setup(t, "bif")
    t.step(30)
    for a, b in zip(ref.get_fields(), t.get_fields()):
        assert np.array_equal(a, b)


# ---------------------------------------------------------------- physics: the wall does not move with tau
DUCT_W, DUCT_LEN, U_IN = 16, 48, 1e-4


def duct_profile(tau, model):
    """normalised steady u_y over the 16 x 16 fluid cross-section at mid-length of a straight square duct along y
    (GEO_Y_INOUT rules: uniform velocity inlet at y = 1, pressure outlet at y = ny - 2), fp64"""
    lib = L()
    m = 3  # ghost plane + wall ring around the fluid section
    nx = nz = DUCT_W + 2 * m
    ny = DUCT_LEN + 4
    flag = np.zeros((nz, ny, nx), dtype=np.int32)
    flag[m - 1:nz - m + 1, :, m - 1:nx - m + 1] = 1  # fluid section + one ring of wall voxels
    d = lib.case_defaults(lib.CASE_GEO_Y_INOUT)
    d.nx, d.ny, d.nz = nx, ny, nz
    d.z_begin, d.z_end = 0, nz
    d.precision, d.math, d.storage, d.tau = lib.F64, lib.MATH_FAST, lib.STORE_DENSE_AB, tau
    c = lib.Case(d)
    c.set_collision(model, MAGIC)
    c.set_flag(flag)
    c.geo_pre()
    c.index_transform()
    geo = c.get_geo()
    inlet = np.where(geo[:, 1, :] == 2, U_IN, 0.0).astype(np.float32)
    assert int((geo[:, 1, :] == 2).sum()) == DUCT_W * DUCT_W
    c.set_bc_planes(inlet, np.zeros_like(inlet))
    c.initialize()
    idx = c.get_index()
    y = ny // 2
    sec = idx[m:nz - m, y, m:nx - m]
    assert (geo[m:nz - m, y, m:nx - m] == 4).all()
    prev = None
    # steady state: the viscous time of the section is W^2 / nu, nu = (tau - 1/2) / 3
    chunk = int(2 * DUCT_W ** 2 / ((tau - 0.5) / 3.0)) // 10 * 2 + 2
    for _ in range(200):
        c.step(chunk)
        uy = c.get_fields()[2][sec]
        prof = uy / uy.mean()
        if prev is not None and np.abs(prof - prev).max() < 1e-9:
            return prof
        prev = prof
    raise AssertionError(f"tau {tau}: no steady state")


def test_trt_wall_does_not_move_with_tau():
    """Spread (largest pairwise max difference) of the normalised mid-length profiles over tau = 0.55, 0.8, 1.4.
    Measured on a B200: TRT (magic 3/16) 5.95e-6, BGK 5.44e-2 -- a factor of 9000.  Thresholds: 5x margin each."""
    lib = L()
    spread = {}
    for model in (lib.COLL_TRT, lib.COLL_BGK):
        profs = [duct_profile(tau, model) for tau in (0.55, 0.8, 1.4)]
        spread[model] = max(float(np.abs(a - b).max()) for i, a in enumerate(profs) for b in profs[i + 1:])
    print(f"profile spread over tau: TRT {spread[lib.COLL_TRT]:.3e}  BGK {spread[lib.COLL_BGK]:.3e}")
    assert spread[lib.COLL_TRT] <= TRT_SPREAD_MAX
    assert spread[lib.COLL_BGK] >= BGK_SPREAD_MIN
    assert spread[lib.COLL_BGK] >= 100 * spread[lib.COLL_TRT]


TRT_SPREAD_MAX = 3e-5
BGK_SPREAD_MIN = 1e-2
