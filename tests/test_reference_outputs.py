"""Pins against the REAL reference: tests/golden/reference_gpu_outputs.npz holds what the reference
programs themselves (ldc.cu, Poiseulle.cu, bifurcation.cu compiled unmodified into oracle/_ref and
run on a B200 by tools/capture_reference.py) wrote into their final VTK files and CONVERGENCE.log.

CPU test: the oracle reproduces the bifurcation run (4401 steps, fp32).
GPU tests: the CUDA library, driven like the reference's main(), reproduces all three -- same
iteration at which the convergence loop stops, same residual log, same fields -- and writes VTK
files with byte-identical headers.

Tolerance: the reference prints 6 significant digits and its kernels are compiled with FMA
contraction, so fields are compared at 2e-5 of max|v|.  ldc is compared at 1e-3: its `update`
kernel bounces the walls in place while fluid nodes of the same launch read them (ldc.cu:75-313),
so a fluid node sees a mix of this step's and two-steps-old wall values.  The stopping rule ends
the run (k = 5119) while the flow is still 6.4e-2 away from its steady state; at that iteration
the reference's field and the defined semantics ("walls first", what the library implements bit
for bit) differ by 7.6e-4.  tests/test_ldc_order_cpu.py accounts for that number: replaying the order
ldc.cu's launch executes in brings the oracle to 3.4e-5 / 4.7e-5 of the real binary, which lies inside
the envelope of the two order models; tests/test_reference_variants.py compares the library with the
real binary at a true steady state, where the order no longer matters (5e-5, fp32 rounding)."""
import numpy as np
import pytest

import helpers as H

GOLD = np.load(H.GOLDEN / "reference_gpu_outputs.npz")
C_U = {"ldc": np.float32(2.4705), "pos": np.float32(1.5441), "bif": np.float32(0.24159041)}


def vtk_box(name, shape):
    nz, ny, nx = shape
    if name == "ldc":
        return slice(2, nz - 2), slice(2, ny - 2), slice(2, nx - 2)
    return slice(1, nz - 1), slice(2, ny - 2), slice(1, nx - 1)


def vtk_velocity(name, geo_shape, idx, ux, uy, uz):
    """the array outputSave prints: u * C_U on the trimmed box, 0 where nothing is stored"""
    comps = []
    for a in (ux, uy, uz):
        full = np.zeros(geo_shape, np.float32)
        m = idx >= 0
        full[m] = a.astype(np.float32)[idx[m]]
        comps.append((full * C_U[name[:3]])[vtk_box(name[:3], geo_shape)])
    return np.stack(comps, -1)


def compare(name, V, tol, sum_tol=None):
    sum_tol = tol if sum_tol is None else sum_tol
    nz, ny, nx = V.shape[:3]
    assert [nx, ny, nz] == list(GOLD[f"{name}_dims"])
    scale = float(GOLD[f"{name}_max_abs"])
    for key, got in (("plane_z", V[nz // 2]), ("plane_y", V[:, ny // 2]), ("plane_x", V[:, :, nx // 2])):
        ref = GOLD[f"{name}_{key}"]
        err = float(np.abs(ref - got).max()) / scale
        assert err < tol, f"{name} {key}: {err:.2e}"
    s = float(np.sqrt((V.astype(np.float64) ** 2).sum(-1)).sum())
    assert abs(s - float(GOLD[f"{name}_sum_abs"])) / float(GOLD[f"{name}_sum_abs"]) < sum_tol
    comp = V.astype(np.float64).sum(axis=(0, 1, 2))
    assert np.abs(comp - GOLD[f"{name}_sum_comp"]).max() / float(GOLD[f"{name}_sum_abs"]) < sum_tol


def test_oracle_reproduces_reference_bifurcation_run():
    o, geo, idx, _ = H.oracle_case("bif", None, np.float32)
    o.step(int(GOLD["bif_last_iter"]) + 1)  # loop index 0..4400 inclusive (bifurcation.cu:1246)
    rho, ux, uy, uz = o.fields()
    compare("bif", vtk_velocity("bif", geo.shape, idx, ux, uy, uz), 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("math_name", ["strict", "fast"])
def test_gpu_reproduces_reference_bifurcation_run(math_name, tmp_path):
    import lattice_boltzmann_method_gpu_b200 as L

    c = H.gpu_case("bif", None, L.F32, L.MATH_STRICT if math_name == "strict" else L.MATH_FAST)
    c.desc.out_dir = str(tmp_path).encode()
    c.close()
    c = L.Case(c.desc)
    c.set_flag(H.bif_flag())
    H.gpu_setup(c, "bif")
    c.run_fixed(4400, 4400, True)  # REPEAT, time_save of bifurcation.cu:19
    geo, idx = c.get_geo(), c.get_index()
    rho, ux, uy, uz = c.get_fields()
    compare("bif", vtk_velocity("bif", geo.shape, idx, ux, uy, uz), 2e-5)
    # files: bif_0.vtk, bif_4400.vtk, CONVERGENCE.log with the two residuals the reference logged
    for t in (0, 4400):
        lines = (tmp_path / f"bif_{t}.vtk").read_text().split("\n")
        assert lines[:9] == [str(s) for s in GOLD["bif_header"]]
    log = [l for l in (tmp_path / "CONVERGENCE.log").read_text().split("\n") if l and not l.startswith("TOTAL")]
    assert float(log[0]) == 1.0
    assert abs(float(log[1]) - GOLD["bif_residuals"][1]) < 1e-4
    # the written velocity block parses back to the same numbers
    body = np.array((tmp_path / "bif_4400.vtk").read_text().split("\n")[9].split(), dtype=np.float32)
    compare("bif", body.reshape(30, 79, 62, 3), 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("name,rule,tol", [("ldc", 0, 1e-3), ("pos", 1, 2e-5)])
def test_gpu_reproduces_reference_convergence_runs(name, rule, tol, tmp_path):
    """ldc.cu:653-685 / Poiseulle.cu:986-1019: residual every step, stop after 51 hits of 1e-6"""
    import lattice_boltzmann_method_gpu_b200 as L

    d = L.case_defaults(rule)
    d.precision, d.math = L.F32, L.MATH_FAST
    d.out_dir = str(tmp_path).encode()
    c = L.Case(d)
    c.geo_pre()
    c.index_transform()
    c.initialize()
    its, res = c.run_converge(10000, 1e-6, 50, 500, True)
    ref_its = int(GOLD[f"{name}_last_iter"])
    # the stopping iteration depends on a float sum of 262144 speeds; thrust's order differs from ours
    assert abs(its - ref_its) <= max(25, ref_its // 50), (its, ref_its)
    prefix = "lid" if name == "ldc" else "pos"
    vtks = sorted(tmp_path.glob(f"{prefix}_*.vtk"))
    assert len(vtks) in (int(GOLD[f"{name}_n_vtk"]), int(GOLD[f"{name}_n_vtk"]) + 1)
    lines = (tmp_path / f"{prefix}_{its}.vtk").read_text().split("\n")
    assert lines[:9] == [str(s) for s in GOLD[f"{name}_header"]]
    # fields at the iteration the REFERENCE stopped at (the loop above may stop a few iterations earlier or
    # later -- its S is an atomic float sum -- and the flow is still evolving there)
    d.out_dir = str(tmp_path / "unused").encode()
    e = L.Case(d)
    e.geo_pre(), e.index_transform(), e.initialize()
    e.step(ref_its)
    geo, idx = e.get_geo(), e.get_index()
    rho, ux, uy, uz = e.get_fields()
    # ldc: the lag of the in-place wall bounce is systematic, so the field SUMS differ more than any point does
    compare(name, vtk_velocity(name, geo.shape, idx, ux, uy, uz), tol, 3e-3 if name == "ldc" else None)
    log = [float(l) for l in (tmp_path / "CONVERGENCE.log").read_text().split("\n") if l and not l.startswith("TOTAL")]
    ref = GOLD[f"{name}_residuals"]
    n = min(len(log), len(ref)) - 1  # the last save iterations are near the 1e-6 noise floor
    # |S_k - S_{k-1}| / S_k is a difference of two float sums: it follows the reference's log closely while
    # the flow still changes fast, then only in order of magnitude (ldc additionally carries the wall race)
    assert np.allclose(log[:2], ref[:2], rtol=0.1 if name == "ldc" else 2e-2)
    # single-step residuals at the save iterations; noisy once below ~1e-4 (order of magnitude only)
    assert all(abs(np.log10(a) - np.log10(b)) < 1.0 for a, b in zip(log[:n], ref[:n]))

