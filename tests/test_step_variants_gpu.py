"""GPU: the step-kernel instantiations the default parity cases never select, against the CPU oracle.

- SPEC, the speculative pull of k_step_dense.  The host picks it when >= 90 % of the launched cells are fluid
  (speculative_pull() in csrc/lbm_api.cu).  The ldc cavity first qualifies at n = 127 and 128; n = 127 also has a
  padding lane in every row.  Section A runs both at their natural setting.  Section B forces the pull form with
  the LBM_SPECULATIVE knob on the small boundary cases (inlet, outlet and static links, slab faces into peer
  buffers and mailboxes), and off at 128^3.  The knob, like LBM_SPW (records per warp of k_step_sparse), is read
  once per process, so those runs happen in a child process (this file run as a script) that only steps and
  saves fields; every comparison is made here.
- RESID, the fused per-step sum of |u| (Section C): lbm_slab_step(S_out) and the persistent kernel's per-step
  slots of lbm_run_converge, against the same sum formed from the oracle's fields; and the switch must not
  change the populations.

Tolerances are the parity suite's: STRICT bit-exact; FAST 1e-12 (fp64) / 1e-5 (fp32) of max|u|, and FAST fp32 at
128^3 against an fp64 oracle (assert_fast_close)."""
import os
import subprocess
import sys
from pathlib import Path
from typing import NamedTuple

if __name__ == "__main__":  # child mode: the package and the oracle live at the repository root
    sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import numpy as np
import pytest

import helpers as H
import trt_reference as TRT

pytestmark = pytest.mark.gpu

MAGIC = 3 / 16
PRECS = ("f32", "f64")
DENSE = ("dense_ab", "dense_aa")
STORAGES = ("dense_ab", "dense_aa", "sparse_ab", "sparse_aa")
STRICT_TOTALS = (1, 2, 3, 8, 37)  # odd and even totals: both phases of the in-place storages
FAST_TOL = {"f32": 1e-5, "f64": 1e-12}
DT = {"f32": np.float32, "f64": np.float64}


def L():
    import lattice_boltzmann_method_gpu_b200 as lib

    return lib


def fluid_label(name):
    return 3 if name == "ldc" else 4


def speculative_by_rule(c):
    """the host rule of speculative_pull() for a single-domain handle: fluid nodes >= 90 % of the launched cells,
    rows padded to a multiple of 32 cells"""
    assert not os.environ.get("LBM_SPECULATIVE"), "these tests check the pull form the host picks: unset LBM_SPECULATIVE"
    d = c.desc
    return c.num_fluid * 10 >= d.nz * d.ny * ((d.nx + 31) // 32 * 32) * 9


class Run(NamedTuple):
    """one single-domain GPU run; fields after each of `totals` steps"""
    name: str
    n: int
    prec: str
    math: str  # "strict" / "fast"
    storage: str
    coll: str  # "bgk" / "trt"
    totals: tuple

    @property
    def key(self):
        return "-".join(str(v) for v in self[:6])

    def case(self):
        lib = L()
        c = H.gpu_case(self.name, self.n, lib.F32 if self.prec == "f32" else lib.F64,
                       lib.MATH_STRICT if self.math == "strict" else lib.MATH_FAST,
                       storage=getattr(lib, "STORE_" + self.storage.upper()))
        if self.coll == "trt":
            c.set_collision(lib.COLL_TRT, MAGIC)
            H.trt_gpu_setup(c, self.name)
        else:
            H.gpu_setup(c, self.name)
        return c

    def run(self):
        c = self.case()
        out, done = {}, 0
        for t in self.totals:
            c.step(t - done)
            done = t
            out[t] = [a.copy() for a in c.get_fields()]
        c.close()
        return out


class Slabs(NamedTuple):
    """virtual dense in-place slabs of one case on one GPU (FAST fp64 BGK), joined fields after each of `totals`"""
    name: str
    n: int
    P: int
    mail: bool
    totals: tuple

    @property
    def key(self):
        return f"slabs-{self.name}-{self.n}-{self.P}-{'mail' if self.mail else 'buffers'}"

    def run(self):
        cs = H.virtual_slabs(self.name, self.n, self.P)
        H.attach_virtual_slabs(cs, mail=self.mail)
        out, done = {}, 0
        for t in self.totals:
            H.step_virtual_slabs(cs, t - done)
            done = t
            out[t] = [np.concatenate([c.get_fields()[k] for c in cs]) for k in range(4)]
        for c in cs:
            c.close()
        return out


# ---------------------------------------------------------------- the child runs
SMALL = [("ldc", 24), ("ldc", 33), ("pos", 24), ("bif", None), ("cor", None), ("corstep", None)]
FAST_TOTALS = (2, 101)
TRT_STEPS = {"f32": 100, "f64": 400}
SLABS = [("ldc", 24, 3), ("bif", None, 4), ("cor", None, 3)]
SLAB_TOTALS = (1, 2, 21)
SPW_CASES = [("bif", None), ("cor", None), ("ldc", 33)]
BIG_TOTALS = (10, 37)

CHILD_ENV = {"spec1": {"LBM_SPECULATIVE": "1"}, "spec0": {"LBM_SPECULATIVE": "0"}, "spw2": {"LBM_SPW": "2"},
             "spw3": {"LBM_SPW": "3"}}
CHILD_TIMEOUT = 900  # seconds; a few seconds to a minute on a B200


def strict_run(name, n, prec, storage):
    return Run(name, n, prec, "strict", storage, "bgk", STRICT_TOTALS)


def fast_run(name, n, storage):
    return Run(name, n, "f64", "fast", storage, "bgk", FAST_TOTALS)


def trt_run(name, prec, storage):
    return Run(name, None, prec, "fast", storage, "trt", (TRT_STEPS[prec],))


def big_run(storage):
    return Run("ldc", 128, "f64", "fast", storage, "bgk", BIG_TOTALS)


def child_jobs(mode):
    if mode == "spec1":
        for name, n in SMALL:
            for prec in PRECS:
                for st in DENSE:
                    yield strict_run(name, n, prec, st)
            for st in DENSE:
                yield fast_run(name, n, st)
        for name in ("bif", "cor"):
            for prec in PRECS:
                for st in DENSE:
                    yield trt_run(name, prec, st)
        for name, n, P in SLABS:
            for mail in (False, True):
                yield Slabs(name, n, P, mail, SLAB_TOTALS)
    elif mode == "spec0":
        for st in DENSE:
            yield big_run(st)
    else:
        for name, n in SPW_CASES:
            for prec in PRECS:
                yield strict_run(name, n, prec, "sparse_ab")


def child_main(mode, out_dir):
    out_dir = Path(out_dir)
    for job in child_jobs(mode):
        fields = job.run()
        np.savez(out_dir / (job.key + ".npz"), **{f"{t}_{k}": a for t, fs in fields.items() for k, a in enumerate(fs)})


class Child(NamedTuple):
    mode: str
    out_dir: Path
    error: str  # empty when the child exited with status 0


def run_child(mode, out_dir):
    """run this file as a child process with the knob of `mode` set; it has exited when this returns"""
    env = {k: v for k, v in os.environ.items() if k not in ("LBM_SPECULATIVE", "LBM_SPW")}
    env.update(CHILD_ENV[mode], PYTHONDONTWRITEBYTECODE="1")
    cmd = [sys.executable, str(Path(__file__).resolve()), mode, str(out_dir)]
    try:
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=CHILD_TIMEOUT)
    except subprocess.TimeoutExpired as e:  # subprocess.run has killed and reaped the child
        err = e.stderr.decode(errors="replace") if isinstance(e.stderr, bytes) else (e.stderr or "")
        return Child(mode, out_dir, f"timed out after {CHILD_TIMEOUT} s\n{err[-4000:]}")
    return Child(mode, out_dir, "" if r.returncode == 0 else f"exit status {r.returncode}\n{r.stderr[-4000:]}")


@pytest.fixture(scope="module")
def child(tmp_path_factory):
    """child(mode): the output of the child run of `mode`, started on first use"""
    done = {}

    def get(mode):
        if mode not in done:
            done[mode] = run_child(mode, tmp_path_factory.mktemp(mode))
        return done[mode]

    return get


def child_fields(ch, job):
    assert not ch.error, f"child process ({ch.mode}, {' '.join(f'{k}={v}' for k, v in CHILD_ENV[ch.mode].items())}) failed: {ch.error}"
    z = np.load(ch.out_dir / (job.key + ".npz"))
    return {t: [z[f"{t}_{k}"] for k in range(4)] for t in job.totals}


def oracle_fields(name, n, prec, coll, totals):
    """the oracle's (or, coll == "trt", the TRT reference's) fields after each of `totals` steps"""
    o, *_ = (H.trt_oracle_case if coll == "trt" else H.oracle_case)(name, n, DT[prec])
    out, done = {}, 0
    for t in totals:
        if coll == "trt":
            TRT.step(o, t - done, MAGIC)
        else:
            o.step(t - done)
        done = t
        out[t] = o.fields()
    o.close()
    return out


def assert_fast_close(got, ref, truth, prec, what):
    """FAST against the oracle of the same precision, at 128^3: within 1e-12 in fp64.  Two fp32 evaluation orders drift
    apart by fp32's own rounding noise, which in the 127^3 / 128^3 cavity passes 1e-5 of max|u| within 80 - 100 steps
    (2.4e-5 BGK, 1.2e-5 TRT, measured on a B200).  So in fp32 the kernel must be no further from the fp64 oracle
    (`truth`) than the oracle's own fp32 run is, the criterion of test_fast_fp32_is_as_accurate_as_the_reference_order."""
    err = H.rel_err(got, ref)
    if prec == "f64":
        assert err <= FAST_TOL["f64"], f"{what}: rel err {err:.3e} > {FAST_TOL['f64']}"
        return
    e_fast, e_ref = H.rel_err(got, truth), H.rel_err(ref, truth)
    assert e_fast <= 2.0 * e_ref + 1e-7, f"{what}: {e_fast:.3e} from the fp64 oracle, the fp32 oracle {e_ref:.3e} (apart: {err:.3e})"


def assert_bitwise(got, ref, what):
    for nm, g, r in zip(("rho", "ux", "uy", "uz"), got, ref):
        assert np.array_equal(g, r), f"{what}: {nm} differs, max {np.abs(g.astype(np.float64) - r).max():.3e}"


# ---------------------------------------------------------------- A. SPEC at its natural threshold
@pytest.mark.parametrize("n", [127, 128])
@pytest.mark.parametrize("prec", PRECS)
def test_natural_spec_bgk_matches_oracle(n, prec):
    """STRICT bit-exact after 1, 2, 3, 8, 37 steps; FAST within tolerance after 100; both dense storages"""
    o, geo, idx, nlat = H.oracle_case("ldc", n, DT[prec])
    strict = {st: Run("ldc", n, prec, "strict", st, "bgk", ()).case() for st in DENSE}
    fast = {st: Run("ldc", n, prec, "fast", st, "bgk", ()).case() for st in DENSE}
    for c in (*strict.values(), *fast.values()):
        assert c.num_fluid == (n - 4) ** 3
        assert speculative_by_rule(c), f"ldc {n} no longer selects the speculative pull"
    done = 0
    for t in STRICT_TOTALS:
        o.step(t - done)
        ref = o.fields()
        for st, c in strict.items():
            c.step(t - done)
            assert_bitwise(c.get_fields(), ref, f"ldc {n} {prec} STRICT {st} after {t} steps")
        done = t
        if n == 127 and prec == "f64" and t == 37:  # the populations of the in-place storage, once
            from oracle import oracle as O

            fo, fg = o.populations(), strict["dense_aa"].get_populations()
            zz, yy, xx = np.nonzero(geo == 3)
            for q in range(19):
                lab = geo[zz - O.CZ[q], yy - O.CY[q], xx - O.CX[q]]
                src = idx[zz - O.CZ[q], yy - O.CY[q], xx - O.CX[q]][lab != 1]  # wall slots lag one step (test_parity_gpu)
                assert np.array_equal(fo[q, src], fg[q, src]), f"direction {q}"
            del fo, fg
    steps = 100
    o.step(steps - done)
    ref = o.fields()
    truth = oracle_fields("ldc", n, "f64", "bgk", (steps,))[steps] if prec == "f32" else None
    for st, c in fast.items():
        c.step(steps)
        assert_fast_close(c.get_fields(), ref, truth, prec, f"ldc {n} {prec} FAST {st}")
    for c in (*strict.values(), *fast.values()):
        c.close()
    o.close()


@pytest.mark.parametrize("prec", PRECS)
def test_natural_spec_trt_matches_trt_oracle(prec):
    steps = 80
    ref = oracle_fields("ldc", 128, prec, "trt", (steps,))[steps]
    truth = oracle_fields("ldc", 128, "f64", "trt", (steps,))[steps] if prec == "f32" else None
    for st in DENSE:
        c = Run("ldc", 128, prec, "fast", st, "trt", ()).case()
        assert speculative_by_rule(c)
        c.step(steps)
        got = c.get_fields()
        c.close()
        assert_fast_close(got, ref, truth, prec, f"ldc 128 {prec} TRT {st}")


# ---------------------------------------------------------------- B. the forced pull form, in child processes
@pytest.mark.parametrize("name,n", SMALL)
def test_small_cases_do_not_select_spec(name, n):
    """the cases of section B reach the speculative kernels only through LBM_SPECULATIVE=1"""
    c = Run(name, n, "f64", "fast", "dense_ab", "bgk", ()).case()
    assert not speculative_by_rule(c)


@pytest.mark.parametrize("name,n", SMALL)
@pytest.mark.parametrize("prec", PRECS)
def test_forced_spec_strict_matches_oracle(child, name, n, prec):
    ch = child("spec1")
    ref = oracle_fields(name, n, prec, "bgk", STRICT_TOTALS)
    for st in DENSE:
        got = child_fields(ch, strict_run(name, n, prec, st))
        for t in STRICT_TOTALS:
            assert_bitwise(got[t], ref[t], f"{name} {prec} STRICT {st} SPEC after {t} steps")


@pytest.mark.parametrize("name,n", SMALL)
@pytest.mark.parametrize("storage", DENSE)
def test_forced_spec_fast_equals_default_pull(child, name, n, storage):
    """FAST arithmetic gives the same bits whichever form the kernel pulls in (DESIGN section 2)"""
    job = fast_run(name, n, storage)
    got = child_fields(child("spec1"), job)
    ref = job.run()
    for t in FAST_TOTALS:
        assert_bitwise(got[t], ref[t], f"{name} FAST {storage} SPEC after {t} steps")


@pytest.mark.parametrize("name", ["bif", "cor"])
@pytest.mark.parametrize("prec", PRECS)
def test_forced_spec_trt_matches_trt_oracle(child, name, prec):
    ch = child("spec1")
    steps = TRT_STEPS[prec]
    ref = oracle_fields(name, None, prec, "trt", (steps,))[steps]
    for st in DENSE:
        err = H.rel_err(child_fields(ch, trt_run(name, prec, st))[steps], ref)
        assert err <= FAST_TOL[prec], f"{name} {prec} TRT {st} SPEC: rel err {err:.3e} > {FAST_TOL[prec]}"


@pytest.mark.parametrize("name,n,P", SLABS)
@pytest.mark.parametrize("mail", [False, True])
def test_forced_spec_virtual_slabs_equal_single_domain(child, name, n, P, mail):
    """speculative face launches storing into the neighbours' buffers or mailboxes"""
    job = Slabs(name, n, P, mail, SLAB_TOTALS)
    got = child_fields(child("spec1"), job)
    ref = Run(name, n, "f64", "fast", "dense_aa", "bgk", SLAB_TOTALS).run()
    for t in SLAB_TOTALS:
        assert_bitwise(got[t], ref[t], f"{job.key} after {t} steps")


@pytest.mark.parametrize("storage", DENSE)
def test_default_pull_at_128_equals_natural_spec(child, storage):
    job = big_run(storage)
    got = child_fields(child("spec0"), job)
    c = job.case()
    assert speculative_by_rule(c)
    c.close()
    ref = job.run()
    for t in BIG_TOTALS:
        assert_bitwise(got[t], ref[t], f"ldc 128 FAST {storage}: LBM_SPECULATIVE=0 against the natural SPEC run, {t} steps")


@pytest.mark.parametrize("spw", [2, 3])
@pytest.mark.parametrize("name,n", SPW_CASES)
@pytest.mark.parametrize("prec", PRECS)
def test_sparse_records_per_warp_strict_matches_oracle(child, spw, name, n, prec):
    job = strict_run(name, n, prec, "sparse_ab")
    got = child_fields(child(f"spw{spw}"), job)
    ref = oracle_fields(name, n, prec, "bgk", STRICT_TOTALS)
    for t in STRICT_TOTALS:
        assert_bitwise(got[t], ref[t], f"{name} {prec} STRICT sparse_ab, {spw} records per warp, after {t} steps")


# ---------------------------------------------------------------- C. the fused per-step sum of |u|
KINDS = {"strict": ("strict", "bgk"), "fast": ("fast", "bgk"), "trt": ("fast", "trt")}
VELSUM_STEPS = 11


def velsum_tol(prec, kind):
    """STRICT: the terms are the oracle's to the bit, only the order of the double sums differs"""
    return 1e-12 if kind == "strict" else FAST_TOL[prec]


def oracle_velsums(name, n, prec, coll, steps):
    """S_k = sum over fluid nodes of T(sqrt(double(ux^2 + uy^2 + uz^2))) after each step k = 1 .. steps, in the field
    precision T (the expression finish_cell forms), summed in float64"""
    dt = DT[prec]
    o, geo, idx, nlat = (H.trt_oracle_case if coll == "trt" else H.oracle_case)(name, n, dt)
    fl = idx[geo == fluid_label(name)]
    S = []
    for _ in range(steps):
        if coll == "trt":
            TRT.step(o, 1, MAGIC)
        else:
            o.step(1)
        _, ux, uy, uz = (a[fl] for a in o.fields())
        S.append(float(np.sqrt((ux * ux + uy * uy + uz * uz).astype(np.float64)).astype(dt).astype(np.float64).sum()))
    o.close()
    return np.array(S)


def assert_sums_close(S, ref, tol, what):
    rel = np.abs(S - ref) / ref
    k = int(rel.argmax())
    assert rel[k] <= tol, f"{what}: step {k + 1}: S = {S[k]!r}, oracle {ref[k]!r}, rel {rel[k]:.3e} > {tol}"


@pytest.mark.parametrize("name,n", [("bif", None), ("cor", None), ("ldc", 33), ("ldc", 128)])
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("kind", list(KINDS))
def test_fused_velsum_per_step_matches_oracle(name, n, prec, kind):
    """lbm_slab_step(S_out) on a single domain, every storage: S_k against the oracle, and the RESID kernels store
    the populations the plain kernels store -- with moments on the last step, and with MOMENTS off throughout"""
    math, coll = KINDS[kind]
    ref = oracle_velsums(name, n, prec, coll, VELSUM_STEPS)
    tol = velsum_tol(prec, kind)
    for st in STORAGES:
        run = Run(name, n, prec, math, st, coll, ())
        a, b, c = run.case(), run.case(), run.case()
        if n == 128 and st in DENSE:
            assert speculative_by_rule(a)
        _, S = a.slab_step(VELSUM_STEPS, velsum=True)
        assert_sums_close(S, ref, tol, f"{name} {prec} {kind} {st}")
        b.step(VELSUM_STEPS)
        assert_bitwise(a.get_fields(), b.get_fields(), f"{name} {prec} {kind} {st}: RESID against plain steps")
        _, S = c.slab_step(VELSUM_STEPS, moments_last=False, velsum=True)
        assert_sums_close(S, ref, tol, f"{name} {prec} {kind} {st}, no moments")
        c.step(1)
        b.step(1)
        assert_bitwise(c.get_fields(), b.get_fields(), f"{name} {prec} {kind} {st}: RESID without MOMENTS, then a step")
        for h in (a, b, c):
            h.close()


@pytest.mark.parametrize("name,n", [("bif", None), ("ldc", 33)])
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("kind", ["strict", "trt"])
@pytest.mark.parametrize("persistent", [1, 0])
def test_run_converge_residual_from_per_step_sums(name, n, prec, kind, persistent):
    """lbm_run_converge on the sparse in-place storage, with one cooperative launch per batch (persistent = 1, the
    per-step slots of k_sparse_aa_persist) or one launch per step.  With tol = 0 the loop runs iterations
    k = 0 .. max_it, and its residual is the host's float formula |S_K - S_{K-1}| / S_K of the last two sums."""
    K = 40
    math, coll = KINDS[kind]
    ref = oracle_velsums(name, n, prec, coll, K + 1)
    c = Run(name, n, prec, math, "sparse_aa", coll, ()).case()
    c.set_option("persistent", persistent)
    its, res = c.run_converge(max_it=K, tol=0.0, stag_max=K + 10, time_save=10 ** 6, write_files=False)
    c.close()
    assert its == K + 1
    a, b = np.float32(ref[K]), np.float32(ref[K - 1])
    expect = float(np.abs(a - b) / a)
    assert expect > 1e-4  # far above the float rounding of the sums
    # each float sum may round to a neighbour of the oracle's (2^-24 relative); FAST sums differ by up to their tolerance
    tol = 4 * 2.0 ** -24 + 2 * velsum_tol(prec, kind) * (1 + expect)
    assert abs(res - expect) <= tol, f"residual {res!r}, from the oracle's sums {expect!r}"


if __name__ == "__main__":
    child_main(sys.argv[1], sys.argv[2])
