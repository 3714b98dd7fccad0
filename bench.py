#!/usr/bin/env python
"""Headline benchmark: MLUPS of the fused D3Q19 BGK step and its HBM-roofline fraction.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--n 512] [--precision f64|f32] [--storage ab|aa] [--no-e2e] [--no-cpu] [--dump-outputs DIR]

Workload (BASELINE.json configs[2]): dense lid-driven cavity 512^3, fp64, one B200.
At N > 1 (torchrun, one rank per GPU) the domain is 1024 x 1024 x (128*N), z-slab sharded -- the
north_star's 1024^2 faces (42 MB per face and direction), 2^27 nodes per GPU like the 512^3 cube, so the
job is weak-scaled and becomes the 1024^3 box at N = 8.  The step kernel stores the 5 crossing
populations per face cell straight into the neighbour GPU's buffer (CUDA IPC peer memory over NVLink)
and the slabs order their steps through progress flags in that memory: the timed loop is
lbm_slab_step inside the library, no NCCL and no Python per step.  --halo nccl packs and sends the faces
with NCCL instead (two-buffer storage only).

`parity_check` (untimed, before the timed region): at N = 1 the benchmarked storage and arithmetic
(in-place, FAST) against the two-buffer storage in the reference's own expression order (STRICT) on the
benchmarked 512^3 box after the same number of steps; at N > 1 a 64 x 64 x 32N cavity and the bifurcation
case stepped on the N ranks and on rank 0 alone, compared bit for bit.

A "step" is one pass of the hot path: one fused pull-stream + collide (+ link-wise boundaries)
launch over every fluid node.  `value` = fluid-node updates / s / 1e6 with all state resident in HBM,
timed with CUDA events on the library's own stream (max over ranks).  `e2e` = the same metric for
one save interval of the reference's main loop driven through the C ABI from host memory: K steps
followed by the D2H copy of rho,ux,uy,uz into pinned host buffers (ldc.cu:669-675), plus -- once,
inside the timed region -- create / geo_pre / index_transform / initialize.
Algorithmic traffic: 2 x 19 x sizeof(real) bytes per fluid-node update (SURVEY 8d).

--impl reference times the CPU restatement of the reference's loop (oracle/, all host threads)
on a bounded sample of the same workload; the reference itself is a CUDA program with the grid
size compiled in (64^3, fp32), so its kernels are reported separately under "reference_cuda": a
patched-constant 480^3 build (baseline/_ref/variants, tools/make_reference_variants.py), with and
without the per-kernel syncs and the thrust::reduce of its loop.

--dump-outputs DIR writes what the last timed step computed -- rho, ux, uy, uz as a caller of get_fields (or of
the oracle's fields) receives them, in the benchmark's precision -- to DIR/<name>.npy, so that two builds can be
compared output for output on identical inputs.  Fields longer than DUMP_SAMPLE entries are replaced by the same
seeded sample of entries on every run; at N > 1 every rank writes its own slab as <name>_rank<r>.npy.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it (it may be read-only)

import numpy as np  # noqa: E402

BYTES_PER_LU = {"f64": 304, "f32": 152}
DUMP_SAMPLE = 1 << 20  # entries per field and process: 32 MB for the four fp64 fields of one GPU


def dump_outputs(out_dir, fields, rank=0, world=1):
    """rho, ux, uy, uz to out_dir/<name>.npy; a field longer than its share of DUMP_SAMPLE is sampled at sorted
    entries drawn with a fixed seed, which depend only on the field's length and the number of ranks"""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    keep = DUMP_SAMPLE // world
    n = fields[0].size
    pick = np.sort(np.random.default_rng(0).choice(n, keep, replace=False)) if n > keep else slice(None)
    for name, a in zip(("rho", "ux", "uy", "uz"), fields):
        assert a.dtype in (np.float32, np.float64) and a.size == n
        np.save(out / (name if world == 1 else f"{name}_rank{rank}"), np.ascontiguousarray(a.reshape(-1)[pick]))


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])), mx.append(float(r[2])), power.append(float(r[3]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(power)), "samples": len(sm)}


def ncu_traffic(precision, n, storage):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture, if one exists for
    exactly this workload"""
    try:
        t = json.loads((ROOT / "profiles" / "traffic.json").read_text())
        return t.get(f"{precision}_{n}_{storage}")
    except Exception:
        return None


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def oracle_threads(n):
    import ctypes

    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(int(n))
    except Exception:
        pass


def cpu_oracle_mlups(n, precision, steps, threads):
    """the oracle's literal update + boundary_stream loop on the host cores"""
    from oracle import oracle as O

    oracle_threads(threads)
    geo = O.geo_pre_ldc(n, n, n)
    idx, nlat = O.index_dense(geo.shape)
    dt = np.float64 if precision == "f64" else np.float32
    o = O.Oracle(O.CASE_LDC, geo, idx, nlat, float(np.float32(0.55)), float(np.float32(0.15) / np.float32(2.4705)), dtype=dt)
    o.initialize()
    o.step(1)
    t = o.time_steps(steps)
    return o.num_fluid() * steps / t / 1e6, t


def reference_cuda_line():
    """The reference's own kernels on this GPU (SURVEY 8d): ldc.cu with NX=NY=NZ=480 -- the largest cube its
    32-bit indexing allows (ldc.cu:80) -- fp32, 30 iterations, timed by the program's own cudaEvent span, (a) as
    shipped: a cudaDeviceSynchronize after each of its three kernels plus a thrust::reduce per step
    (ldc.cu:655-662), (b) kernels only.  Patched-constant builds from tools/make_reference_variants.py (only the
    grid constants and the loop's sync / reduce lines are edited, `update` and `boundary_stream` are untouched)."""
    var = ROOT / "baseline" / "_ref" / "variants"
    out = {"program": "Lid_driven_cavity/ldc.cu, NX=NY=NZ=480 patched in (nvcc -O3 sm_100a), fp32, 30 iterations, own cudaEvent span"}
    import tempfile

    for key, exe in (("as_shipped_loop", var / "ldc_480"), ("kernels_only", var / "ldc_480_stripped")):
        if not exe.exists():
            continue
        try:
            with tempfile.TemporaryDirectory() as wd:
                os.makedirs(os.path.join(wd, "out"))
                r = subprocess.run([str(exe)], cwd=wd, capture_output=True, text=True, timeout=300)
                m = re.search(r"TOTAL RUNNING TIME: ([0-9.eE+-]+) MILLI", r.stdout)
                if m:
                    ms = float(m.group(1)) / 30
                    out[key] = {"ms_per_step": ms, "mlups_fluid": 476 ** 3 / (ms * 1e-3) / 1e6,
                                "GBps_at_152B_per_update": 476 ** 3 * 152 / (ms * 1e-3) / 1e9}
        except Exception as e:  # noqa: BLE001
            out[key] = {"error": str(e)[:200]}
    return out if len(out) > 1 else None


def run_reference_arm(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = args.ref_n
    if n <= 0:  # the arm's own box when the host can hold it (57 GB in fp64), else the largest cube that fits
        avail = 0.0
        try:
            for ln in open("/proc/meminfo"):
                if ln.startswith("MemAvailable"):
                    avail = int(ln.split()[1]) / 2 ** 20
        except OSError:
            pass
        per_node = (2 * 19 + 4) * (8 if args.precision == "f64" else 4) + 19 * 4 + 12  # two buffers, moments, pull table, masks
        n = args.n
        while n > 64 and (n ** 3 * per_node / 2 ** 30 > 0.6 * avail or n ** 3 * (args.steps + args.warmup) > 8e9):
            n -= 64  # also bounds the run to about a minute of stepping at ~120 MLUPS
    # W warm-up + exactly K timed steps of the bounded sample
    from oracle import oracle as O

    oracle_threads(threads)
    geo = O.geo_pre_ldc(n, n, n)
    idx, nlat = O.index_dense(geo.shape)
    dt = np.float64 if args.precision == "f64" else np.float32
    o = O.Oracle(O.CASE_LDC, geo, idx, nlat, float(np.float32(0.55)), float(np.float32(0.15) / np.float32(2.4705)), dtype=dt)
    o.initialize()
    o.step(args.warmup)
    t = o.time_steps(args.steps)
    val = o.num_fluid() * args.steps / t / 1e6
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, o.fields())
    whole = n == args.n and world == 1
    sample = (f"LDC {n}^3 {args.precision}, {args.steps} steps, oracle port of ldc.cu:57-458 on {threads} host threads: "
              + ("the arm's whole workload" if whole else f"a bounded sample of the arm's workload (one {args.n}^3-sized share does not fit / is not needed: "
                                                          "MLUPS of this memory-bound loop is size-independent to first order)"))
    cfg = workload_config(args, world)
    line = {
        "impl": "reference", "metric": "MLUPS", "value": val, "unit": "MLUPS (fluid-node updates/s/1e6)",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": val, "unit": "MLUPS", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "MLUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def global_dims(args, world):
    if args.dims:
        return tuple(args.dims)
    if world > 1 and args.n == 512:
        return 1024, 1024, 128 * world  # 1024^2 faces, 2^27 nodes per GPU (north_star: 1024^3 on 8 GPUs)
    return args.n, args.n, args.n * world


def bind_to_gpu_numa_node(local):
    """run this rank on the cores NVML lists as close to its GPU, so that pinned host buffers are first-touched
    (and the D2H copies land) in that NUMA node; returns the number of cores bound to, or None"""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local]) if os.environ.get("CUDA_VISIBLE_DEVICES", "").replace(",", "").isdigit() else local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return None


def vessel_edge(n, world):
    """cube edge of the vessel workload: --n on one GPU, the same number of nodes per GPU on N (1024 at N = 8)"""
    return n if world == 1 else int(round(n * world ** (1.0 / 3.0) / 32.0)) * 32


def vessel_inputs(n, z0, z1, k=4, rfrac=0.38):
    """host-side synthetic inputs of BASELINE config 5 (same generator as tools/sparse_bench.py and
    tools/vessel_scale.py): planes z0..z1 of a k x k bundle of sinusoidally bent tubes along y as a uint8 voxel
    field [z][y][x], and the parabolic inlet speed plane [z][x] (outlet: pressure, zero plane)"""
    sys.path.insert(0, str(ROOT / "tools"))
    from sparse_bench import tube_bundle

    flag = tube_bundle(n, k, rfrac, z0, z1).astype(np.uint8)
    pitch = n / k
    zz, xx = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    rr2 = ((xx % pitch - pitch / 2) ** 2 + (zz % pitch - pitch / 2) ** 2) / (rfrac * pitch) ** 2
    inlet = (0.05 * np.clip(1 - rr2, 0, None)).astype(np.float32)
    return flag, inlet


def vessel_desc(L, n, z_range, prec, storage, math, device):
    d = L.case_defaults(L.CASE_GEO_Y_INOUT)
    d.nx = d.ny = d.nz = n
    d.z_begin, d.z_end = z_range
    d.precision, d.storage, d.math, d.device = prec, storage, math, device
    d.pulse_amp, d.pulse_period = 0.3, 200.0  # pulsatile inlet (curved vessel/README.md:1: planned by the reference, never written)
    d.bc[0].pulsatile = 1
    return d


def parity_check_vessel(args, L, prec, local, n, flag, inlet, steps):
    """benchmarked storage (FAST) vs box-dense two-buffer STRICT on the benchmarked vessel, same step count"""
    fields = {}
    st = {"ab": L.STORE_DENSE_AB, "aa": L.STORE_DENSE_AA, "sparse_aa": L.STORE_SPARSE_AA, "sparse": L.STORE_SPARSE_AB}[args.storage]
    for name, storage, math in (("bench", st, L.MATH_FAST), ("strict_ab", L.STORE_DENSE_AB, L.MATH_STRICT)):
        c = L.Case(vessel_desc(L, n, (0, n), prec, storage, math, local))
        c.set_flag_slab(flag, 0)
        c.geo_pre(), c.index_transform(), c.set_bc_planes(inlet, np.zeros_like(inlet)), c.initialize()
        c.step(steps)
        fields[name] = c.get_fields()
        c.close()
        del c
    scale = max(float(np.abs(a).max()) for a in fields["strict_ab"][1:])
    err = max(float(np.abs(a - b).max()) / (1.0 if k == 0 else scale) for k, (a, b) in enumerate(zip(fields["bench"], fields["strict_ab"])))
    tol = 1e-10 if args.precision == "f64" else 2e-4
    return {"what": f"vessel bundle {n}^3 {args.precision}, {steps} steps: bench storage '{args.storage}' FAST vs box-dense two-buffer "
                    "STRICT (the arithmetic that is bit-exact with the CPU oracle in tests/); max over rho,ux,uy,uz relative to max|u|",
            "max_rel_err": err, "tol": tol, "ok": bool(err <= tol)}


def parity_check_single(args, L, prec, local, nfluid_expected):
    """benchmarked kernel (in-place, FAST) vs two-buffer STRICT on the benchmarked box, same step count"""
    n, steps = args.n, args.warmup + args.steps
    fields = {}
    for name, storage, math in (("bench", {"ab": L.STORE_DENSE_AB, "aa": L.STORE_DENSE_AA, "sparse_aa": L.STORE_SPARSE_AA,
                                           "sparse": L.STORE_SPARSE_AB}[args.storage], L.MATH_FAST),
                                ("strict_ab", L.STORE_DENSE_AB, L.MATH_STRICT)):
        d = L.case_defaults(L.CASE_LDC)
        d.nx = d.ny = d.nz = n
        d.z_begin, d.z_end = 0, n
        d.precision, d.storage, d.math, d.device = prec, storage, math, local
        c = L.Case(d)
        c.geo_pre(), c.index_transform(), c.initialize()
        c.step(steps)
        fields[name] = c.get_fields()
        assert c.num_fluid == nfluid_expected
        c.close()
        del c
    scale = max(float(np.abs(a).max()) for a in fields["strict_ab"][1:])
    err = 0.0
    for k, (a, b) in enumerate(zip(fields["bench"], fields["strict_ab"])):
        e = float(np.abs(a - b).max()) / (1.0 if k == 0 else scale)
        err = max(err, e)
    tol = 1e-10 if args.precision == "f64" else 2e-4
    return {"what": f"LDC {n}^3 {args.precision}, {steps} steps: bench storage '{args.storage}' FAST vs two-buffer STRICT "
                    "(bit-exact with the CPU oracle, tests/test_parity_512_gpu.py); max over rho,ux,uy,uz relative to max|u|",
            "max_rel_err": err, "tol": tol, "ok": bool(err <= tol)}


def parity_check_multi(args, L, slab, prec, rank, world, local):
    """N ranks == rank 0 alone, bit for bit, on a small cavity and on the bifurcation case"""
    import torch
    import torch.distributed as dist

    sys.path.insert(0, str(ROOT / "tests"))
    results = {}
    gold = ROOT / "tests" / "golden"
    cases = [("ldc_64x64x%d" % (32 * world), L.CASE_LDC, (64, 64, 32 * world), None, None)]
    if world <= 16 and (gold / "bif_flag_bits.npy").exists():
        bits = np.load(gold / "bif_flag_bits.npy")
        flag = np.unpackbits(bits)[: 64 * 83 * 32].astype(np.int32).reshape(32, 83, 64)
        bc = np.load(gold / "bif_bc.npy")
        cases.append(("bifurcation_64x83x32", L.CASE_GEO_Y_INOUT, None, flag, (bc[1], bc[2])))
    storage = {"ab": L.STORE_DENSE_AB, "aa": L.STORE_DENSE_AA, "sparse_aa": L.STORE_SPARSE_AA, "sparse": L.STORE_SPARSE_AB}[args.storage]
    for name, rule, dims, flag, planes in cases:
        def desc(z0, z1):
            d = L.case_defaults(rule)
            if dims:
                d.nx, d.ny, d.nz = dims
            d.z_begin, d.z_end = (0, d.nz) if z0 is None else (z0, z1)
            d.precision, d.storage, d.math, d.device = prec, storage, L.MATH_FAST, local
            return d

        nz = desc(None, None).nz
        z0, z1 = slab.slab_ranges(nz, world)[rank]
        c = slab.SlabCase(desc(z0, z1))
        c.setup(flag=flag, bc_planes=planes)
        fused = args.halo == "p2p" and c.enable_p2p()
        if not fused and storage == L.STORE_DENSE_AA:
            c.enable_staged()
        steps = 41
        c.step(steps)
        mine = [torch.from_numpy(a).cuda() for a in c.get_fields()]
        cnt = torch.tensor([mine[0].numel()], dtype=torch.int64, device="cuda")
        counts = [torch.zeros_like(cnt) for _ in range(world)]
        dist.all_gather(counts, cnt)
        counts = [int(t.item()) for t in counts]
        same = True
        ref = None
        if rank == 0:
            one = L.Case(desc(None, None))
            if flag is not None:
                one.set_flag(flag)
            one.geo_pre(), one.index_transform()
            if planes is not None:
                one.set_bc_planes(*planes)
            one.initialize()
            one.step(steps)
            ref = one.get_fields()
            one.close()
        for k in range(4):
            parts = []
            for r in range(world):
                buf = mine[k] if r == rank else torch.zeros(counts[r], dtype=mine[k].dtype, device="cuda")
                if counts[r]:
                    dist.broadcast(buf, r)
                parts.append(buf)
            if rank == 0:
                same = same and bool(np.array_equal(torch.cat(parts).cpu().numpy(), ref[k]))
        c.close()
        results[name] = {"bitwise_equal": same if rank == 0 else None, "steps": steps, "fused_exchange": bool(fused),
                         "nlattice": int(sum(counts))}
        dist.barrier()
    ok = all(v["bitwise_equal"] for v in results.values()) if rank == 0 else True
    return {"what": f"{world} ranks (z-slabs, storage '{args.storage}', FAST {args.precision}) vs the same case on rank 0 alone, rho,ux,uy,uz compared bit for bit",
            "cases": results, "ok": bool(ok)}


def workload_config(args, world):
    n = args.n
    if args.workload == "vessel":
        e = vessel_edge(n, world)
        return {"workload": f"vessel bundle {e}^3 (4x4 sinusoidally bent tubes along y, ~43 % of the box is fluid), D3Q19 BGK {args.precision}, "
                            f"parabolic pulsatile velocity inlet (amplitude 0.3, period 200 steps), pressure outlet, bifurcation.cu rules; "
                            f"z-slabs of {e // world} planes per GPU (BASELINE config 5)",
                "storage": args.storage, "math": "fast", "bytes_per_node_update": BYTES_PER_LU[args.precision],
                "parallelism": f"zslab{world}", "halo_exchange": args.halo if world > 1 else None,
                "l2_policy": "working set (>=10 GB) far exceeds the 126 MB L2; no flush needed"}
    gx, gy, gz = global_dims(args, world)
    return {"workload": f"dense lid-driven cavity {gx}x{gy}x{gz} D3Q19 BGK {args.precision}, tau=0.55, Re~222 (ldc.cu rules), "
                        f"z-slabs of {gz // world} planes per GPU",
            "storage": args.storage, "math": "fast", "bytes_per_node_update": BYTES_PER_LU[args.precision],
            "parallelism": f"zslab{world}", "halo_exchange": args.halo if world > 1 else None, "l2_policy": "working set (>=20 GB) far exceeds the 126 MB L2; no flush needed"}


def run_ours(args):
    import torch

    import lattice_boltzmann_method_gpu_b200 as L
    from lattice_boltzmann_method_gpu_b200 import slab

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.n
    prec = L.F64 if args.precision == "f64" else L.F32
    storage = {"ab": L.STORE_DENSE_AB, "aa": L.STORE_DENSE_AA, "sparse_aa": L.STORE_SPARSE_AA, "sparse": L.STORE_SPARSE_AB}[args.storage]
    dtype = np.float64 if args.precision == "f64" else np.float32

    vessel = args.workload == "vessel"
    gnx, gny, gnz = (vessel_edge(n, world),) * 3 if vessel else global_dims(args, world)
    z_lo, z_hi = slab.slab_ranges(gnz, world)[rank]
    parity = None
    if not args.no_parity and world > 1:
        parity = parity_check_multi(args, L, slab, prec, rank, world, local)
    if vessel:  # the planes of the voxel field this rank reads (its slab +- 3), generated once, outside every timed region
        fz0, fz1 = max(0, z_lo - 3), min(gnz, z_hi + 3)
        v_flag, v_inlet = vessel_inputs(gnz, fz0, fz1)
        v_zero = np.zeros_like(v_inlet)

    def build_case():
        if vessel:
            d = vessel_desc(L, gnz, (z_lo, z_hi), prec, storage, L.MATH_FAST, local)
            return slab.SlabCase(d) if world > 1 else L.Case(d)
        d = L.case_defaults(L.CASE_LDC)
        d.nx, d.ny, d.nz = gnx, gny, gnz
        d.z_begin, d.z_end = z_lo, z_hi
        d.precision, d.storage, d.math, d.device = prec, storage, L.MATH_FAST, local
        return slab.SlabCase(d) if world > 1 else L.Case(d)

    def setup(c):
        """returns the case ready to step (a different one if the peer mapping is unavailable)"""
        nonlocal storage
        if world == 1:
            if vessel:
                c.set_flag_slab(v_flag, fz0)
            c.geo_pre()
            c.index_transform()
            if vessel:
                c.set_bc_planes(v_inlet, v_zero)
            c.initialize()
            return c
        if args.halo != "p2p" and storage == L.STORE_SPARSE_AA:
            raise SystemExit("the sparse in-place storage exchanges slab faces by peer stores only: use --halo p2p or --storage aa / ab")
        if vessel:
            c.setup(flag_slab=(v_flag, fz0), bc_planes=(v_inlet, v_zero))
        else:
            c.setup()
        if args.halo != "p2p" and storage == L.STORE_DENSE_AA:
            c.enable_staged()  # mailbox exchange through staging buffers that NCCL send/recv moves
            return c
        if args.halo == "p2p" and not c.enable_p2p():  # the decision is all-reduced: every rank takes the same branch
            args.halo = "nccl (peer mapping unavailable)"
            if storage == L.STORE_DENSE_AA:
                c.enable_staged()
                return c
            if storage == L.STORE_SPARSE_AA:
                c.close()
                storage, args.storage = L.STORE_DENSE_AB, "ab"
                c = build_case()
                c.setup(flag_slab=(v_flag, fz0), bc_planes=(v_inlet, v_zero)) if vessel else c.setup()
        return c

    c = setup(build_case())
    nfluid_local = c.num_fluid
    nfluid = nfluid_local
    if not args.no_parity and world == 1 and not args.dims:
        c.close()
        del c
        parity = (parity_check_vessel(args, L, prec, local, gnz, v_flag, v_inlet, args.warmup + args.steps) if vessel
                  else parity_check_single(args, L, prec, local, nfluid_local))
        c = setup(build_case())
    if world > 1:
        t_ = torch.tensor([nfluid_local], dtype=torch.int64, device="cuda")
        dist.all_reduce(t_)
        nfluid = int(t_.item())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: W warm-up, exactly K timed steps, CUDA events, max over ranks
    c.step(args.warmup)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = c.launch_count
    barrier()
    t0 = time.perf_counter()
    ms = c.step_timed(args.steps)
    barrier()
    wall = time.perf_counter() - t0
    launches = c.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t_ = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        ms = float(t_.item())
        l_ = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(l_)
        launches = int(l_.item())
    value = nfluid * args.steps / (ms * 1e-3) / 1e6
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, c.get_fields(), rank, world)

    # the dominant kernel alone (rank 0's slab), CUDA events on the launching stream
    bpl = BYTES_PER_LU[args.precision]
    k_ms = ms / args.steps  # one launch per step (plus face launches at N>1, same kernel)
    achieved = nfluid_local * bpl / (k_ms * 1e-3) / 1e9
    peak, peak_src = measured_peak()

    # ---- end to end through the C ABI from host memory
    e2e = None
    if not args.no_e2e:
        nstored_v = c.local_stored_count() if vessel else 0
        c.close()
        del c
        torch.cuda.empty_cache()
        nstored = nstored_v if vessel else gnx * gny * (z_hi - z_lo)  # LDC stores every node of the slab
        pinned = [torch.empty(nstored, dtype=torch.float64 if args.precision == "f64" else torch.float32).pin_memory()
                  for _ in range(4)]
        outs = [p.numpy() for p in pinned]
        # the whole job e2e_reps times, the median reported: cudaMalloc of the 27 GB slab alone varies between 10 ms
        # and several 100 ms from run to run on a shared host (tools/setup_probe.py), which is not the library's doing
        runs = []
        for rep in range(max(1, args.e2e_reps)):
            if rep:
                c.close()
                del c
            barrier()
            t0 = time.perf_counter()
            c = setup(build_case())
            t1 = time.perf_counter()
            c.step(args.steps)
            t2 = time.perf_counter()
            c.get_fields(outs)
            barrier()
            t_run = time.perf_counter() - t0
            ph = {"setup_s": t1 - t0, "steps_s": t2 - t1, "d2h_s": time.perf_counter() - t2, "cores_bound_near_gpu": numa}
            if getattr(c, "timing", None):
                ph["setup_breakdown_s"] = {k: round(v, 4) for k, v in c.timing.items()}
            if world > 1:
                t_ = torch.tensor([t_run], dtype=torch.float64, device="cuda")
                dist.all_reduce(t_, op=dist.ReduceOp.MAX)
                t_run = float(t_.item())
            runs.append((t_run, ph))
        order = sorted(range(len(runs)), key=lambda i: runs[i][0])
        t_e2e, phases = runs[order[len(order) // 2]]
        phases["all_runs_s"] = [round(r[0], 4) for r in runs]
        e2e = {"value": nfluid * args.steps / t_e2e / 1e6, "unit": "MLUPS",
               "h2d_bytes_per_step": int((__import__("ctypes").sizeof(L.CaseDesc) + (world * (v_flag.nbytes + 2 * v_inlet.nbytes) if vessel else 0)) / args.steps),
               "d2h_bytes_per_step": int(world * 4 * nstored * outs[0].itemsize / args.steps),
               "what": f"median of {len(runs)} runs of: create+geo_pre+index_transform+initialize, {args.steps} steps, D2H of rho,ux,uy,uz into pinned host buffers; "
                       + ("H2D: the descriptor, the uint8 voxel planes of the slab and the two boundary planes" if vessel else
                          "the case is described by a 4.7 KB descriptor (the LDC mask is analytic, ldc.cu:468-502), so H2D is only that"),
               "seconds": t_e2e, "phases": phases}
        assert max(float(np.abs(o).max()) for o in outs[1:]) > 0.0

    if rank == 0:
        cpu = None
        if not args.no_cpu and world == 1:
            cn, csteps = args.cpu_n, args.cpu_steps
            v, t = cpu_oracle_mlups(cn, args.precision, csteps, 1)
            cpu = {"value": v, "unit": "MLUPS", "cores": 1, "kind": "port",
                   "sample": f"LDC {cn}^3 {args.precision}, {csteps} steps ({t:.1f} s) of the oracle's serial update+boundary_stream loop; "
                             f"host has {os.cpu_count()} cores" + ("; the oracle's cost per fluid node does not depend on the geometry" if vessel else "")}
        line = {
            "metric": "MLUPS", "value": value, "unit": "MLUPS (fluid-node updates/s/1e6)", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": workload_config(args, world),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": args.traffic_bytes if args.traffic_bytes else ncu_traffic(args.precision, n, ("vessel_" if vessel else "") + args.storage),
                         "peak_source": peak_src,
                         "kernel": "k_step_dense" if args.storage in ("ab", "aa") else ("k_sparse_aa_even / k_sparse_aa_odd" if args.storage == "sparse_aa" else "k_step_sparse"), "algorithmic_bytes_per_launch": nfluid_local * bpl,
                         "frac_of_spec_8TBs": achieved / 8000.0},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "parity_check": parity,
            "wall_ms_per_step": wall / args.steps * 1e3, "fluid_nodes": int(nfluid),
            "mlups_all_nodes": value * (gnx * gny * gnz) / nfluid,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if world == 1 and not args.no_cpu:
            rc = reference_cuda_line()
            if rc:
                line["reference_cuda"] = rc
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"])
    ap.add_argument("--storage", default=None, choices=["ab", "aa", "sparse_aa", "sparse"],
                    help="aa: box-dense, one population buffer streamed in place (default); ab: two buffers; "
                         "sparse_aa: fluid nodes only, one buffer, in place; sparse: reference compact order, two buffers")
    ap.add_argument("--dims", type=int, nargs=3, default=None, metavar=("NX", "NY", "NZ"),
                    help="global box (default n x n x n*gpus, i.e. weak scaling with one n^3 slab per GPU)")
    ap.add_argument("--halo", default="p2p", choices=["p2p", "nccl"],
                    help="multi-GPU halo exchange: peer stores fused into the step kernel, or pack + NCCL send/recv")
    ap.add_argument("--workload", default="cavity", choices=["cavity", "vessel"],
                    help="cavity: dense lid-driven cavity (BASELINE configs 2-3, the default); vessel: 4x4 bundle of bent tubes, "
                         "~43 %% fluid, pulsatile inlet, sparse in-place storage (BASELINE config 5)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-reps", type=int, default=3, help="end-to-end runs; the median is reported")
    ap.add_argument("--no-parity", action="store_true", help="skip the untimed parity_check")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-n", type=int, default=128)
    ap.add_argument("--cpu-steps", type=int, default=25)
    ap.add_argument("--ref-n", type=int, default=0, help="cube edge of the CPU reference arm (0: the arm's own n when host memory allows)")
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram__bytes_read.sum+dram__bytes_write.sum per launch from the committed ncu capture")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed (rho, ux, uy, uz) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.storage is None:
        args.storage = "sparse_aa" if args.workload == "vessel" else "aa"
    args.warmup = max(args.warmup, 3)
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # started by hand without a launcher: become `torchrun --nproc-per-node N bench.py ...` (one rank per GPU)
        import socket

        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        os.execv(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                  "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
