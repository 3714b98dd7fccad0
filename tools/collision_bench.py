#!/usr/bin/env python3
"""Cost of the two-relaxation-time (TRT) collision against BGK on the benchmark workloads.

One case per workload is built once; BGK and TRT (magic parameter 3/16) then alternate on it, window after
window, so that both operators see the same card, clocks and state.  Each window is timed with CUDA events
(lbm_step_timed) after a warm-up, and holds at least --min-window seconds of stepping.  The card name and power
limit are read by the same process.  Prints one JSON line: MLUPS per operator (median over the windows) and the
TRT/BGK ratio per workload.

    python tools/collision_bench.py [--n 512] [--rounds 3] [--workloads cavity_f64,cavity_f32,vessel_f64,vessel_f32]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # writes nothing into the tree it runs from

import numpy as np  # noqa: E402

import bench  # noqa: E402  (vessel_inputs / vessel_desc: the benchmark's own workload builders)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    name, limit = (s.strip() for s in out[0].split(","))
    return {"name": name, "power_limit": limit}


def build(L, workload, n):
    kind, prec = workload.split("_")
    p = L.F64 if prec == "f64" else L.F32
    if kind == "cavity":  # bench.py --workload cavity --storage aa
        d = L.case_defaults(L.CASE_LDC)
        d.nx = d.ny = d.nz = n
        d.z_begin, d.z_end = 0, n
        d.precision, d.storage, d.math = p, L.STORE_DENSE_AA, L.MATH_FAST
        c = L.Case(d)
        c.geo_pre(), c.index_transform(), c.initialize()
        return c
    # bench.py --workload vessel --storage sparse_aa
    flag, inlet = bench.vessel_inputs(n, 0, n)
    c = L.Case(bench.vessel_desc(L, n, (0, n), p, L.STORE_SPARSE_AA, L.MATH_FAST, 0))
    c.set_flag_slab(flag, 0)
    c.geo_pre(), c.index_transform()
    c.set_bc_planes(inlet, np.zeros_like(inlet))
    c.initialize()
    return c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3, help="BGK / TRT window pairs per workload")
    ap.add_argument("--min-window", type=float, default=1.0, help="seconds of stepping per timed window")
    ap.add_argument("--magic", type=float, default=3 / 16)
    ap.add_argument("--workloads", default="cavity_f64,cavity_f32,vessel_f64,vessel_f32")
    args = ap.parse_args()

    import lattice_boltzmann_method_gpu_b200 as L

    result = {"card": card(), "n": args.n, "magic": args.magic, "workloads": {}}
    for w in args.workloads.split(","):
        c = build(L, w, args.n)
        nfluid = c.num_fluid
        steps = {}
        for model in (L.COLL_BGK, L.COLL_TRT):  # warm-up of both operators; sizes the windows
            c.set_collision(model, args.magic)
            c.step(args.warmup)
            ms = c.step_timed(args.warmup)
            steps[model] = max(args.warmup, int(np.ceil(args.min_window * 1e3 / ms * args.warmup)))
            steps[model] += steps[model] % 2  # whole AA step pairs
        mlups = {L.COLL_BGK: [], L.COLL_TRT: []}
        for _ in range(args.rounds):
            for model in (L.COLL_BGK, L.COLL_TRT):
                c.set_collision(model, args.magic)
                ms = c.step_timed(steps[model])
                mlups[model].append(nfluid * steps[model] / (ms * 1e-3) / 1e6)
        c.close()
        bgk, trt = float(np.median(mlups[L.COLL_BGK])), float(np.median(mlups[L.COLL_TRT]))
        result["workloads"][w] = {"nodes": nfluid, "steps_per_window": {"bgk": steps[L.COLL_BGK], "trt": steps[L.COLL_TRT]},
                                  "mlups_bgk": round(bgk, 1), "mlups_trt": round(trt, 1), "trt_over_bgk": round(trt / bgk, 4),
                                  "windows_bgk": [round(v, 1) for v in mlups[L.COLL_BGK]],
                                  "windows_trt": [round(v, 1) for v in mlups[L.COLL_TRT]]}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
