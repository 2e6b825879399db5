#!/usr/bin/env python
"""Cost of background fields: BASELINE config 3 (512 x 512 x 256, stretched Bounded z, RK3, F64) with B = N² z on b and a shear
U(z) on u, and the 256^3 headline (triply periodic, WENO5, buoyancy tracer, RK3, F64) with B = N² z, each against the same model
without backgrounds.  The two models are stepped alternately in one process: warm-up steps, then timed rounds of
steps (CUDA events, profiling off) and one round with the library's per-phase timing on for the `tendency` phase.  Prints one
JSON line per workload with the GPU name and power limit read in the same run; --out appends them to a file.
usage: tools/background_bench.py [--steps 20] [--warmup 3] [--rounds 3] [--out profiles/background_bench.jsonl]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "clima-oceananigans.jl_b200")):
    sys.path.insert(0, p)
from tools.c3_bench import z_faces  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as e:          # the numbers are still CUDA-event timings; say what could not be read
        return f"unknown ({e})", "unknown"


def c3_model(ob, arch, background):
    Nx, Ny, Nz = 512, 512, 256
    zf = z_faces(Nz)
    g = ob.RectilinearGrid(arch, np.float64, size=(Nx, Ny, Nz), x=(0, 64), y=(0, 64), z=zf,
                           topology=("Periodic", "Periodic", "Bounded"))
    bcs = {"u": {"top": ob.BoundaryCondition("Flux", -1e-4)},
           "b": {"top": ob.BoundaryCondition("Flux", 1e-8), "bottom": ob.BoundaryCondition("Gradient", 1e-5)}}
    bg = None
    if background:        # stratification N² = 1e-5 and a surface-intensified shear
        bg = {"b": lambda x, y, z, t: 1e-5 * z, "u": lambda x, y, z, t: 0.05 * np.exp(z / 8.0)}
    m = ob.NonhydrostaticModel(g, advection=ob.WENO5(grid=g), tracers=("b",), buoyancy=ob.Buoyancy(ob.BuoyancyTracer(), None),
                               coriolis=ob.FPlane(1e-4), closure=ob.ScalarDiffusivity("ThreeDimensional", ν=1e-4, κ=1e-4),
                               timestepper="RungeKutta3", boundary_conditions=bcs, background_fields=bg)
    rng = np.random.default_rng(3)
    vals = {n: 1e-2 * rng.uniform(-1, 1, m.fields[n].size()) for n in "uvw"}
    vals["b"] = 1e-7 * rng.uniform(-1, 1, (Nx, Ny, Nz))
    ob.set_model(m, **vals)
    return m, 0.05


def headline_model(ob, arch, background):
    N = 256
    g = ob.RectilinearGrid(arch, np.float64, size=(N, N, N), extent=(1, 1, 1), topology=("Periodic",) * 3)
    bg = {"b": lambda x, y, z, t: 1e-5 * z} if background else None
    m = ob.NonhydrostaticModel(g, advection=ob.WENO5(), tracers=("b",), buoyancy=ob.BuoyancyTracer(), timestepper="RungeKutta3",
                               background_fields=bg)
    rng = np.random.default_rng(2)
    vals = {}
    for n in "uvw":
        a = rng.uniform(-1, 1, (N, N, N))
        vals[n] = a - a.mean()
    vals["b"] = 1e-3 * rng.uniform(-1, 1, (N, N, N))
    ob.set_model(m, **vals)
    return m, 0.1 / N


def measure(ob, lib, torch, stream, models, dt, steps, warmup, rounds):
    for m in models.values():
        for _ in range(warmup):
            ob.time_step(m, dt)
    torch.cuda.synchronize()
    ms = {k: [] for k in models}
    for _ in range(rounds):                       # alternate the two models, round by round
        for k, m in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                ob.time_step(m, dt)
            e1.record(stream)
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / steps)
    tend = {}
    for k, m in models.items():                  # the tendency phase in a round of its own (event pairs per launch)
        lib.ob200_profile_reset()
        lib.ob200_profile_enable(1)
        for _ in range(steps):
            ob.time_step(m, dt)
        torch.cuda.synchronize()
        lib.ob200_profile_enable(0)
        t, c = C.c_double(), C.c_int64()
        lib.ob200_profile_query(b"tendency", C.byref(t), C.byref(c))
        tend[k] = t.value / steps
    return ms, tend


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import ocean_b200 as ob
    from ocean_b200._lib import lib
    if not torch.cuda.is_available():
        raise SystemExit("background_bench needs a CUDA device")
    arch = ob.B200(0)
    stream = torch.cuda.current_stream()
    lib.ob200_set_stream(C.c_void_p(stream.cuda_stream))
    name, power = gpu_info()
    lines = []
    for wl, mk in (("C3 512x512x256 F64 RK3, B = N^2 z on b, U(z) on u", c3_model),
                   ("headline 256^3 F64 RK3, B = N^2 z on b", headline_model)):
        models = {}
        for background in (False, True):
            models["background" if background else "none"], dt = mk(ob, arch, background)
        ms, tend = measure(ob, lib, torch, stream, models, dt, a.steps, a.warmup, a.rounds)
        rec = {"workload": wl, "gpu": name, "power_limit": power, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
               "ms_per_step": {k: [round(v, 4) for v in vs] for k, vs in ms.items()},
               "ms_per_step_min": {k: round(min(vs), 4) for k, vs in ms.items()},
               "tendency_ms_per_step": {k: round(v, 4) for k, v in tend.items()},
               "tendency_slowdown_pct": round(100 * (tend["background"] / tend["none"] - 1), 2),
               "step_slowdown_pct": round(100 * (min(ms["background"]) / min(ms["none"]) - 1), 2)}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        for m in models.values():
            m.destroy()
        del models
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
