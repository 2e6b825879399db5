#!/usr/bin/env python
"""Cost of array boundary conditions: BASELINE config 3 (512 x 512 x 256, stretched Bounded z, WENO5(grid), RK3, F64) with top
Flux arrays on u, v, b and a bottom Gradient array on b, against the same model with constant conditions.  The two models are
stepped alternately in one process: warm-up steps, then timed rounds of steps (CUDA events, profiling off) and one round per model
with the library's per-phase timing on for the `tendency` phase and the array Flux pass (`boundary_flux`).  Prints one JSON line
with the GPU name and power limit read in the same run; --out appends it to a file.
usage: tools/bc_array_bench.py [--steps 20] [--warmup 3] [--rounds 3] [--out profiles/r4_bc_array_bench.jsonl]"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "clima-oceananigans.jl_b200")):
    sys.path.insert(0, p)
from tools.c3_bench import z_faces  # noqa: E402
from tools.forcing_bench import gpu_info  # noqa: E402


def c3_model(ob, arch, arrays):
    Nx, Ny, Nz = 512, 512, 256
    zf = z_faces(Nz)
    g = ob.RectilinearGrid(arch, np.float64, size=(Nx, Ny, Nz), x=(0, 64), y=(0, 64), z=zf,
                           topology=("Periodic", "Periodic", "Bounded"))
    if arrays:        # a wind-stress pattern, a cooling patch and a bottom gradient varying along x
        x = (np.arange(Nx) + 0.5) / Nx
        y = (np.arange(Ny) + 0.5) / Ny
        X, Y = np.meshgrid(x, y, indexing="ij")
        bcs = {"u": {"top": ob.FluxBoundaryCondition(-1e-4 * (1 + 0.5 * np.sin(2 * np.pi * Y)))},
               "v": {"top": ob.FluxBoundaryCondition(2e-5 * np.cos(2 * np.pi * X))},
               "b": {"top": ob.FluxBoundaryCondition(1e-8 * np.exp(-((X - 0.5) ** 2 + (Y - 0.5) ** 2) / 0.02)),
                     "bottom": ob.GradientBoundaryCondition(1e-5 * (1 + 0.1 * np.sin(2 * np.pi * X)))}}
    else:
        bcs = {"u": {"top": ob.FluxBoundaryCondition(-1e-4)}, "v": {"top": ob.FluxBoundaryCondition(2e-5)},
               "b": {"top": ob.FluxBoundaryCondition(1e-8), "bottom": ob.GradientBoundaryCondition(1e-5)}}
    m = ob.NonhydrostaticModel(g, advection=ob.WENO5(grid=g), tracers=("b",), buoyancy=ob.Buoyancy(ob.BuoyancyTracer(), None),
                               coriolis=ob.FPlane(1e-4), closure=ob.ScalarDiffusivity("ThreeDimensional", ν=1e-4, κ=1e-4),
                               timestepper="RungeKutta3", boundary_conditions=bcs)
    rng = np.random.default_rng(3)
    vals = {n: 1e-2 * rng.uniform(-1, 1, m.fields[n].size()) for n in "uvw"}
    zc = 0.5 * (zf[1:] + zf[:-1])
    vals["b"] = 1e-5 * zc.reshape(1, 1, Nz) + 1e-7 * rng.uniform(-1, 1, (Nx, Ny, Nz))
    ob.set_model(m, **vals)
    return m, 0.05


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
        raise SystemExit("bc_array_bench needs a CUDA device")
    arch = ob.B200(0)
    stream = torch.cuda.current_stream()
    lib.ob200_set_stream(C.c_void_p(stream.cuda_stream))
    name, power = gpu_info()
    models = {}
    for arrays in (False, True):
        models["arrays" if arrays else "constants"], dt = c3_model(ob, arch, arrays)
    for m in models.values():
        for _ in range(a.warmup):
            ob.time_step(m, dt)
    torch.cuda.synchronize()
    ms = {k: [] for k in models}
    for _ in range(a.rounds):                     # alternate the two models, round by round
        for k, m in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(a.steps):
                ob.time_step(m, dt)
            e1.record(stream)
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / a.steps)
    phases = {}
    for k, m in models.items():                  # per-phase timing in a round of its own (event pairs per launch)
        lib.ob200_profile_reset()
        lib.ob200_profile_enable(1)
        for _ in range(a.steps):
            ob.time_step(m, dt)
        torch.cuda.synchronize()
        lib.ob200_profile_enable(0)
        phases[k] = {}
        for ph in ("tendency", "boundary_flux"):
            t, c = C.c_double(), C.c_int64()
            lib.ob200_profile_query(ph.encode(), C.byref(t), C.byref(c))
            phases[k][ph] = {"ms_per_step": round(t.value / a.steps, 4), "launches_per_step": c.value / a.steps}
    rec = {"workload": "C3 512x512x256 F64 RK3, top Flux arrays on u, v, b + bottom Gradient array on b vs constants",
           "gpu": name, "power_limit": power, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
           "ms_per_step": {k: [round(v, 4) for v in vs] for k, vs in ms.items()},
           "ms_per_step_min": {k: round(min(vs), 4) for k, vs in ms.items()},
           "phases": phases,
           "step_slowdown_pct": round(100 * (min(ms["arrays"]) / min(ms["constants"]) - 1), 2)}
    print(json.dumps(rec), flush=True)
    for m in models.values():
        m.destroy()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
