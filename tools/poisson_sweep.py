#!/usr/bin/env python
"""BASELINE.json config 4: standalone pressure-solve sweep, N^3 for N in 128..1024, Float64, one B200.

  python tools/poisson_sweep.py [fft|ft|cpu] N [N ...]

  fft  FFTBasedPoissonSolver, triply periodic (solve_for_pressure!: divergence of a seeded velocity field fused in)
  ft   FourierTridiagonalPoissonSolver, (Periodic, Periodic, Bounded) with the vertical stretching of the ocean
       wind-mixing / convection example (examples/ocean_wind_mixing_and_convection.jl:41-54)
  topo FFTBasedPoissonSolver on a regular grid for all eight (Periodic | Bounded)^3 topologies (Bounded = DCT by Makhoul's
       algorithm; a non-power-of-two N runs Bluestein's)
  cpu  the CPU stand-in of SURVEY.md 8(d)(iii): the same triply periodic solve with scipy.fft (pocketfft, all host
       threads) -- rfftn, eigenvalue divide, irfftn -- timed on the box's host cores (bounded: N <= 256)

Prints solves/s, points/s and achieved GB/s against the 12-words-per-point algorithmic traffic of SURVEY.md 8(d), plus
the residual max|lap(phi) - R| / max|R| of the reference's own check (test/dependencies_for_poisson_solvers.jl:86-104)."""
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "clima-oceananigans.jl_b200")):
    sys.path.insert(0, p)


def z_faces(Nz, Lz=1.0, refinement=1.2, stretching=12.0):
    k = np.arange(1, Nz + 2)
    h = (k - 1) / Nz
    zeta0 = 1 + (h - 1) / refinement
    Sigma = (1 - np.exp(-stretching * h)) / (1 - np.exp(-stretching))
    return Lz * (zeta0 * Sigma - 1)


def cpu_solve_time(N, reps=3):
    import scipy.fft as sf
    rng = np.random.default_rng(4)
    rhs = rng.uniform(-1, 1, (N, N, N))
    rhs -= rhs.mean()
    d = 1.0 / N
    lam = (2 * np.sin(np.arange(N) * np.pi / N) / d) ** 2
    lamh = (2 * np.sin(np.arange(N // 2 + 1) * np.pi / N) / d) ** 2
    den = -(lam[:, None, None] + lam[None, :, None] + lamh[None, None, :])
    den[0, 0, 0] = 1.0
    workers = os.cpu_count() or 1
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        s = sf.rfftn(rhs, workers=workers)
        s /= den
        s[0, 0, 0] = 0
        phi = sf.irfftn(s, s=rhs.shape, workers=workers)
        best = min(best, time.perf_counter() - t0)
    lap = sum((np.roll(phi, -1, a) - 2 * phi + np.roll(phi, 1, a)) / d ** 2 for a in range(3))
    return best * 1e3, workers, float(np.max(np.abs(lap - rhs)) / np.max(np.abs(rhs)))


def main():
    args = sys.argv[1:]
    mode = "fft"
    if args and args[0] in ("fft", "ft", "cpu", "topo"):
        mode = args.pop(0)
    sizes = [int(x) for x in (args or ["128", "256", "512"])]
    out = []
    if mode == "cpu":
        for N in sizes:
            ms, workers, res = cpu_solve_time(N)
            out.append({"solver": "scipy.fft rfftn/irfftn (CPU stand-in)", "N": N, "ms_per_solve": ms, "threads": workers,
                        "points_per_s": N ** 3 / (ms * 1e-3), "residual": res})
        print(json.dumps(out))
        return
    import torch
    import ocean_b200 as ob
    from ocean_b200._lib import lib
    arch = ob.B200(0)
    stream = torch.cuda.current_stream()
    lib.ob200_set_stream(C.c_void_p(stream.cuda_stream))
    if mode == "topo":
        for N in sizes:
            for topo in [(a, b, c) for a in "PB" for b in "PB" for c in "PB"]:
                names = tuple({"P": "Periodic", "B": "Bounded"}[t] for t in topo)
                g = ob.RectilinearGrid(arch, np.float64, size=(N, N, N), extent=(1, 1, 1), topology=names)
                s = ob.FFTBasedPoissonSolver(g)
                rng = np.random.default_rng(4)
                U = {}
                for d, (n, f) in enumerate((("u", ob.XFaceField), ("v", ob.YFaceField), ("w", ob.ZFaceField))):
                    U[n] = f(g)
                    a = rng.uniform(-1, 1, U[n].size())
                    if topo[d] == "B":                    # impenetrable walls
                        sl = [slice(None)] * 3
                        sl[d] = 0
                        a[tuple(sl)] = 0
                        sl[d] = -1
                        a[tuple(sl)] = 0
                    U[n].set(a)
                ob.fill_halo_regions(list(U.values()))
                phi = ob.CenterField(g)
                for _ in range(2):
                    ob.solve_for_pressure(phi, s, 1.0, U)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                reps = 10
                torch.cuda.synchronize()
                e0.record(stream)
                for _ in range(reps):
                    ob.solve_for_pressure(phi, s, 1.0, U)
                e1.record(stream)
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / reps
                # the reference's own check: lap(phi) == div(U) (test/dependencies_for_poisson_solvers.jl:86-104)
                ob.fill_halo_regions(phi)
                p = phi.parent()
                d_, H = 1.0 / N, 3
                I = slice(H, N + H)
                c = p[I, I, I]
                lap = ((p[H + 1:N + H + 1, I, I] - 2 * c + p[H - 1:N + H - 1, I, I]) +
                       (p[I, H + 1:N + H + 1, I] - 2 * c + p[I, H - 1:N + H - 1, I]) +
                       (p[I, I, H + 1:N + H + 1] - 2 * c + p[I, I, H - 1:N + H - 1])) / d_ ** 2
                u, v, w = (U[n].parent() for n in "uvw")
                div = ((u[H + 1:N + H + 1, I, I] - u[I, I, I]) + (v[I, H + 1:N + H + 1, I] - v[I, I, I]) +
                       (w[I, I, H + 1:N + H + 1] - w[I, I, I])) / d_
                res = float(np.max(np.abs(lap - div)) / np.max(np.abs(div)))
                out.append({"solver": "FFTBasedPoissonSolver", "topology": "".join(topo), "N": N, "ms_per_solve": ms,
                            "points_per_s": N ** 3 / (ms * 1e-3), "residual": res})
                del s, phi, U, g
        print(json.dumps(out))
        return
    for N in sizes:
        if mode == "fft":
            g = ob.RectilinearGrid(arch, np.float64, size=(N, N, N), extent=(1, 1, 1), topology=("Periodic",) * 3)
            s = ob.FFTBasedPoissonSolver(g)
        else:
            g = ob.RectilinearGrid(arch, np.float64, size=(N, N, N), x=(0, 1), y=(0, 1), z=z_faces(N),
                                   topology=("Periodic", "Periodic", "Bounded"))
            s = ob.FourierTridiagonalPoissonSolver(g)
        rng = np.random.default_rng(4)
        U = {}
        for n, f in (("u", ob.XFaceField), ("v", ob.YFaceField), ("w", ob.ZFaceField)):
            U[n] = f(g)
            a = rng.uniform(-1, 1, U[n].size())
            if n == "w" and mode == "ft":
                a[:, :, 0] = 0
                a[:, :, -1] = 0           # impenetrable top and bottom
            U[n].set(a)
        ob.fill_halo_regions(list(U.values()))
        phi = ob.CenterField(g)
        for _ in range(3):
            ob.solve_for_pressure(phi, s, 1.0, U)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20 if N <= 512 else 5
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(reps):
            ob.solve_for_pressure(phi, s, 1.0, U)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        res = None
        if N <= 256 and mode == "fft":     # the reference's own check: lap(phi) == div(U)
            ob.fill_halo_regions(phi)
            p = phi.parent()
            d, H = 1.0 / N, 3
            I = slice(H, N + H)
            c = p[I, I, I]
            lap = ((p[H + 1:N + H + 1, I, I] - 2 * c + p[H - 1:N + H - 1, I, I]) +
                   (p[I, H + 1:N + H + 1, I] - 2 * c + p[I, H - 1:N + H - 1, I]) +
                   (p[I, I, H + 1:N + H + 1] - 2 * c + p[I, I, H - 1:N + H - 1])) / d ** 2
            u, v, w = (U[n].parent() for n in "uvw")
            div = ((u[H + 1:N + H + 1, I, I] - u[I, I, I]) + (v[I, H + 1:N + H + 1, I] - v[I, I, I]) +
                   (w[I, I, H + 1:N + H + 1] - w[I, I, I])) / d
            res = float(np.max(np.abs(lap - div)) / np.max(np.abs(div)))
        out.append({"solver": "FFTBasedPoissonSolver (P,P,P)" if mode == "fft" else "FourierTridiagonalPoissonSolver (P,P,B) stretched",
                    "N": N, "ms_per_solve": ms, "solves_per_s": 1e3 / ms, "points_per_s": N ** 3 / (ms * 1e-3),
                    "algorithmic_GBps": 96.0 * N ** 3 / (ms * 1e-3) / 1e9, "residual": res})
        del s, phi, U, g
    print(json.dumps(out))


if __name__ == "__main__":
    main()
