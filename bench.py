#!/usr/bin/env python
"""bench.py -- grid-point updates/sec of one RK3 step of NonhydrostaticModel on B200, the HBM roofline fraction of the
dominant kernel, an end-to-end number with host buffers and a CPU baseline.  Contract: task statement / DESIGN.md 5.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c5-weak|c5-strong] [--ftype f64|f32]
                  [--size n] [--impl ours|reference] [--dump-outputs DIR]

Configurations (BASELINE.json `configs`, SURVEY.md 8(d)):
  c2        (default, the headline) 256^3 triply periodic, WENO5 + tracer b + BuoyancyTracer, FFT solver, RK3.
            With --gpus N > 1: weak scaling, 256^3 per GPU, global grid 256 x 256 N x 256 slab-decomposed in y.
  c3        512 x 512 x 256, Bounded vertically stretched z, WENO5(grid), closure, FPlane, flux / gradient BCs,
            Fourier-tridiagonal solver (one GPU).
  c5-weak   C2 physics, 512^3 per GPU (global 512 x 512 N x 512).
  c5-strong C2 physics, global 1024^3 split over the N GPUs (N >= 2: one B200 cannot hold it with out-of-place substeps).
  (c4, the stand-alone Poisson sweep, has its own metric: tools/poisson_sweep.py, results under profiles/.)
--size n scales a configuration down (n replaces 256 / 512 / 1024) for quick checks; the JSON line names what ran.

N > 1 is launched by torchrun (one rank per GPU).  One "step" = one full RK3 time step (3 stages, 3 pressure solves) of
every cell of the workload.  Prints ONE JSON line on rank 0.

--dump-outputs DIR writes the prognostic fields (u, v, w and the tracers) as they stand after the last timed step to
DIR/<name>.npy (rank 0's slab with several GPUs), so that two builds run with the same arguments -- hence the same seeded
inputs -- can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "clima-oceananigans.jl_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

# DRAM bytes of one fused tendency launch at 256^3 F64 (all four fields of a stage) from the committed ncu capture
# (profiles/r2_summary.md: dram__bytes_read.sum + dram__bytes_write.sum = 1.40 + 1.05 GB)
NCU_TRAFFIC_BYTES_PER_FUSED_LAUNCH = 2.45e9
# ... and of one per-field launch of the round-1 kernel (profiles/r1_summary.md), used when the fused kernel is switched off
NCU_TRAFFIC_BYTES_PER_FIELD_LAUNCH = 8.93e8

# ... and of one fused Bounded-z launch of BASELINE config 3 at 512 x 512 x 256 F64 (profiles/r2_summary.md, capture r2i:
# 6.12 + 4.28 GB against 8.41 GB algorithmic)
NCU_TRAFFIC_BYTES_PER_FUSED_LAUNCH_C3 = 1.04e10

METRIC = "grid-point updates/sec (RK3 step, 256^3 WENO5+FFT)"
UNIT = "grid-point updates/s"

# --dump-outputs writes at most this many bytes in all
DUMP_BYTES = 64 * 10 ** 6


def synthetic_state(shape, seed=2):
    """SURVEY.md 8(d) C2: uniform(-1,1) velocities with the mean removed, b = N^2 z + noise."""
    import numpy as np
    rng = np.random.default_rng(seed)
    vals = {}
    for n in "uvw":
        a = rng.uniform(-1, 1, shape)
        vals[n] = a - a.mean()
    z = (np.arange(shape[2]) + 0.5) / shape[2]
    vals["b"] = 1e-5 * z.reshape(1, 1, -1) + 1e-3 * rng.uniform(-1, 1, shape)
    return vals


def c3_z_faces(Nz, Lz=32.0, refinement=1.2, stretching=12.0):
    """examples/ocean_wind_mixing_and_convection.jl:41-54, scaled to Nz levels"""
    import numpy as np
    k = np.arange(1, Nz + 2)
    h = (Nz + 1 - k) / Nz
    zeta0 = 1 + (h - 1) / refinement
    Sigma = (1 - np.exp(-stretching * h)) / (1 - np.exp(-stretching))
    return Lz * (zeta0 * Sigma - 1)


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons every 20 ms.  It is started BEFORE the warm-up (the nvidia-smi
    process needs ~0.1 s to deliver its first line); mark_begin()/mark_end() bracket the timed region and the
    summary reports the samples that fall inside it (and, beside them, all samples taken under load)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append((time.perf_counter(), parts))
                if self.stop_flag:
                    break
            self.proc.terminate()
        except Exception:
            pass

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def summ(samples):
            sm = sorted(int(s[0]) for _, s in samples if s[0].isdigit())
            reasons = [n for k, n in enumerate(names) if any(s[2 + k].lower().startswith("active") for _, s in samples)]
            return (sm[len(sm) // 2] if sm else None), reasons
        inside = [x for x in self.samples if self.t0 is not None and self.t1 is not None and self.t0 <= x[0] <= self.t1 + 0.02]
        load = [x for x in self.samples if self.t0 is None or x[0] >= self.t0 - 1.0]
        med_in, reasons_in = summ(inside) if inside else (None, [])
        med_load, reasons_load = summ(load if load else self.samples)
        return {"sm_mhz": med_in if med_in is not None else med_load, "sm_max_mhz": int(self.samples[0][1][1]),
                "reasons": sorted(set(reasons_in) | set(reasons_load)), "samples": len(inside),
                "samples_under_load": len(load), "sm_mhz_under_load": med_load}


def cpu_reference_run(steps, warmup, sample_n=256, budget_s=150.0):
    """The reference's CPU path is pure Julia and cannot run here (no Julia toolchain, SURVEY.md 8(c)).
    What is timed is the oracle port -- the compiled OpenMP twin oracle/oracle_cpu.c, same arithmetic and same work per
    point as the reference's CPU kernels (both faces, both WENO sides per cell), on all host cores -- on a bounded sample
    of the C2 workload: `steps` RK3 steps (after `warmup` untimed ones) of the triply periodic WENO5 + b + FFT model at
    sample_n^3, halved until (steps + warmup) steps fit the time budget (the per-point cost does not depend on N).
    Returns (points/s, s per step, cores, sample description, sample_n actually run)."""
    from oracle import cpu_twin
    # all host cores, whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1 to its workers)
    cores = max(cpu_twin.max_threads(), len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    # probe the per-point cost on a small case to size the sample
    Np = 64
    vals = synthetic_state((Np,) * 3)
    pargs = ((Np,) * 3, (1.0, 1.0, 1.0), vals["u"], vals["v"], vals["w"], vals["b"])
    t0 = time.perf_counter(); cpu_twin.rk3_run(*pargs, 0, 0.1 / Np, project=False, nthreads=cores); ts = time.perf_counter() - t0
    t0 = time.perf_counter(); cpu_twin.rk3_run(*pargs, 1, 0.1 / Np, project=False, nthreads=cores)
    per_point = max(time.perf_counter() - t0 - ts, 1e-6) / Np ** 3
    N = sample_n
    while N > 32 and per_point * N ** 3 * (steps + warmup) * 1.3 > budget_s:
        N //= 2
    vals = synthetic_state((N,) * 3)
    dt = 0.1 / N
    args = ((N, N, N), (1.0, 1.0, 1.0), vals["u"], vals["v"], vals["w"], vals["b"])
    # the set-up (halo allocation, copies) is inside the call; the run of `warmup` steps is timed too and differenced away
    t0 = time.perf_counter()
    cpu_twin.rk3_run(*args, warmup, dt, project=False, nthreads=cores)
    t_warm = time.perf_counter() - t0
    t0 = time.perf_counter()
    cpu_twin.rk3_run(*args, warmup + steps, dt, project=False, nthreads=cores)
    el = max(time.perf_counter() - t0 - t_warm, 1e-9)
    return (N ** 3 * steps / el, el / steps, cores,
            f"{steps} RK3 step(s) after {warmup} warm-up step(s) of the C2 model at {N}^3 "
            f"(compiled OpenMP twin of the oracle, {cores} threads)", N)


def dump_outputs(model, out_dir, seed=0):
    """Writes every prognostic field's interior to out_dir/<name>.npy in the run's float type.  When the fields together
    exceed DUMP_BYTES, each is replaced by its values at a seeded, sorted sample of flat column-major interior indices:
    the sample depends only on the seed and the field's shape, so it is the same from run to run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {n: model.fields[n].interior() for n in model.names}
    budget = DUMP_BYTES - 4096 * len(arrays)                   # room for the .npy headers
    sample = sum(x.nbytes for x in arrays.values()) > budget
    for n, x in arrays.items():
        if sample:
            k = budget // (len(arrays) * x.itemsize)
            idx = np.unique(np.random.default_rng(seed).integers(0, x.size, k))
            x = x.ravel(order="F")[idx]
        np.save(os.path.join(out_dir, f"{n}.npy"), np.ascontiguousarray(x))


def build_config(ob, np, a, arch, world, rank, FTYPE):
    """returns (model, dt, points per GPU, global shape, workload string, fields, algorithmic words per point per step)"""
    cfg = a.config
    if cfg == "c3":
        # weak scaling on several GPUs: the slab of every rank is the single-GPU grid, y is decomposed
        s = a.size or 512
        Nx, Ny, Nz = s, s, max(16, s // 2)
        g = ob.RectilinearGrid(arch, FTYPE, size=(Nx, Ny * world, Nz), x=(0, 64), y=(0, 64 * world), z=c3_z_faces(Nz),
                               topology=("Periodic", "Periodic", "Bounded"))
        bcs = {"u": {"top": ob.BoundaryCondition("Flux", -1e-4)},
               "b": {"top": ob.BoundaryCondition("Flux", 1e-8), "bottom": ob.BoundaryCondition("Gradient", 1e-5)}}
        m = ob.NonhydrostaticModel(g, advection=ob.WENO5(grid=g),
                                   tracers=("b",), buoyancy=ob.Buoyancy(ob.BuoyancyTracer(), None), coriolis=ob.FPlane(1e-4),
                                   closure=(ob.AnisotropicMinimumDissipation() if a.closure == "amd" else
                                            ob.SmagorinskyLilly() if a.closure == "smagorinsky" else
                                            ob.ScalarDiffusivity("ThreeDimensional", ν=1e-4, κ=1e-4)),
                                   timestepper="RungeKutta3", boundary_conditions=bcs)
        rng = np.random.default_rng(3)
        vals = {n: 1e-2 * rng.uniform(-1, 1, m.fields[n].size()) for n in "uvw"}
        zf = c3_z_faces(Nz)
        zc = 0.5 * (zf[1:] + zf[:-1])
        vals["b"] = 1e-5 * zc.reshape(1, 1, Nz) + 1e-7 * rng.uniform(-1, 1, (Nx, Ny, Nz))
        ob.set_model(m, **vals)
        wl = (f"C3: {Nx}x{Ny * world}x{Nz} (Periodic, Periodic, Bounded) vertically stretched z, WENO5(grid) + tracer b + FPlane + "
              f"ScalarDiffusivity + flux/gradient BCs, Fourier-tridiagonal pressure solve, RK3"
              + (f", y slab-decomposed over {world} GPUs" if world > 1 else "")
              + ("" if a.closure == "scalar" else f" [closure: {a.closure} instead of ScalarDiffusivity]"))
        return m, 0.05, Nx * Ny * Nz, (Nx, Ny * world, Nz), wl, 4, 110.0
    if cfg == "c5-strong":
        s = a.size or 1024
        if s % world:
            raise SystemExit("global size must be divisible by the number of GPUs")
        if s >= 1024 and world < 2:
            raise SystemExit("c5-strong at 1024^3 needs >= 2 GPUs: 18 field buffers of 8.7 GB (out-of-place substeps) "
                             "plus the solver storage exceed one B200; use --size 512 for a one-GPU run")
        shape_l, shape_g, name = (s, s // world, s), (s, s, s), "C5 strong"
    elif cfg == "c5-weak":
        s = a.size or 512
        shape_l, shape_g, name = (s, s, s), (s, s * world, s), "C5 weak"
    else:
        s = a.size or 256
        shape_l, shape_g, name = (s, s, s), (s, s * world, s), "C2"
    grid = ob.RectilinearGrid(arch, FTYPE, size=shape_g, extent=(1, shape_g[1] / shape_g[0], 1), topology=("Periodic",) * 3)
    model = ob.NonhydrostaticModel(grid, advection=ob.WENO5(FTYPE), tracers=("b",), buoyancy=ob.BuoyancyTracer(),
                                   timestepper="RungeKutta3")
    ob.set_model(model, **synthetic_state(shape_l, seed=2 + rank))
    wl = (f"{name}: {shape_g[0]}x{shape_g[1]}x{shape_g[2]} triply-periodic NonhydrostaticModel, WENO5 + tracer b + "
          f"BuoyancyTracer, FFT pressure solve, RK3, " + ("Float64" if FTYPE is np.float64 else "Float32"))
    return model, 0.1 / s, shape_l[0] * shape_l[1] * shape_l[2], shape_g, wl, 4, 110.0


def distributed_parity(ob, np, arch, world, rank):
    """decomposed vs single-domain on the same global initial condition (the logic of tests/dist_check.py without the
    oracle: the single-domain run is THIS library on one GPU, which the GPU test suite pins to the oracle): every rank
    steps the slab-decomposed model AND, on its own GPU, the whole 64 x 16R x 32 domain, and compares its slab."""
    N = (64, max(32, 16 * world), 32)
    L = (1.0, 2.0, 1.5)
    topo = ("Periodic",) * 3
    gd = ob.RectilinearGrid(arch, np.float64, size=N, extent=L, topology=topo)
    gs = ob.RectilinearGrid(arch.child, np.float64, size=N, extent=L, topology=topo)
    mk = lambda g: ob.NonhydrostaticModel(g, advection=ob.WENO5(), tracers=("b",), buoyancy=ob.BuoyancyTracer(),
                                          timestepper="RungeKutta3")
    md, ms = mk(gd), mk(gs)
    rng = np.random.default_rng(5)
    vals = {}
    for n in "uvw":
        x = rng.uniform(-1, 1, N)
        vals[n] = x - x.mean()
    zc = (np.arange(N[2]) + 0.5) / N[2] * L[2] - L[2]
    vals["b"] = 0.5 * zc.reshape(1, 1, -1) + 0.1 * rng.uniform(-1, 1, N)
    sl = gd.local_slice()
    ob.set_model(ms, **vals)
    ob.set_model(md, **{n: v[sl] for n, v in vals.items()})
    worst = 0.0
    for _ in range(3):
        ob.time_step(ms, 2e-3)
        ob.time_step(md, 2e-3)
        for n in ms.names:
            ref = ms.fields[n].interior()
            worst = max(worst, float(np.max(np.abs(md.fields[n].interior() - ref[sl])) / np.max(np.abs(ref))))
    worst = arch.allreduce([worst], "max")[0]
    return {"worst_rel_err": worst, "ranks": world, "global_grid": list(N), "steps": 3, "tolerance": 1e-12,
            "against": "the same library on one GPU, whole domain (pinned to the oracle by tests/test_gpu_parity.py)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--size", type=int, default=0, help="scale the configuration: replaces 256 (c2) / 512 (c3, c5-weak) / 1024")
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c5-weak", "c5-strong"])
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--closure", default="scalar", choices=["scalar", "amd", "smagorinsky"],
                    help="config c3 only: ScalarDiffusivity (BASELINE configs[2]) or the LES closure of its source example")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-dist-parity", action="store_true")
    ap.add_argument("--ftype", default="f64", choices=["f64", "f32"],
                    help="arithmetic type of the run (the headline configuration is Float64; f32 is reported for reference)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the fields computed by the last timed step to DIR/<name>.npy (at most 64 MB in all)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if a.impl == "reference":
        if rank != 0:
            return
        steps, warmup = a.steps, a.warmup
        v, spstep, cores, sample, Ns = cpu_reference_run(steps, warmup, sample_n=a.size or 256)
        workload = (f"C2: {Ns}^3 triply-periodic NonhydrostaticModel, WENO5 + tracer b + BuoyancyTracer, FFT pressure solve, "
                    f"RK3, Float64 (CPU arm: bounded sample of the 256^3 workload; the per-point cost does not depend on N)")
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": spstep * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "grid": [Ns, Ns, Ns], "config": "c2"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import numpy as np
    import torch
    import ocean_b200 as ob
    from ocean_b200._lib import lib
    import ctypes as C

    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.current_stream()
    lib.ob200_set_stream(C.c_void_p(stream.cuda_stream))
    # With several GPUs the GLOBAL domain is slab-decomposed in y (ranks = (1, world, 1) as in the reference's distributed
    # benchmarks): peer-memory / NCCL halo exchange + all-to-all transposes inside the FFT pressure solve (DESIGN.md 6)
    arch = ob.MultiArch.from_torch_distributed(local_rank) if world > 1 else ob.B200(local_rank)
    FTYPE = np.float64 if a.ftype == "f64" else np.float32

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dist_parity = None
    if world > 1 and not a.no_dist_parity:
        dist_parity = distributed_parity(ob, np, arch, world, rank)
        assert dist_parity["worst_rel_err"] <= 1e-12, dist_parity
        barrier()

    model, dt, pts_gpu, shape_g, workload, F, words_step = build_config(ob, np, a, arch, world, rank, FTYPE)

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(a.warmup):
        ob.time_step(model, dt)
    barrier()
    lib.ob200_profile_reset()
    lib.ob200_profile_enable(1)
    n0 = ob.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    ev0.record(stream)
    for _ in range(a.steps):
        ob.time_step(model, dt)
    ev1.record(stream)
    barrier()
    sampler.mark_end()
    ms = ev0.elapsed_time(ev1)
    launches = ob.launch_count() - n0
    lib.ob200_profile_enable(0)
    if a.dump_outputs and rank == 0:
        dump_outputs(model, a.dump_outputs)
    phases = {}
    fft_names = ("fft_x_fwd", "fft_y", "fft_z", "fft_z_fwd", "fft_z_inv", "fft_sync", "fft_x_inv", "fft_y_butterfly",
                 "fft_y_lines", "fft_y_copywait")
    for ph in ("tendency", "poisson", "halo", "pressure_correct", "hydrostatic") + fft_names:
        t, c = C.c_double(), C.c_int64()
        lib.ob200_profile_query(ph.encode(), C.byref(t), C.byref(c))
        phases[ph] = {"ms_total": t.value, "count": c.value}
    fft_phases = {k: phases.pop(k) for k in fft_names}
    if world > 1:
        tt = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    value = world * pts_gpu * a.steps / (ms * 1e-3)
    d = model.diagnostics()
    if world > 1:
        d["max_abs_div"] = arch.allreduce([d["max_abs_div"]], "max")[0]
        d["kinetic_energy"] = arch.allreduce([d["kinetic_energy"]], "sum")[0]
    assert np.isfinite(d["kinetic_energy"]) and d["max_abs_div"] < (1e-8 if a.ftype == "f64" else 1e-1), d

    # ---- roofline of the dominant kernel: tendencies + substep ---------------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    tend = phases["tendency"]
    W = 8 if a.ftype == "f64" else 4
    fused = os.environ.get("OB200_NO_FUSED_TENDENCY") is None and (
        a.config != "c3" or (os.environ.get("OB200_NO_FUSED_BOUNDED") is None and shape_g[0] % 32 == 0 and a.closure == "scalar"))
    # algorithmic words per point: 4F+1 for stages 2,3 and 3F+1 for stage 1 (SURVEY.md 8(d) P1), per stage;
    # the fused kernel does a whole stage per launch, the per-field kernels a F-th of it
    words_stage = ((3 * F + 1) + 2 * (4 * F + 1)) / 3.0
    per_launch = 1 if fused else F
    alg_bytes = words_stage / per_launch * W * pts_gpu
    tend_launches = a.steps * 3 * per_launch
    avg_ms = tend["ms_total"] / max(1, tend_launches)
    achieved = alg_bytes / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
    headline_shape = a.config in ("c2", "c3") and not a.size and a.ftype == "f64" and (fused or a.config == "c2")
    ncu_traffic = (NCU_TRAFFIC_BYTES_PER_FUSED_LAUNCH_C3 if a.config == "c3" else
                   (NCU_TRAFFIC_BYTES_PER_FUSED_LAUNCH if fused else NCU_TRAFFIC_BYTES_PER_FIELD_LAUNCH))
    kname = ("fz::tendency_fused_kernel: tendencies + substep of all prognostic fields, one launch per stage" if fused else
             ("tendency_shared_kernel (general, per prognostic field)" if a.config == "c3"
              else "tma::tendency_tma_kernel (per prognostic field)"))
    roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic if headline_shape else None,
                "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of one launch "
                                  "(profiles/r2_summary.md)" if headline_shape else None,
                "algorithmic_bytes_per_launch": alg_bytes,
                "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback",
                "avg_launch_ms": avg_ms, "launches": tend_launches,
                "share_of_step": tend["ms_total"] / ms if ms > 0 else None,
                "whole_step": {"algorithmic_GB_per_step": words_step * W * pts_gpu / 1e9,
                               "achieved_GBps": words_step * W * pts_gpu * a.steps / (ms * 1e-3) / 1e9,
                               "frac": words_step * W * pts_gpu * a.steps / (ms * 1e-3) / 1e9 / peak},
                "phases_ms_per_step": {k: v["ms_total"] / a.steps for k, v in phases.items()},
                "poisson_ms_per_step": {k: v["ms_total"] / a.steps for k, v in fft_phases.items() if v["count"]}}

    # ---- e2e: host buffers in, host buffers out, every step (pinned; copies inside the timed region) ----
    e2e = None
    if not a.no_e2e:
        names = list(model.names)
        hin = {n: torch.from_numpy(np.asfortranarray(model.fields[n].parent()).ravel(order="K").copy()).pin_memory()
               for n in names}
        # two sets of pinned output buffers: step n writes set n % 2 and the host "consumes" (checksums one value of)
        # set (n - 1) % 2 while the GPU works, as a streaming caller would
        hout = [{n: torch.empty_like(hin[n]).pin_memory() for n in names} for _ in range(2)]
        nbytes = sum(t.numel() * t.element_size() for t in hin.values())
        ksteps = max(4, min(a.steps, 10))

        def enqueue(step):
            """one step through the C ABI with HOST buffers: H2D of the four parent arrays, time_step!, D2H of the
            four parent arrays.  Everything is asynchronous (pinned memory; uploads and downloads run on the library's
            two copy streams), so the upload of the next step and the download of the previous one overlap the kernels."""
            for n in names:
                lib.ob200_field_set_parent_async(model.fields[n].handle, C.c_void_p(hin[n].data_ptr()))
            ob.time_step(model, dt)
            for n in names:
                lib.ob200_field_get_parent_async(model.fields[n].handle, C.c_void_p(hout[step % 2][n].data_ptr()))
            lib.ob200_mark_download_batch()

        def run_pipelined(k):
            acc = 0.0
            for step in range(k):
                if step >= 2:
                    lib.ob200_sync_downloads(1)                 # the set about to be overwritten (step - 2) has been delivered
                    acc += float(hout[step % 2][names[0]][12345])
                enqueue(step)
            lib.ob200_sync()
            return acc
        run_pipelined(2)
        barrier()
        t0 = time.perf_counter()
        run_pipelined(ksteps)
        barrier()
        el = time.perf_counter() - t0
        # the unpipelined variant (one step at a time, synchronised after every step) for comparison
        t0 = time.perf_counter()
        for step in range(2):
            enqueue(step)
            lib.ob200_sync()
        el_serial = (time.perf_counter() - t0) / 2
        if world > 1:
            tt = torch.tensor([el], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            el = float(tt.item())
        # resident-state variant: the call a user of the B200() architecture makes inside run!:
        # time_step!(model, dt) + the per-step scalar diagnostics read back (NaN check / CFL)
        t0 = time.perf_counter()
        for _ in range(ksteps):
            ob.time_step(model, dt)
            model.velocities["u"].reduce()
        barrier()
        el_res = time.perf_counter() - t0
        e2e = {"value": world * pts_gpu * ksteps / el, "unit": UNIT, "h2d_bytes_per_step": nbytes,
               "d2h_bytes_per_step": nbytes, "steps": ksteps,
               "note": "every step: H2D of u,v,w,b parent arrays from pinned host memory, time_step!, D2H of the same; "
                       "copies on two copy streams overlap the kernels of neighbouring steps (PCIe-bound)",
               "one_step_at_a_time": {"value": world * pts_gpu / el_serial,
                                      "note": "same, host synchronises after every step (no overlap)"},
               "resident_state": {"value": world * pts_gpu * ksteps / el_res, "d2h_bytes_per_step": 32,
                                  "note": "state stays on the device (how run! uses the architecture); per step a scalar reduction is read back"}}

    sampler.stop_flag = True
    sampler.join(timeout=2)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        # BASELINE.md section 3: the CPU arm at 256^3 (and 128^3 beside it), bounded to ~20-30 s of CPU work
        v, spstep, cores, sample, Ns = cpu_reference_run(2, 0, sample_n=256, budget_s=40.0)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
        if Ns == 256:
            v2, _, _, sample2, _ = cpu_reference_run(2, 0, sample_n=128, budget_s=20.0)
            cpu["at_128"] = {"value": v2, "sample": sample2}

    if rank == 0:
        par = "single GPU" if world == 1 else (
            f"slab decomposition in y, ranks=(1,{world},1): global grid {shape_g[0]}x{shape_g[1]}x{shape_g[2]}; "
            "peer-memory halo exchange + 2 all-to-all transposes per pressure solve")
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True,
            "scaling": "strong" if a.config == "c5-strong" else "weak", "vs_baseline": None,
            "dtype": a.ftype, "data": "synthetic",
            "config": {"workload": workload, "config": a.config, "grid": list(shape_g), "timestepper": "RungeKutta3",
                       "advection": "WENO5 (Z)", "fields": F, "dt": dt, "ftype": a.ftype,
                       "l2": "inputs larger than L2 (state, tendencies and pressures: 18 buffers, 2.6 GB at 256^3 F64, against 126 MB)",
                       "parallelism": par},
            "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
            "cpu_baseline": cpu}
        if dist_parity is not None:
            out["dist_parity"] = dist_parity
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
