"""GPU: the CUDA path (through the C ABI) against the committed golden vectors (tests/golden/*.npz) and, at sizes that
take the SPECIALISED kernels of the headline path (TMA-staged tendency kernels, fast FFT solver, fused periodic
stage), against the live oracle.  Float64 <= 1e-12, Float32 <= 1e-5 per step (BASELINE.json)."""
import os

import numpy as np
import pytest

import oracle as O
from golden_cases import MODEL_CASES, POISSON_CASES, build_model, build_oracle_model, model_initial_values, poisson_rhs

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ob():
    import ocean_b200 as ob
    ob.arch = ob.B200()
    return ob


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.mark.parametrize("name", list(MODEL_CASES))
def test_cuda_path_reproduces_golden_model_steps(ob, name):
    cfg = MODEL_CASES[name]
    gold = np.load(os.path.join(GOLD, f"model_{name}.npz"))
    mo = build_oracle_model(O, cfg)                       # only for the seeded initial values
    vals = model_initial_values(mo, cfg["seed"])
    mb = build_model(ob, ob.RectilinearGrid(ob.arch, np.float64, **cfg["grid"]), cfg)
    ob.set_model(mb, **vals)
    for step in range(cfg["steps"]):
        ob.time_step(mb, cfg["dt"])
        if step == 0:
            for n in mb.names:
                assert rel(mb.fields[n].interior(), gold[f"step1_{n}"]) < 1e-12, (name, n)
    for n in mb.names:
        assert rel(mb.fields[n].interior(), gold[f"final_{n}"]) < 1e-12, (name, n)
    ke = mb.diagnostics()["kinetic_energy"]
    assert abs(ke - float(gold["kinetic_energy"])) <= 1e-11 * abs(float(gold["kinetic_energy"]))


@pytest.mark.parametrize("name", list(POISSON_CASES))
def test_cuda_path_reproduces_golden_poisson(ob, name):
    cfg = POISSON_CASES[name]
    gold = np.load(os.path.join(GOLD, f"poisson_{name}.npz"))["phi"]
    go = O.RectilinearGrid(np.float64, **cfg["grid"])
    gb = ob.RectilinearGrid(ob.arch, np.float64, **cfg["grid"])
    rhs = poisson_rhs(go, cfg["seed"])
    phi = ob.CenterField(gb)
    solver = (ob.FourierTridiagonalPoissonSolver if cfg["solver"] == "ft" else ob.FFTBasedPoissonSolver)(gb)
    ob.solve(phi, solver, rhs)
    assert rel(phi.interior(), gold) < 1e-11


# ---- the specialised kernels of the headline path, at sizes the oracle finishes in seconds ---------------------
# (all Periodic -> fused tendency kernel for u, v, w and the first tracer, fused stage with wrap-around reads and the
# shell fill; power-of-two sizes -> fast FFT + TMA line passes; Nx % 32 == 0 and Ny % 8 == 0 -> tendency_tma_kernel for
# the tracers beyond the first).  Ny = 20 and 9 give ragged last tiles in y.
FAST_CASES = {
    "rk3_zweno": dict(size=(32, 16, 16), ts="RungeKutta3", zweno=True, f=None, steps=3),
    "rk3_zweno_ragged": dict(size=(64, 20, 8), ts="RungeKutta3", zweno=True, f=None, steps=2),
    "ab2_fplane": dict(size=(32, 9, 16), ts="QuasiAdamsBashforth2", zweno=True, f=0.7, steps=3),
    "rk3_js": dict(size=(32, 8, 32), ts="RungeKutta3", zweno=False, f=None, steps=2),
    # field counts of the fused tendency kernel: no tracer, two tracers, and a third one (stepped by the per-field kernel)
    "rk3_no_tracer": dict(size=(32, 20, 16), ts="RungeKutta3", zweno=True, f=0.3, steps=2, tracers=()),
    "rk3_two_tracers": dict(size=(32, 12, 16), ts="RungeKutta3", zweno=True, f=None, steps=2, tracers=("b", "c")),
    "ab2_three_tracers": dict(size=(64, 9, 8), ts="QuasiAdamsBashforth2", zweno=True, f=0.5, steps=2,
                              tracers=("b", "c", "d")),
    # c and d on the per-field TMA kernel (Ny % 8 == 0), in both weight kinds and substep modes
    "rk3_three_tracers_tma": dict(size=(32, 16, 16), ts="RungeKutta3", zweno=True, f=None, steps=2,
                                  tracers=("b", "c", "d")),
    "ab2_js_fplane_three_tracers_tma": dict(size=(32, 16, 16), ts="QuasiAdamsBashforth2", zweno=False, f=0.5, steps=2,
                                            tracers=("b", "c", "d")),
}


def _fast_pair(ob, cfg, FT):
    kw = dict(size=cfg["size"], extent=(1.0, 1.5, 0.75), topology=("Periodic",) * 3)
    go, gb = O.RectilinearGrid(FT, **kw), ob.RectilinearGrid(ob.arch, FT, **kw)
    tracers = cfg.get("tracers", ("b",))
    mk = lambda M, g: M.NonhydrostaticModel(
        g, advection=M.WENO5(FT, zweno=cfg["zweno"]), tracers=tracers,
        buoyancy=M.Buoyancy(M.BuoyancyTracer(), None) if "b" in tracers else None,
        coriolis=M.FPlane(cfg["f"]) if cfg["f"] else None, timestepper=cfg["ts"])
    return mk(O, go), mk(ob, gb)


@pytest.mark.parametrize("FT,tol", [(np.float64, 1e-12), (np.float32, 1e-5)])
@pytest.mark.parametrize("name", list(FAST_CASES))
def test_specialised_kernels_match_oracle(ob, name, FT, tol):
    cfg = FAST_CASES[name]
    mo, mb = _fast_pair(ob, cfg, FT)
    vals = {n: v.astype(FT) for n, v in model_initial_values(mo, 77).items()}
    mo.set(**vals)
    ob.set_model(mb, **vals)
    dt = 2e-3
    for step in range(cfg["steps"]):
        mo.time_step(dt)
        ob.time_step(mb, dt)
        for n in mo.names:
            assert rel(mb.fields[n].interior(), mo.fields[n].interior) < tol, (name, step, n)
    # halos after the step are the periodic images (shell fill), bit for bit
    for n in mo.names:
        p = mb.fields[n].parent()
        Nx, Ny, Nz = cfg["size"]
        H = 3
        assert np.array_equal(p[:H], p[Nx:Nx + H]) and np.array_equal(p[Nx + H:], p[H:2 * H])
        assert np.array_equal(p[:, :H], p[:, Ny:Ny + H]) and np.array_equal(p[:, :, Nz + H:], p[:, :, H:2 * H])


def test_specialised_and_general_kernels_agree(ob):
    """same state through the specialised kernels and through the general ones (use_fast_kernels(False))"""
    cfg = FAST_CASES["rk3_zweno_ragged"]
    mo, m1 = _fast_pair(ob, cfg, np.float64)
    _, m2 = _fast_pair(ob, cfg, np.float64)
    m2.use_fast_kernels(False)
    vals = model_initial_values(mo, 78)
    ob.set_model(m1, **vals)
    ob.set_model(m2, **vals)
    for _ in range(2):
        ob.time_step(m1, 2e-3)
        ob.time_step(m2, 2e-3)
    for n in m1.names:
        assert rel(m1.fields[n].interior(), m2.fields[n].interior()) < 1e-13


# ---- fast Fourier-tridiagonal solve (half-spectrum x / y passes + Thomas sweep on the half spectrum) ------------
def _zf(n, p=1.5):
    return -np.linspace(1, 0, n + 1) ** p


@pytest.mark.parametrize("ytopo", ["Periodic", "Bounded"])
@pytest.mark.parametrize("size", [(32, 16, 12), (64, 32, 20)])
def test_fast_fourier_tridiagonal_matches_oracle(ob, size, ytopo):
    """half-spectrum x passes, Periodic y lines or the DCT over a Bounded y (channel), Thomas sweep on the half spectrum"""
    kw = dict(size=size, x=(0, 1), y=(0, 2), z=_zf(size[2]), topology=("Periodic", ytopo, "Bounded"))
    go, gb = O.RectilinearGrid(np.float64, **kw), ob.RectilinearGrid(ob.arch, np.float64, **kw)
    rhs = poisson_rhs(go, 301)
    po = O.Field(go, auxiliary=True)
    O.FourierTridiagonalPoissonSolver(go).solve(po, rhs)
    pb = ob.CenterField(gb)
    ob.solve(pb, ob.FourierTridiagonalPoissonSolver(gb), rhs)
    assert rel(pb.interior(), po.interior) < 1e-11


@pytest.mark.parametrize("FT,tol", [(np.float64, 1e-12), (np.float32, 2e-5)])
def test_c3_physics_with_fast_tridiagonal_solver(ob, FT, tol):
    """config 3 physics (stretched Bounded z, WENO5(grid), closure, FPlane, flux / gradient BCs) at a size whose pressure
    solve takes the fast Fourier-tridiagonal path (Nx >= 32, Ny >= 16 powers of two)"""
    cfg = dict(MODEL_CASES["c3_stretched_weno_rk3"])
    cfg["grid"] = dict(size=(32, 16, 14), x=(0, 1), y=(0, 1), z=_zf(14), topology=("Periodic", "Periodic", "Bounded"))
    go, gb = O.RectilinearGrid(FT, **cfg["grid"]), ob.RectilinearGrid(ob.arch, FT, **cfg["grid"])
    mo, mb = build_model(O, go, cfg), build_model(ob, gb, cfg)
    vals = {n: v.astype(FT) for n, v in model_initial_values(mo, 104).items()}
    mo.set(**vals)
    ob.set_model(mb, **vals)
    for step in range(3):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        for n in mo.names:
            assert rel(mb.fields[n].interior(), mo.fields[n].interior) < tol, (step, n)
    assert mb.diagnostics()["max_abs_div"] < (1e-12 if FT == np.float64 else 1e-4)


def test_async_parent_transfers_round_trip_and_pipeline(ob):
    """ob200_field_{set,get}_parent_async + ob200_mark_download_batch / ob200_sync_downloads: uploads and downloads on
    the copy streams deliver exactly what the synchronous calls deliver, also when several batches are in flight"""
    import ctypes as C
    from ocean_b200._lib import lib
    g = ob.RectilinearGrid(ob.arch, np.float64, size=(32, 16, 8), extent=(1, 1, 1), topology=("Periodic",) * 3)
    f = ob.CenterField(g)
    rng = np.random.default_rng(9)
    shape = f.parent_size
    outs = []
    for step in range(4):
        a = np.asfortranarray(rng.random(shape))
        out = np.zeros(shape, order="F")
        assert lib.ob200_field_set_parent_async(f.handle, a.ctypes.data_as(C.c_void_p)) == 0
        assert lib.ob200_field_get_parent_async(f.handle, out.ctypes.data_as(C.c_void_p)) == 0
        assert lib.ob200_mark_download_batch() == 0
        outs.append((a, out))
        if step >= 2:
            assert lib.ob200_sync_downloads(1) == 0            # everything but the newest batch has arrived
            assert np.array_equal(outs[step - 1][0], outs[step - 1][1])
    assert lib.ob200_sync() == 0
    for a, out in outs:
        assert np.array_equal(a, out)
    assert np.array_equal(f.parent(), outs[-1][0])


def test_full_size_256_step_matches_compiled_oracle(ob):
    """BASELINE.json configs[1] AT ITS FULL SIZE (256^3, triply periodic, WENO5 + b, FFT solve, RK3, Float64): one full
    time step of the CUDA path against the compiled OpenMP twin of the oracle (oracle/oracle_cpu.c, itself pinned to
    the NumPy oracle and the golden vectors by tests/test_golden_oracle.py), every prognostic field <= 1e-12."""
    from oracle import cpu_twin
    N = 256
    rng = np.random.default_rng(2)
    vals = {}
    for n in "uvw":
        a = rng.uniform(-1, 1, (N, N, N))
        vals[n] = a - a.mean()
    z = (np.arange(N) + 0.5) / N
    vals["b"] = 1e-5 * z.reshape(1, 1, N) + 1e-3 * rng.uniform(-1, 1, (N, N, N))
    gb = ob.RectilinearGrid(ob.arch, np.float64, size=(N, N, N), extent=(1, 1, 1), topology=("Periodic",) * 3)
    mb = ob.NonhydrostaticModel(gb, advection=ob.WENO5(), tracers=("b",), buoyancy=ob.BuoyancyTracer(),
                                timestepper="RungeKutta3")
    ob.set_model(mb, **vals)
    dt = 0.1 / N
    ob.time_step(mb, dt)
    ref = cpu_twin.rk3_run((N, N, N), (1.0, 1.0, 1.0), vals["u"], vals["v"], vals["w"], vals["b"], 1, dt, project=True,
                           nthreads=len(__import__("os").sched_getaffinity(0)))
    for n, r in zip("uvwb", ref):
        assert rel(mb.fields[n].interior(), r) < 1e-12, n
