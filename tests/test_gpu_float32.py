"""The Float32 CUDA path against a Float64 reference.  The reference is the oracle in Float64 on exactly what the Float32 model
sees (initial state, stretched faces and boundary arrays rounded to Float32; the same parameters).  The yardstick is the same
case on the oracle in Float32, i.e. a plain Float32 evaluation of the reference's arithmetic.  Every field at every checkpoint
must satisfy

    relerr(CUDA Float32, oracle Float64) <= 4 (relerr(oracle Float32, oracle Float64) + eps32),    eps32 = 2^-23

which follows the conditioning of each case: a Float32-only mistake (a constant or table rounded in the wrong precision, a fast
divide in the wrong place) of a few eps32 fails it, where a fixed 1e-5 would not.  States also keep the absolute 1e-5.

Besides: the Fourier-tridiagonal solve on domains of 100 - 1000 km (its pivot guard is relative to the diagonal; the reference's
absolute 10 eps broke the lowest modes' columns in Float32 there), the batched tridiagonal solver against dense solves, and a
CPU check that the Float32 yardstick really is evaluated in Float32."""
import numpy as np
import pytest
import scipy.linalg

import oracle as O
from test_gpu_bc_arrays import CASES as BC_CASES, build as build_bc, random_arrays
from test_gpu_forcing import CASES as FORCING_CASES, build_forced
from test_gpu_parity import CONFIGS, TOPOS8, _rhs, _zf, build_models, init_state, make_pair, relerr

EPS32 = 2.0 ** -23
FACTOR = 4
STATE_TOL = 1e-5                 # the absolute per-step bound of BASELINE.json


@pytest.fixture(scope="module")
def ob():
    import ocean_b200 as ob
    ob.arch = ob.B200()
    return ob


class _OracleOnly:
    """stands in for the ocean_b200 module in the builders of test_gpu_parity / test_gpu_forcing / test_gpu_bc_arrays, so that
    they build the oracle model alone: device objects become None, the host-side forcing descriptions stay the module's own"""
    def __init__(self, ob=None):
        self.ob = ob
        self.arch = None

    def __getattr__(self, name):
        if name in ("Relaxation", "GaussianMask", "LinearTarget"):
            return getattr(self.ob, name)
        return lambda *a, **k: None


class _Recorder:
    """the `ob` of init_state: keeps the values it would give the CUDA model"""
    def set_model(self, model, **vals):
        self.vals = vals


def f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def rounded(cfg):
    """cfg with its stretched faces rounded to Float32 (intervals and extents are exact in Float32 here)"""
    coords = cfg.get("coords")
    if not coords:
        return cfg
    return dict(cfg, coords={d: f32(v) if isinstance(v, np.ndarray) else v for d, v in coords.items()})


def check(what, cuda, o32, o64, absolute=None):
    e_c, e_o = relerr(cuda, o64), relerr(o32, o64)
    ratio = e_c / (e_o + EPS32)
    print(f"F32 {what}: e_cuda {e_c:.3e} e_o32 {e_o:.3e} ratio {ratio:.3f}")
    assert e_c <= FACTOR * (e_o + EPS32), \
        f"{what}: CUDA Float32 rel err {e_c:.3e} = {ratio:.2f} x (Float32 oracle's {e_o:.3e} + eps32)"
    if absolute is not None:
        assert e_c <= absolute, f"{what}: CUDA Float32 rel err {e_c:.3e} > {absolute:g}"


def run_model_case(ob, what, build, cfg, seed, steps=3, expected_over=()):
    """build(M, cfg, FT) -> (oracle model, M's model).  After set! and the projection: states, pHY′, νₑ / κₑ (halos included);
    then the tendencies; then states and pNHS after each of `steps` steps.  The checks named in `expected_over` ("set/w",
    "G/v", "step1/pNHS", ...) may exceed the relative bound: they are measured and keep any absolute bound, every other check is
    asserted as usual.  Returns {check: ratio to (the Float32 oracle's error + eps32)} of those checks."""
    measured = {}

    def check_(label, cuda, o32, o64, absolute=None):
        if label not in expected_over:
            return check(f"{what}/{label}", cuda, o32, o64, absolute)
        e_c, e_o = relerr(cuda, o64), relerr(o32, o64)
        measured[label] = e_c / (e_o + EPS32)
        print(f"F32 {what}/{label}: e_cuda {e_c:.3e} e_o32 {e_o:.3e} ratio {measured[label]:.3f} (expected over)")
        if absolute is not None:
            assert e_c <= absolute, f"{what}/{label}: CUDA Float32 rel err {e_c:.3e} > {absolute:g}"

    mo32, mb = build(ob, cfg, np.float32)
    mo64, _ = build(_OracleOnly(ob), rounded(cfg), np.float64)
    rec = _Recorder()
    init_state(mo32, None, rec, seed)
    ob.set_model(mb, **rec.vals)
    mo64.set(**{n: v.astype(np.float64) for n, v in rec.vals.items()})

    def states(when):
        for n in mo64.names:
            check_(f"{when}/{n}", mb.fields[n].interior(), mo32.fields[n].interior, mo64.fields[n].interior, STATE_TOL)

    states("set")
    if mo64.pHY is not None:
        check_("set/pHY", mb.pressures["pHY′"].interior(), mo32.pHY.interior, mo64.pHY.interior)
    if getattr(mo64, "νe", None) is not None:
        check_("set/nu_e", mb.diffusivity_fields["νₑ"].parent(), mo32.νe.parent, mo64.νe.parent)
        if getattr(mo64, "κe", None) is not None:
            for n in mo64.tracer_names:
                check_(f"set/kappa_e_{n}", mb.diffusivity_fields["κₑ"][n].parent(), mo32.κe[n].parent, mo64.κe[n].parent)
    mo32.calculate_tendencies()
    mo64.calculate_tendencies()
    ob.calculate_tendencies(mb)
    g = mo64.grid
    ijk = O.R(1, g.Nx), O.R(1, g.Ny), O.R(1, g.Nz)
    for n in mo64.names:
        check_(f"G/{n}", mb.Gn[n].interior()[:g.Nx, :g.Ny, :g.Nz], mo32.Gn[n][ijk], mo64.Gn[n][ijk])
    for step in range(1, steps + 1):
        mo32.time_step(cfg["dt"])
        mo64.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        states(f"step{step}")
        check_(f"step{step}/pNHS", mb.pressures["pNHS"].interior(), mo32.pNHS.interior, mo64.pNHS.interior)
    return measured


# ---- a. every parity configuration ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_configs_float32_against_float64(ob, name):
    run_model_case(ob, f"a/{name}", build_models, CONFIGS[name], 22)


# ---- b. the forcing and boundary-array cases, on their own builders ------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FORCING_CASES))
def test_forced_float32_against_float64(ob, name):
    cfg, forcing = FORCING_CASES[name]
    run_model_case(ob, f"b/forcing/{name}", lambda M, c, FT: build_forced(M, c, FT, forcing), cfg, 62)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BC_CASES))
def test_bc_arrays_float32_against_float64(ob, name):
    cfg, spec, forcing = BC_CASES[name]
    go = make_pair(ob, np.float64, cfg["size"], cfg["topology"], coords=cfg.get("coords"), extent=cfg.get("extent"))[0]
    arrays = {n: {s: (k, f32(Q)) for s, (k, Q) in d.items()} for n, d in random_arrays(go, spec, 73).items()}
    run_model_case(ob, f"b/bc_arrays/{name}", lambda M, c, FT: build_bc(M, c, FT, arrays, forcing), cfg, 74)


# ---- c. fused-kernel shapes: Bounded z (regular and stretched) and triply periodic ---------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("size", [(32, 5, 6), (64, 13, 7), (96, 25, 9), (32, 12, 33), (32, 3, 16)])
@pytest.mark.parametrize("stretched", [True, False])
def test_fused_bounded_z_shapes_float32_against_float64(ob, size, stretched):
    cfg = dict(CONFIGS["c3_fused_stretched_weno_rk3"], size=size)
    if stretched:
        cfg["coords"] = dict(x=(0, 1), y=(0, 1), z=_zf(size[2]))
    else:
        cfg.pop("coords")
        cfg["extent"], cfg["adv"] = (1, 1, 1), "WENO5"
    run_model_case(ob, f"c/bounded/{size}/{'stretched' if stretched else 'regular'}", build_models, cfg, 37)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(32, 5, 6), (64, 13, 7), (96, 25, 9)])
def test_fused_periodic_shapes_float32_against_float64(ob, size):
    run_model_case(ob, f"c/periodic/{size}", build_models, dict(CONFIGS["c2_periodic_weno_rk3"], size=size), 38)


# ---- d. Poisson solvers ----------------------------------------------------------------------------------------------------------
def compatible_rhs(size, zF, seed):
    """uniform noise with its Δz-weighted mean removed (in Float64): the Neumann problem in z is solvable"""
    rhs = np.random.default_rng(seed).uniform(-1, 1, size)
    dz = np.diff(zF).reshape(1, 1, -1)
    return rhs - (rhs * dz).sum() / (dz.sum() * size[0] * size[1])


def solve_ft_three_ways(ob, FT, size, topology, coords, rhs):
    """the Fourier-tridiagonal solve of `rhs` on the CUDA path in FT, on the oracle in Float32 and in Float64, all on the faces
    rounded to Float32.  The Float32 runs see the right-hand side rounded to Float32; the Float64 reference solves the exactly
    compatible one (a rounded right-hand side is compatible only to eps32, and the reference's elimination would divide that
    residual by its noise pivot in the horizontal-mean column)"""
    kw = dict(size=size, topology=topology, **rounded(dict(coords=coords))["coords"])
    out = []
    for M, T in ((ob, FT), (O, np.float32), (O, np.float64)):
        r = rhs.astype(T)
        if M is ob:
            g = ob.RectilinearGrid(ob.arch, FT, **kw)
            p = ob.CenterField(g)
            ob.solve(p, ob.FourierTridiagonalPoissonSolver(g), r)
            out.append(p.interior())
        else:
            g = O.RectilinearGrid(T, **kw)
            p = O.Field(g, auxiliary=True)
            O.FourierTridiagonalPoissonSolver(g).solve(p, r)
            out.append(np.array(p.interior))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("topo", TOPOS8)
@pytest.mark.parametrize("N", [(16, 8, 32), (7, 11, 6), (48, 20, 96), (64, 32, 24)])
def test_fft_poisson_float32_against_float64(ob, topo, N):
    """radix-2, Makhoul DCT, Bluestein and the half-spectrum passes in Float32"""
    go32, gb = make_pair(ob, np.float32, N, topo, extent=(1.0, 2.0, 3.0))
    rhs = _rhs(go32, np.random.default_rng(13))[0].astype(np.float32)
    out = []
    for T in (np.float32, np.float64):
        go = O.RectilinearGrid(T, size=N, topology=topo, extent=(1.0, 2.0, 3.0))
        so, po = O.FFTBasedPoissonSolver(go), O.Field(go, auxiliary=True)
        so.storage[...] = rhs.astype(T)
        so.solve(po)
        out.append(np.array(po.interior))
    pb = ob.CenterField(gb)
    ob.solve(pb, ob.FFTBasedPoissonSolver(gb), rhs)
    check(f"d/fft/{N}/{''.join(t[0] for t in topo)}", pb.interior(), *out)


@pytest.mark.gpu
@pytest.mark.parametrize("topo", [(a, b, O.Bounded) for a in (O.Periodic, O.Bounded) for b in (O.Periodic, O.Bounded)])
def test_fourier_tridiagonal_float32_against_float64(ob, topo):
    rng = np.random.default_rng(15)
    zF = np.concatenate([[0.0], np.cumsum(0.5 + rng.random(12))])
    zF = zF / zF[-1] - 1
    coords = dict(x=(0, 1), y=(0, 2), z=zF)
    out = solve_ft_three_ways(ob, np.float32, (16, 8, 12), topo, coords, compatible_rhs((16, 8, 12), f32(zF), 16))
    check(f"d/ft/{''.join(t[0] for t in topo)}", *out)


@pytest.mark.gpu
@pytest.mark.parametrize("ytopo", [O.Periodic, O.Bounded])
@pytest.mark.parametrize("size", [(32, 16, 12), (64, 32, 20)])
def test_fast_fourier_tridiagonal_float32_against_float64(ob, size, ytopo):
    """half-spectrum x passes, Periodic y lines or the DCT over a Bounded y, Thomas sweep on the half spectrum"""
    coords = dict(x=(0, 1), y=(0, 2), z=_zf(size[2]))
    out = solve_ft_three_ways(ob, np.float32, size, (O.Periodic, ytopo, O.Bounded), coords,
                              compatible_rhs(size, f32(_zf(size[2])), 17))
    check(f"d/ft_fast/{size}/{ytopo[0]}", *out)


# ---- e. the Fourier-tridiagonal solve on large domains ---------------------------------------------------------------------------
LARGE = [((O.Bounded, O.Periodic, O.Bounded), 1e5, 1e3), ((O.Bounded, O.Bounded, O.Bounded), 1e5, 1e3),
         ((O.Periodic, O.Periodic, O.Bounded), 1e6, 4e3)]


@pytest.mark.gpu
@pytest.mark.parametrize("FT,tol", [(np.float32, 3e-3), (np.float64, 1e-10)])
@pytest.mark.parametrize("size", [(16, 8, 12), (32, 16, 12)])
@pytest.mark.parametrize("topo,Lx,H", LARGE)
def test_fourier_tridiagonal_large_domains(ob, topo, Lx, H, size, FT, tol):
    """Lx x Lx/2 x H with stretched z: the lowest horizontal modes' last pivot is about λ H ~ (π / Lx)² H, below the
    reference's absolute guard 10 eps(Float32) from Lx ~ 100 km on, and the broken columns gave 0.3 - 0.85.  The guard here is
    relative to the diagonal; what is left in Float32 is the conditioning of those modes, 3e-4 - 7.5e-4 on a B200 (the bound is
    4x that).  (32, 16, 12) on (P, P, B) takes the half-spectrum path."""
    zF = H * _zf(size[2])
    coords = dict(x=(0, Lx), y=(0, Lx / 2), z=zF)
    cuda, _, o64 = solve_ft_three_ways(ob, FT, size, topo, coords, compatible_rhs(size, f32(zF), 1))
    e = relerr(cuda, o64)
    print(f"F32 e/{''.join(t[0] for t in topo)}/{size}/{FT.__name__}: rel err {e:.3e}")
    assert e <= tol, e


# ---- f. the batched tridiagonal solver ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("Nz", [1, 2, 9, 64])
def test_batched_tridiagonal_float32_against_dense(ob, Nz, cplx):
    """the user-facing solver (caller's coefficients, the reference's absolute pivot guard) against dense Float64 solves of the
    same Float32 right-hand side, with the oracle's Float32 sweep as the yardstick"""
    rng = np.random.default_rng(16 + Nz)
    Nx, Ny = 5, 4
    _, gb = make_pair(ob, np.float32, (Nx, Ny, Nz), (O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1))
    go = O.RectilinearGrid(np.float32, size=(Nx, Ny, Nz), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1))
    a, c = rng.uniform(-1, 1, Nz - 1), rng.uniform(-1, 1, Nz - 1)
    b = 2.5 + rng.random((Nx, Ny, Nz))
    f = rng.uniform(-1, 1, (Nx, Ny, Nz)) + (1j * rng.uniform(-1, 1, (Nx, Ny, Nz)) if cplx else 0)
    f = f.astype(np.complex64 if cplx else np.float32)
    cuda = ob.BatchedTridiagonalSolver(gb, a, b, c).solve(f)
    o32 = O.BatchedTridiagonalSolver(go, a, b, c).solve(np.zeros_like(f), f)
    dense = np.empty((Nx, Ny, Nz), dtype=np.complex128 if cplx else np.float64)
    for i in range(Nx):
        for j in range(Ny):
            dense[i, j] = np.linalg.solve(np.diag(b[i, j]) + np.diag(a, -1) + np.diag(c, 1), f[i, j].astype(dense.dtype))
    assert cuda.dtype == f.dtype
    if cplx:
        check(f"f/Nz{Nz}/re", cuda.real, o32.real, dense.real)
        check(f"f/Nz{Nz}/im", cuda.imag, o32.imag, dense.imag)
    else:
        check(f"f/Nz{Nz}", cuda, o32, dense)


# ---- the yardstick is real Float32 (CPU) ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["c2_periodic_weno_rk3", "c3_stretched_weno_rk3"])
def test_float32_oracle_is_evaluated_in_float32(name):
    """if a promotion rule or an oracle change evaluated the "Float32" oracle in Float64, the bound above would collapse to
    4 eps32 without anyone noticing"""
    cfg = CONFIGS[name]
    mo32, _ = build_models(_OracleOnly(), cfg, np.float32)
    mo64, _ = build_models(_OracleOnly(), rounded(cfg), np.float64)
    rec = _Recorder()
    init_state(mo32, None, rec, 22)
    mo64.set(**{n: v.astype(np.float64) for n, v in rec.vals.items()})
    mo32.calculate_tendencies()
    mo64.calculate_tendencies()
    mo32.time_step(cfg["dt"])
    mo64.time_step(cfg["dt"])
    g = mo64.grid
    ijk = O.R(1, g.Nx), O.R(1, g.Ny), O.R(1, g.Nz)
    for n in mo64.names:
        assert mo32.fields[n].parent.dtype == np.float32 and mo32.Gn[n].parent.dtype == np.float32, n
        assert relerr(mo32.Gn[n][ijk], mo64.Gn[n][ijk]) > 1e-8, f"tendency {n}"
        assert relerr(mo32.fields[n].interior, mo64.fields[n].interior) > 1e-8, n


def test_float32_oracle_poisson_solve_is_evaluated_in_float32():
    size, zF = (16, 8, 12), f32(_zf(12))
    rhs = compatible_rhs(size, zF, 1)
    out = []
    for T in (np.float32, np.float64):
        g = O.RectilinearGrid(T, size=size, topology=(O.Periodic, O.Periodic, O.Bounded), x=(0, 1), y=(0, 2), z=zF)
        p = O.Field(g, auxiliary=True)
        O.FourierTridiagonalPoissonSolver(g).solve(p, rhs.astype(T))
        out.append(p.interior)
    assert out[0].dtype == np.float32
    assert relerr(out[0], out[1]) > 1e-8
