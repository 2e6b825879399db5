"""GPU parity tests: the CUDA path, called through the C ABI (via the ctypes host mirror), against
the oracle on identical seeded inputs.  Tolerances are BASELINE.json's: max relative error per
step <= 1e-12 in Float64 and <= 1e-5 in Float32 (relative to the field's max magnitude)."""
import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu

TOL = {np.float64: 1e-12, np.float32: 1e-5}


@pytest.fixture(scope="module")
def ob():
    import ocean_b200 as ob
    ob.arch = ob.B200()
    return ob


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = max(np.max(np.abs(b)), 1e-300)
    return float(np.max(np.abs(a - b)) / scale)


def make_pair(ob, FT, size, topology, coords=None, extent=None, halo=None):
    kw = dict(size=size, topology=topology)
    if extent is not None:
        kw["extent"] = extent
    if coords:
        kw.update(coords)
    if halo is not None:
        kw["halo"] = halo
    return O.RectilinearGrid(FT, **kw), ob.RectilinearGrid(ob.arch, FT, **kw)


LOCS = [("f", "c", "c"), ("c", "f", "c"), ("c", "c", "f"), ("c", "c", "c")]
LMAP = {"c": "Center", "f": "Face"}


# ---- halos -----------------------------------------------------------------------------------
@pytest.mark.parametrize("topo", [(O.Periodic, O.Periodic, O.Periodic), (O.Periodic, O.Periodic, O.Bounded),
                                  (O.Bounded, O.Periodic, O.Bounded), (O.Bounded, O.Bounded, O.Bounded),
                                  (O.Periodic, O.Bounded, O.Flat)])
@pytest.mark.parametrize("FT", [np.float64, np.float32])
def test_fill_halo_regions_bit_exact(ob, topo, FT):
    rng = np.random.default_rng(11)
    size = tuple(n for n, t in zip((9, 6, 5), topo) if t != O.Flat)
    halo = tuple(h for h, t in zip((3, 2, 1), topo) if t != O.Flat)
    go, gb = make_pair(ob, FT, size, topo, extent=tuple(1.0 for _ in size), halo=halo)
    fo_list, fb_list = [], []
    for loc in LOCS:
        fo = O.Field(go, loc)
        fb = ob.Field(tuple(LMAP[l] for l in loc), gb)
        assert fb.parent_size == fo.parent.shape
        a = rng.random(fo.parent.shape).astype(FT)
        fo.parent[...] = a
        fb.set_parent(a)
        assert np.array_equal(fb.parent(), a)           # layout round trip
        fo_list.append(fo), fb_list.append(fb)
    O.fill_halo_regions(fo_list)
    ob.fill_halo_regions(fb_list)
    for fo, fb in zip(fo_list, fb_list):
        assert np.array_equal(fb.parent(), fo.parent)


def test_fill_halo_value_gradient_bcs(ob):
    rng = np.random.default_rng(12)
    zF = -np.linspace(1, 0, 8) ** 1.5
    topo = (O.Periodic, O.Periodic, O.Bounded)
    go, gb = make_pair(ob, np.float64, (6, 5, 7), topo, coords=dict(x=(0, 1), y=(0, 1), z=zF))
    bo = O.FieldBoundaryConditions(go, ("c", "c", "c"), top=O.BoundaryCondition("Value", 2.0),
                                   bottom=O.BoundaryCondition("Gradient", -0.5))
    fo = O.Field(go, ("c", "c", "c"), bo)
    fb = ob.CenterField(gb, dict(top=ob.ValueBoundaryCondition(2.0), bottom=ob.GradientBoundaryCondition(-0.5)))
    a = rng.random(fo.parent.shape)
    fo.parent[...] = a
    fb.set_parent(a)
    O.fill_halo_regions(fo)
    ob.fill_halo_regions(fb)
    assert relerr(fb.parent(), fo.parent) < 1e-15


# ---- Poisson solvers ---------------------------------------------------------------------------
def _rhs(go, rng):
    u, v, w = O.Field(go, LOCS[0]), O.Field(go, LOCS[1]), O.Field(go, LOCS[2])
    for f in (u, v, w):
        f.set(rng.random(f.size()))
    O.fill_halo_regions([u, v, w])
    i, j, k = O.R(1, go.Nx), O.R(1, go.Ny), O.R(1, go.Nz)
    from oracle.operators import div_ccc
    return np.array(div_ccc(i, j, k, go, u, v, w)), (u, v, w)


TOPOS8 = [(a, b, c) for a in (O.Periodic, O.Bounded) for b in (O.Periodic, O.Bounded) for c in (O.Periodic, O.Bounded)]


@pytest.mark.parametrize("topo", TOPOS8)
@pytest.mark.parametrize("N", [(16, 8, 32), (7, 11, 6), (48, 20, 96), (32, 16, 16), (64, 32, 24)])
def test_fft_poisson_matches_oracle_and_laplacian(ob, topo, N):
    """power-of-two lengths: radix-2 butterflies (Periodic) / Makhoul's DCT around them (Bounded); other lengths: Bluestein; the
    last two sizes take the half-spectrum x passes when x is Periodic and y a power of two (y Periodic or Bounded, any z)"""
    rng = np.random.default_rng(13)
    go, gb = make_pair(ob, np.float64, N, topo, extent=(1.0, 2.0, 3.0))
    rhs, _ = _rhs(go, rng)
    so = O.FFTBasedPoissonSolver(go)
    ϕo = O.Field(go, auxiliary=True)
    so.storage[...] = rhs
    so.solve(ϕo)
    sb = ob.FFTBasedPoissonSolver(gb)
    ϕb = ob.CenterField(gb)
    ob.solve(ϕb, sb, rhs)
    assert relerr(ϕb.interior(), ϕo.interior) < 1e-12
    # reference's own check: lap(phi) == rhs (test/dependencies_for_poisson_solvers.jl:86-104)
    ob.fill_halo_regions(ϕb)
    ϕo.parent[...] = ϕb.parent()
    from oracle.operators import laplacian_ccc
    lap = laplacian_ccc(O.R(1, go.Nx), O.R(1, go.Ny), O.R(1, go.Nz), go, ϕo)
    assert np.linalg.norm(lap - rhs) <= 1e-8 * np.linalg.norm(rhs)


@pytest.mark.parametrize("N,topo", [((32, 16, 16), (O.Periodic,) * 3), ((64, 32, 128), (O.Periodic,) * 3),
                                    ((128, 64, 32), (O.Periodic,) * 3), ((32, 256, 16), (O.Periodic,) * 3),
                                    ((64, 16, 512), (O.Periodic,) * 3),
                                    ((64, 32), (O.Periodic, O.Periodic, O.Flat))])
@pytest.mark.parametrize("FT", [np.float64, np.float32])
def test_fast_fft_path_matches_oracle(ob, N, topo, FT):
    """power-of-two periodic sizes take the half-spectrum / register-radix path (fft_fast.cu)"""
    rng = np.random.default_rng(17)
    go, gb = make_pair(ob, FT, N, topo, extent=tuple(1.0 + 0.5 * d for d in range(len(N))))
    rhs, _ = _rhs(go, rng)
    so = O.FFTBasedPoissonSolver(go)
    ϕo = O.Field(go, auxiliary=True)
    so.storage[...] = rhs
    so.solve(ϕo)
    ϕb = ob.CenterField(gb)
    ob.solve(ϕb, ob.FFTBasedPoissonSolver(gb), rhs)
    assert relerr(ϕb.interior(), ϕo.interior) < (1e-12 if FT == np.float64 else 2e-5)
    # periodic x halos are written by the last pass itself
    p = ϕb.parent()
    H = gb.Hx
    assert np.array_equal(p[:H, H:-H or None], p[N[0]:N[0] + H, H:-H or None])


def test_fast_fft_solve_for_pressure_fused_divergence(ob):
    """solve_for_pressure! with the divergence fused into the first FFT pass vs the oracle"""
    rng = np.random.default_rng(18)
    go, gb = make_pair(ob, np.float64, (32, 32, 16), (O.Periodic,) * 3, extent=(1.0, 2.0, 0.5))
    rhs, (u, v, w) = _rhs(go, rng)
    dt = 0.37
    so = O.FFTBasedPoissonSolver(go)
    ϕo = O.Field(go, auxiliary=True)
    so.storage[...] = rhs / dt
    so.solve(ϕo)
    U = {}
    for n, f, loc in (("u", u, ("Face", "Center", "Center")), ("v", v, ("Center", "Face", "Center")),
                      ("w", w, ("Center", "Center", "Face"))):
        U[n] = ob.Field(loc, gb)
        U[n].set_parent(f.parent)
    ϕb = ob.CenterField(gb)
    ob.solve_for_pressure(ϕb, ob.FFTBasedPoissonSolver(gb), dt, U)
    assert relerr(ϕb.interior(), ϕo.interior) < 1e-12


def test_fft_poisson_float32_flat(ob):
    rng = np.random.default_rng(14)
    go, gb = make_pair(ob, np.float32, (32, 16), (O.Periodic, O.Bounded, O.Flat), extent=(1.0, 1.0))
    rhs, _ = _rhs(go, rng)
    so = O.FFTBasedPoissonSolver(go)
    ϕo = O.Field(go, auxiliary=True)
    so.storage[...] = rhs
    so.solve(ϕo)
    ϕb = ob.CenterField(gb)
    ob.solve(ϕb, ob.FFTBasedPoissonSolver(gb), rhs)
    assert relerr(ϕb.interior(), ϕo.interior) < 1e-5


@pytest.mark.parametrize("topo", [(a, b, O.Bounded) for a in (O.Periodic, O.Bounded) for b in (O.Periodic, O.Bounded)])
def test_fourier_tridiagonal_matches_oracle(ob, topo):
    rng = np.random.default_rng(15)
    zF = np.concatenate([[0.0], np.cumsum(0.5 + rng.random(12))])
    zF = zF / zF[-1] - 1
    go, gb = make_pair(ob, np.float64, (16, 8, 12), topo, coords=dict(x=(0, 1), y=(0, 2), z=zF))
    rhs, _ = _rhs(go, rng)
    ϕo = O.Field(go, auxiliary=True)
    O.FourierTridiagonalPoissonSolver(go).solve(ϕo, rhs)
    ϕb = ob.CenterField(gb)
    ob.solve(ϕb, ob.FourierTridiagonalPoissonSolver(gb), rhs)
    assert relerr(ϕb.interior(), ϕo.interior) < 1e-11


def test_batched_tridiagonal_vs_dense(ob):
    rng = np.random.default_rng(16)
    Nx, Ny, Nz = 5, 4, 9
    _, gb = make_pair(ob, np.float64, (Nx, Ny, Nz), (O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1))
    a, c = rng.random(Nz - 1), rng.random(Nz - 1)
    b = 3 + rng.random((Nx, Ny, Nz))
    f = rng.random((Nx, Ny, Nz)) + 1j * rng.random((Nx, Ny, Nz))
    ϕ = ob.BatchedTridiagonalSolver(gb, a, b, c).solve(f)
    for i in range(Nx):
        for j in range(Ny):
            M = np.diag(b[i, j]) + np.diag(a, -1) + np.diag(c, 1)
            assert np.allclose(np.linalg.solve(M, f[i, j]), ϕ[i, j], rtol=1e-12)


# ---- model configurations ------------------------------------------------------------------------
def _zf(n, p=1.5):
    return -np.linspace(1, 0, n + 1) ** p


CONFIGS = {
    # headline physics at a small size: triply periodic, WENO5, buoyancy tracer, RK3
    "c2_periodic_weno_rk3": dict(size=(16, 12, 10), topology=(O.Periodic,) * 3, extent=(1, 1, 1),
                                 adv="WENO5", tracers=("b",), buoyancy=True, ts="RungeKutta3", dt=2e-3),
    "periodic_weno_closure_fplane_ab2": dict(size=(12, 16, 8), topology=(O.Periodic,) * 3, extent=(1, 2, 1),
                                             adv="WENO5", tracers=("b", "c"), buoyancy=True, closure=("ThreeDimensional", 1e-3, 2e-3),
                                             f=0.7, ts="QuasiAdamsBashforth2", dt=2e-3),
    # config 1 physics: 2-D periodic turbulence, Flat z, AB2 (README example)
    "c1_2d_flat_weno_ab2": dict(size=(32, 24), topology=(O.Periodic, O.Periodic, O.Flat), extent=(2 * np.pi, 2 * np.pi),
                                adv="WENO5", tracers=(), buoyancy=False, ts="QuasiAdamsBashforth2", dt=5e-3),
    # config 3 physics: bounded stretched z, WENO5(grid), Fourier-tridiagonal, flux/gradient BCs
    "c3_stretched_weno_rk3": dict(size=(12, 8, 14), topology=(O.Periodic, O.Periodic, O.Bounded),
                                  coords=dict(x=(0, 1), y=(0, 1), z=_zf(14)), adv="WENO5grid", tracers=("b",),
                                  buoyancy=True, closure=("ThreeDimensional", 1e-4, 1e-4), f=1e-2, ts="RungeKutta3", dt=5e-3,
                                  bcs={"u": {"top": ("Flux", -1e-3)}, "b": {"top": ("Flux", 1e-4), "bottom": ("Gradient", 1e-2)}}),
    # the same physics on the fused persistent kernel (Nx a multiple of 32; tendency_fused.cu, Bounded-z variant): rows per
    # tile 12 against Ny = 16 (a partial tile); JS weights + AB2 + no closure + no Coriolis; value / gradient BCs on u, v
    "c3_fused_stretched_weno_rk3": dict(size=(32, 16, 14), topology=(O.Periodic, O.Periodic, O.Bounded),
                                        coords=dict(x=(0, 1), y=(0, 1), z=_zf(14)), adv="WENO5grid", tracers=("b",),
                                        buoyancy=True, closure=("ThreeDimensional", 1e-4, 2e-4), f=1e-2, ts="RungeKutta3", dt=5e-3,
                                        bcs={"u": {"top": ("Flux", -1e-3)},
                                             "b": {"top": ("Flux", 1e-4), "bottom": ("Gradient", 1e-2)}}),
    "c3_fused_js_ab2_no_closure": dict(size=(32, 12, 8), topology=(O.Periodic, O.Periodic, O.Bounded),
                                       coords=dict(x=(0, 2), y=(0, 1), z=_zf(8)), adv="WENO5grid_js", tracers=("b", "c"),
                                       buoyancy=True, ts="QuasiAdamsBashforth2", dt=5e-3,
                                       bcs={"v": {"top": ("Value", 0.1), "bottom": ("Gradient", -0.2)},
                                            "b": {"bottom": ("Flux", -2e-4)}, "c": {"top": ("Flux", 3e-4)}}),
    # regular Bounded z, the usual horizontally periodic LES box: fused Bounded-z kernel with the uniform coefficients in table
    # form, FFT-based solver with the half-spectrum x / y passes around a Makhoul DCT in z (Nz = 16) / Bluestein inside it (12)
    "ppb_regular_fused_weno_rk3": dict(size=(32, 16, 16), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(2, 1, 1),
                                       adv="WENO5", tracers=("b",), buoyancy=True, closure=("ThreeDimensional", 2e-4, 1e-4),
                                       f=1e-2, ts="RungeKutta3", dt=4e-3,
                                       bcs={"u": {"top": ("Flux", -1e-3)}, "b": {"bottom": ("Flux", -1e-4)}}),
    "ppb_regular_fused_nz12_ab2": dict(size=(32, 16, 12), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 0.5),
                                       adv="WENO5", tracers=("b",), buoyancy=True, ts="QuasiAdamsBashforth2", dt=4e-3),
    # closures the fused kernel does not evaluate itself: their flux divergence alone goes through the general shared-face kernel
    # into G^n, the fused kernel adds advection, Coriolis, pressure gradient, BC fluxes and the substep
    "amd_c3_fused_split": dict(size=(32, 16, 14), topology=(O.Periodic, O.Periodic, O.Bounded),
                               coords=dict(x=(0, 1), y=(0, 1), z=_zf(14)), adv="WENO5grid", tracers=("b",), buoyancy=True,
                               amd=dict(Cb=1.0), f=1e-2, ts="RungeKutta3", dt=5e-3,
                               bcs={"u": {"top": ("Flux", -1e-3)}, "b": {"top": ("Flux", 1e-4), "bottom": ("Gradient", 1e-2)}}),
    "smagorinsky_ppb_fused_split_ab2": dict(size=(32, 16, 16), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(2, 1, 1),
                                            adv="WENO5", tracers=("b", "c"), buoyancy=True, smagorinsky={}, ts="QuasiAdamsBashforth2",
                                            dt=4e-3, bcs={"b": {"bottom": ("Flux", -1e-4)}}),
    "scalar3d_periodic_fused_split": dict(size=(32, 12, 16), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5",
                                          tracers=("b",), buoyancy=True, closure=("ThreeDimensional", 1e-3, 2e-3), f=0.3,
                                          ts="RungeKutta3", dt=2e-3),
    "channel_bounded_yz_weno": dict(size=(8, 12, 10), topology=(O.Periodic, O.Bounded, O.Bounded), extent=(1, 1, 1),
                                    adv="WENO5", tracers=("b",), buoyancy=True, closure=("Horizontal", 1e-3, 1e-3),
                                    ts="RungeKutta3", dt=2e-3),
    "box_bbb_upwind5_vertical": dict(size=(8, 9, 10), topology=(O.Bounded,) * 3, extent=(1, 1, 1), adv="UpwindBiasedFifthOrder",
                                     tracers=("b",), buoyancy=True, closure=("Vertical", 1e-3, 1e-3), ts="QuasiAdamsBashforth2", dt=2e-3),
    "centered2_default": dict(size=(8, 8, 8), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1),
                              adv="CenteredSecondOrder", tracers=("b",), buoyancy=True, ts="QuasiAdamsBashforth2", dt=2e-3),
    "centered4_tilted": dict(size=(8, 10, 8), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1),
                             adv="CenteredFourthOrder", tracers=("b",), buoyancy=True, tilt=(0.0, 0.6, 0.8),
                             ts="RungeKutta3", dt=2e-3),
    "upwind3_jsweno_none": dict(size=(8, 8, 8), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="UpwindBiasedThirdOrder",
                                tracers=("c",), buoyancy=False, ts="RungeKutta3", dt=2e-3),
    "weno_js": dict(size=(10, 8, 8), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5js",
                    tracers=("b",), buoyancy=True, ts="RungeKutta3", dt=2e-3),
    # SeawaterBuoyancy with the linear equation of state (SURVEY.md 8(f) rank 2): T and S active (general kernels, Bounded z),
    # T and S active on the specialised path (fused kernel for u, v, w, T + per-field kernel for S), temperature only
    # with tilted gravity, salinity only
    "seawater_TS_bounded": dict(size=(8, 10, 12), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1),
                                adv="WENO5", tracers=("T", "S"), seawater={}, closure=("ThreeDimensional", 1e-3, 1e-3),
                                f=0.5, ts="RungeKutta3", dt=2e-3),
    "seawater_TS_periodic_fast": dict(size=(32, 12, 16), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5",
                                      tracers=("T", "S"), seawater=dict(gravitational_acceleration=3.0,
                                                                        eos=(2e-1, 7e-1)), ts="RungeKutta3", dt=2e-3),
    "seawater_T_tilted": dict(size=(8, 8, 10), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1),
                              adv="CenteredFourthOrder", tracers=("T",), seawater=dict(constant_salinity=35.0, eos=(0.3, 0.2)),
                              tilt=(0.6, 0.0, 0.8), ts="QuasiAdamsBashforth2", dt=2e-3),
    # SmagorinskyLilly LES closure (SURVEY.md 8(f) rank 1): eddy viscosity recomputed in update_state!, variable-ν stresses,
    # κₑ = νₑ / Pr; with a buoyancy tracer (stability correction), on a stretched Bounded z with WENO5(grid), with seawater
    # buoyancy and per-tracer Prandtl numbers, and in 2-D (Flat z)
    "smagorinsky_bounded_b": dict(size=(8, 10, 12), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1),
                                  adv="CenteredSecondOrder", tracers=("b",), buoyancy=True, smagorinsky={}, f=0.5,
                                  ts="RungeKutta3", dt=2e-3),
    "smagorinsky_stretched_weno": dict(size=(12, 8, 14), topology=(O.Periodic, O.Periodic, O.Bounded),
                                       coords=dict(x=(0, 1), y=(0, 1), z=_zf(14)), adv="WENO5grid", tracers=("b", "c"),
                                       buoyancy=True, smagorinsky=dict(C=0.2, Cb=0.5, Pr={"b": 0.7, "c": 2.0}),
                                       ts="RungeKutta3", dt=2e-3,
                                       bcs={"u": {"top": ("Flux", -1e-3)}, "b": {"top": ("Flux", 1e-4)}}),
    "smagorinsky_seawater_periodic": dict(size=(32, 8, 8), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5",
                                          tracers=("T", "S"), seawater=dict(eos=(0.3, 0.2)), smagorinsky=dict(Cb=1.0, Pr=1.0),
                                          ts="QuasiAdamsBashforth2", dt=2e-3),
    "smagorinsky_2d_flat": dict(size=(16, 12), topology=(O.Periodic, O.Bounded, O.Flat), extent=(1, 1),
                                adv="UpwindBiasedThirdOrder", tracers=("c",), buoyancy=False, smagorinsky=dict(Pr=0.5),
                                ts="RungeKutta3", dt=2e-3),
    # AnisotropicMinimumDissipation (the closure of the C3 source example, ocean_wind_mixing_and_convection.jl:151): C3 physics
    # with AMD instead of ScalarDiffusivity; with the buoyancy modification Cb and per-tracer Poincaré constants; seawater
    "amd_c3_stretched_weno": dict(size=(12, 8, 14), topology=(O.Periodic, O.Periodic, O.Bounded),
                                  coords=dict(x=(0, 1), y=(0, 1), z=_zf(14)), adv="WENO5grid", tracers=("b",), buoyancy=True,
                                  amd={}, f=1e-2, ts="RungeKutta3", dt=5e-3,
                                  bcs={"u": {"top": ("Flux", -1e-3)}, "b": {"top": ("Flux", 1e-4), "bottom": ("Gradient", 1e-2)}}),
    "amd_Cb_bounded": dict(size=(8, 10, 12), topology=(O.Periodic, O.Bounded, O.Bounded), extent=(1, 2, 1),
                           adv="CenteredSecondOrder", tracers=("b", "c"), buoyancy=True,
                           amd=dict(Cν=0.1, Cκ={"b": 0.08, "c": 0.2}, Cb=1.0), ts="QuasiAdamsBashforth2", dt=2e-3),
    "amd_seawater_periodic": dict(size=(32, 8, 8), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5", tracers=("T", "S"),
                                  seawater=dict(eos=(0.3, 0.2)), amd=dict(C=1 / 6, Cb=0.5), ts="RungeKutta3", dt=2e-3),
    # VerticallyImplicitTimeDiscretization (SURVEY.md 8(f) rank 3): the z-derivative parts of the vertical fluxes go through the
    # batched tridiagonal solve after every substep; C3 physics (stretched Bounded z) with the ThreeDimensional formulation, and
    # the Vertical formulation in a closed box with AB2
    "vitd_c3_stretched_weno": dict(size=(12, 8, 14), topology=(O.Periodic, O.Periodic, O.Bounded),
                                   coords=dict(x=(0, 1), y=(0, 1), z=_zf(14)), adv="WENO5grid", tracers=("b",), buoyancy=True,
                                   closure=("ThreeDimensional", 1e-2, 2e-2), vitd=True, f=1e-2, ts="RungeKutta3", dt=5e-3,
                                   bcs={"u": {"top": ("Flux", -1e-3)}, "b": {"top": ("Flux", 1e-4), "bottom": ("Gradient", 1e-2)}}),
    "vitd_vertical_box_ab2": dict(size=(8, 9, 10), topology=(O.Bounded,) * 3, extent=(1, 1, 1), adv="UpwindBiasedFifthOrder",
                                  tracers=("b", "c"), buoyancy=True, closure=("Vertical", 5e-2, 3e-2), vitd=True,
                                  ts="QuasiAdamsBashforth2", dt=2e-2),
    "seawater_S_only": dict(size=(8, 8, 8), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="UpwindBiasedFifthOrder",
                            tracers=("S", "c"), seawater=dict(constant_temperature=True, eos=(0.3, 0.2)),
                            ts="RungeKutta3", dt=2e-3),
}


def build_models(ob, cfg, FT):
    go, gb = make_pair(ob, FT, cfg["size"], cfg["topology"], coords=cfg.get("coords"), extent=cfg.get("extent"))
    adv = cfg["adv"]
    if adv is None:
        ao = ab = None
    elif adv == "WENO5":
        ao, ab = O.WENO5(FT), ob.WENO5(FT)
    elif adv == "WENO5js":
        ao, ab = O.WENO5(FT, zweno=False), ob.WENO5(FT, zweno=False)
    elif adv == "WENO5grid":
        ao, ab = O.WENO5(grid=go), ob.WENO5(grid=gb)
    elif adv == "WENO5grid_js":
        ao, ab = O.WENO5(grid=go, zweno=False), ob.WENO5(grid=gb, zweno=False)
    else:
        ao, ab = getattr(O, adv)(), getattr(ob, adv)()
    clo_o = clo_b = None
    if cfg.get("closure"):
        form, nu, ka = cfg["closure"]
        td = "VerticallyImplicit" if cfg.get("vitd") else "Explicit"
        clo_o = O.ScalarDiffusivity(form, ν=nu, κ=ka, time_discretization=td)
        clo_b = ob.ScalarDiffusivity(form, ν=nu, κ=ka, time_discretization=td)
    if cfg.get("smagorinsky") is not None:
        clo_o, clo_b = O.SmagorinskyLilly(**cfg["smagorinsky"]), ob.SmagorinskyLilly(**cfg["smagorinsky"])
    if cfg.get("amd") is not None:
        clo_o, clo_b = O.AnisotropicMinimumDissipation(**cfg["amd"]), ob.AnisotropicMinimumDissipation(**cfg["amd"])
    cor_o = O.FPlane(cfg["f"]) if cfg.get("f") else None
    cor_b = ob.FPlane(cfg["f"]) if cfg.get("f") else None
    bu_o = bu_b = None
    if cfg.get("buoyancy"):
        bu_o = O.Buoyancy(O.BuoyancyTracer(), cfg.get("tilt"))
        bu_b = ob.Buoyancy(ob.BuoyancyTracer(), cfg.get("tilt"))
    if cfg.get("seawater") is not None:
        kw = dict(cfg["seawater"])
        eos = kw.pop("eos", None)
        mk = lambda M: M.Buoyancy(M.SeawaterBuoyancy(equation_of_state=M.LinearEquationOfState(*eos) if eos else None, **kw),
                                  cfg.get("tilt"))
        bu_o, bu_b = mk(O), mk(ob)
    bcs_o = bcs_b = None
    if cfg.get("bcs"):
        bcs_o = {n: {s: O.BoundaryCondition(*kv) for s, kv in d.items()} for n, d in cfg["bcs"].items()}
        bcs_b = {n: {s: ob.BoundaryCondition(*kv) for s, kv in d.items()} for n, d in cfg["bcs"].items()}
    mo = O.NonhydrostaticModel(go, advection=ao, closure=clo_o, coriolis=cor_o, buoyancy=bu_o,
                               tracers=cfg["tracers"], timestepper=cfg["ts"], boundary_conditions=bcs_o)
    mb = ob.NonhydrostaticModel(gb, advection=ab, closure=clo_b, coriolis=cor_b, buoyancy=bu_b,
                                tracers=cfg["tracers"], timestepper=cfg["ts"], boundary_conditions=bcs_b)
    return mo, mb


def init_state(mo, mb, ob, seed):
    rng = np.random.default_rng(seed)
    vals = {}
    for n in mo.names:
        f = mo.fields[n]
        a = rng.uniform(-1, 1, f.size())
        if n in "uvw":
            a = a - a.mean()
        else:
            z = mo.grid.nodes(f.loc)[2]
            a = 0.5 * z + 0.1 * a
        vals[n] = a.astype(mo.grid.FT)
    mo.set(**vals)
    ob.set_model(mb, **vals)


def compare_fields(mo, mb, tol, what="state"):
    worst = 0.0
    for n in mo.names:
        e = relerr(mb.fields[n].interior(), mo.fields[n].interior)
        worst = max(worst, e)
        assert e < tol, f"{what}: field {n} differs: rel err {e:.3e}"
    return worst


@pytest.mark.parametrize("name", list(CONFIGS))
def test_tendencies_and_steps_match_oracle_f64(ob, name):
    cfg = CONFIGS[name]
    FT = np.float64
    mo, mb = build_models(ob, cfg, FT)
    init_state(mo, mb, ob, 21)
    compare_fields(mo, mb, 1e-12, "after set!/projection")
    if mo.pHY is not None:
        assert relerr(mb.pressures["pHY′"].interior(), mo.pHY.interior) < 1e-13
    if getattr(mo, "νe", None) is not None:          # the eddy viscosity of the LES closure, halos included
        assert relerr(mb.diffusivity_fields["νₑ"].parent(), mo.νe.parent) < 1e-12
        if getattr(mo, "κe", None) is not None:
            for n in mo.tracer_names:
                assert relerr(mb.diffusivity_fields["κₑ"][n].parent(), mo.κe[n].parent) < 1e-12, n
    # tendencies alone
    mo.calculate_tendencies()
    ob.calculate_tendencies(mb)
    g = mo.grid
    for n in mo.names:
        Go = mo.Gn[n][O.R(1, g.Nx), O.R(1, g.Ny), O.R(1, g.Nz)]
        Gb = mb.Gn[n].interior()[:g.Nx, :g.Ny, :g.Nz]
        assert relerr(Gb, Go) < 1e-12, f"tendency {n}"
    # time steps, checked after every step
    for step in range(4):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        compare_fields(mo, mb, 1e-12, f"step {step + 1}")
        assert relerr(mb.pressures["pNHS"].interior(), mo.pNHS.interior) < 1e-9
    d = mb.diagnostics()
    assert d["max_abs_div"] < 1e-10
    assert abs(d["kinetic_energy"] - mo.kinetic_energy()) <= 1e-11 * mo.kinetic_energy()
    assert abs(mb.clock.time - mo.clock.time) < 1e-15 and mb.clock.iteration == 4


@pytest.mark.parametrize("name", ["c2_periodic_weno_rk3", "c3_stretched_weno_rk3", "c3_fused_stretched_weno_rk3", "c1_2d_flat_weno_ab2"])
def test_steps_match_oracle_f32(ob, name):
    cfg = CONFIGS[name]
    mo, mb = build_models(ob, cfg, np.float32)
    init_state(mo, mb, ob, 22)
    for step in range(3):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        compare_fields(mo, mb, 1e-5, f"f32 step {step + 1}")


def test_fast_and_general_kernels_agree(ob):
    """the specialised headline kernels against the general ones on the same state"""
    cfg = CONFIGS["c2_periodic_weno_rk3"]
    mo, m1 = build_models(ob, cfg, np.float64)
    _, m2 = build_models(ob, cfg, np.float64)
    m2.use_fast_kernels(False)
    init_state(mo, m1, ob, 23)
    init_state(mo, m2, ob, 23)
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert relerr(m1.fields[n].interior(), m2.fields[n].interior()) < 1e-13


def test_fused_bounded_z_kernel_agrees_with_general_kernels(ob):
    """C3 physics at 64 x 40 x 48 (five tile rows of 12, the last partial; chunks of the leftover tiles split along z): the
    fused Bounded-z kernel against the general per-field kernels on the same state, three RK3 steps"""
    cfg = dict(CONFIGS["c3_fused_stretched_weno_rk3"], size=(64, 40, 48), coords=dict(x=(0, 2), y=(0, 1.5), z=_zf(48)))
    mo, m1 = build_models(ob, cfg, np.float64)
    _, m2 = build_models(ob, cfg, np.float64)
    m2.use_fast_kernels(False)
    init_state(mo, m1, ob, 29)
    init_state(mo, m2, ob, 29)
    ob.calculate_tendencies(m1)
    ob.calculate_tendencies(m2)
    for n in m1.names:
        assert relerr(m1.Gn[n].interior(), m2.Gn[n].interior()) < 1e-12, f"tendency {n}"
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert relerr(m1.fields[n].interior(), m2.fields[n].interior()) < 1e-12, n


@pytest.mark.parametrize("size", [(32, 5, 6), (64, 13, 7), (96, 25, 9), (32, 12, 33), (32, 3, 16)])
@pytest.mark.parametrize("stretched", [True, False])
def test_fused_bounded_z_kernel_odd_shapes(ob, size, stretched):
    """tile rows of 12 against Ny smaller than, equal to and not a multiple of it; Nz at the minimum the kernel takes (6), odd and
    longer than the ring; regular and stretched z: fused Bounded-z kernel against the general kernels, tendencies and two steps"""
    cfg = dict(CONFIGS["c3_fused_stretched_weno_rk3"], size=size)
    if stretched:
        cfg["coords"] = dict(x=(0, 1), y=(0, 1), z=_zf(size[2]))
    else:
        cfg.pop("coords")
        cfg["extent"] = (1, 1, 1)
        cfg["adv"] = "WENO5"
    mo, m1 = build_models(ob, cfg, np.float64)
    _, m2 = build_models(ob, cfg, np.float64)
    m2.use_fast_kernels(False)
    init_state(mo, m1, ob, 37)
    init_state(mo, m2, ob, 37)
    ob.calculate_tendencies(m1)
    ob.calculate_tendencies(m2)
    for n in m1.names:
        assert relerr(m1.Gn[n].interior(), m2.Gn[n].interior()) < 1e-12, f"tendency {n}"
    for _ in range(2):
        ob.time_step(m1, cfg["dt"])
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert relerr(m1.fields[n].interior(), m2.fields[n].interior()) < 1e-12, n


def test_c3_128x128x64_one_step_matches_oracle(ob):
    """BASELINE config 3 physics on a 128 x 128 x 64 slice of its grid, one RK3 step on the fused Bounded-z kernel against
    the NumPy oracle (about 20 s of oracle time)"""
    cfg = dict(CONFIGS["c3_fused_stretched_weno_rk3"], size=(128, 128, 64), coords=dict(x=(0, 4), y=(0, 4), z=_zf(64)))
    mo, mb = build_models(ob, cfg, np.float64)
    init_state(mo, mb, ob, 31)
    mo.time_step(cfg["dt"])
    ob.time_step(mb, cfg["dt"])
    compare_fields(mo, mb, 1e-12, "C3 128x128x64, one step")
    assert relerr(mb.pressures["pNHS"].interior(), mo.pNHS.interior) < 1e-9


def test_c3_full_size_fused_and_general_kernels_agree(ob):
    """BASELINE config 3 at its full size, 512 x 512 x 256: tendencies and one RK3 step of the fused Bounded-z kernel against
    the general per-field kernels; the stepped state is divergence free and w vanishes on the walls"""
    n = (512, 512, 256)
    cfg = dict(CONFIGS["c3_fused_stretched_weno_rk3"], size=n, coords=dict(x=(0, 64), y=(0, 64), z=_zf(256)))
    mb = []
    for fast in (True, False):
        gb = ob.RectilinearGrid(ob.arch, np.float64, size=n, topology=("Periodic", "Periodic", "Bounded"), **cfg["coords"])
        form, nu, ka = cfg["closure"]
        bcs = {f: {s: ob.BoundaryCondition(*kv) for s, kv in d.items()} for f, d in cfg["bcs"].items()}
        m = ob.NonhydrostaticModel(gb, advection=ob.WENO5(grid=gb), closure=ob.ScalarDiffusivity(form, ν=nu, κ=ka),
                                   coriolis=ob.FPlane(cfg["f"]), buoyancy=ob.Buoyancy(ob.BuoyancyTracer(), None), tracers=("b",),
                                   timestepper="RungeKutta3", boundary_conditions=bcs)
        m.use_fast_kernels(fast)
        mb.append(m)
    rng = np.random.default_rng(33)
    vals = {}
    for name in mb[0].names:
        a = rng.uniform(-1, 1, mb[0].fields[name].size())
        vals[name] = a - a.mean() if name in "uvw" else 1e-2 * a
    for m in mb:
        ob.set_model(m, **vals)
        ob.calculate_tendencies(m)
    for name in mb[0].names:
        assert relerr(mb[0].Gn[name].interior(), mb[1].Gn[name].interior()) < 1e-12, f"tendency {name}"
    for m in mb:
        ob.time_step(m, 1e-3)
    for name in mb[0].names:
        assert relerr(mb[0].fields[name].interior(), mb[1].fields[name].interior()) < 1e-12, name
    assert mb[0].diagnostics()["max_abs_div"] < 1e-9
    w = mb[0].fields["w"].interior()
    assert np.all(w[:, :, 0] == 0)


def test_ab2_first_step_is_euler_and_simulation_runs(ob):
    cfg = CONFIGS["c1_2d_flat_weno_ab2"]
    mo, mb = build_models(ob, cfg, np.float64)
    init_state(mo, mb, ob, 24)
    sim = ob.Simulation(mb, Δt=cfg["dt"], stop_iteration=6)
    ob.run(sim)
    for _ in range(6):
        mo.time_step(cfg["dt"])
    compare_fields(mo, mb, 1e-11, "run!")
    assert mb.clock.iteration == 6


# ---- full-size properties (BASELINE.json config 2: 256^3) ----------------------------------------
def test_full_size_256_properties(ob):
    """size-independent properties at the headline size: the projected state is divergence free,
    tracer mean is conserved by flux-form advection on a periodic domain, and halos are periodic."""
    N = 256
    gb = ob.RectilinearGrid(ob.arch, np.float64, size=(N, N, N), extent=(1, 1, 1), topology=("Periodic",) * 3)
    m = ob.NonhydrostaticModel(gb, advection=ob.WENO5(), tracers=("b",), buoyancy=ob.BuoyancyTracer(),
                               timestepper="RungeKutta3")
    rng = np.random.default_rng(2)
    vals = {}
    for n in "uvw":
        a = rng.uniform(-1, 1, (N, N, N))
        vals[n] = a - a.mean()
    z = gb.nodes(("Center",) * 3)[2]
    vals["b"] = 1e-5 * z + 1e-3 * rng.uniform(-1, 1, (N, N, N))
    ob.set_model(m, **vals)
    b0 = m.tracers["b"].reduce()["sum"]
    d0 = m.diagnostics()
    assert d0["max_abs_div"] < 1e-9
    dt = 0.1 / N
    for _ in range(2):
        ob.time_step(m, dt)
    d1 = m.diagnostics()
    assert d1["max_abs_div"] < 1e-9
    assert 0 < d1["kinetic_energy"] <= d0["kinetic_energy"] * (1 + 1e-12)     # WENO is dissipative
    b1 = m.tracers["b"].reduce()["sum"]
    assert abs(b1 - b0) <= 1e-10 * (abs(b0) + N ** 3 * 1e-3)
    p = m.velocities["u"].parent()
    assert np.array_equal(p[:3], p[N:N + 3]) and np.array_equal(p[:, :, N + 3:], p[:, :, 3:6])


def test_slab_decomposition_two_gpus_matches_oracle():
    """runs tests/dist_check.py under torchrun when the box has >= 2 GPUs (skipped otherwise)"""
    import os
    import subprocess
    import sys
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533",
                          os.path.join(root, "tests", "dist_check.py")], capture_output=True, text=True, timeout=600)
    assert "DIST_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


# ---- SURVEY.md 8(f) rank 2: TimeStepWizard / CFL reductions -------------------------------------------------------
def test_cell_advection_timescale_and_wizard(ob):
    """cell_advection_timescale (Utils/cell_advection_timescale.jl:4-21: maxima over the PARENT arrays, halos included) and
    the TimeStepWizard arithmetic (time_step_wizard.jl:78-95) against the same formulas evaluated on the oracle's arrays"""
    for name in ("c3_stretched_weno_rk3", "c2_periodic_weno_rk3", "c1_2d_flat_weno_ab2"):
        cfg = CONFIGS[name]
        mo, mb = build_models(ob, cfg, np.float64)
        init_state(mo, mb, ob, 31)
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        g = mo.grid
        umax = [float(np.max(np.abs(mo.velocities[n].parent))) for n in "uvw"]
        got = ob.max_abs_velocities(mb)
        for a, b in zip(got, umax):
            assert abs(a - b) <= 1e-12 * max(b, 1e-300), (name, got, umax)
        dmin = []
        for d in range(3):
            if g.topology[d] == O.Flat:
                dmin.append(np.inf)
            else:
                dc = g.dC[d]
                dmin.append(float(dc) if g.regular[d] else float(np.min(dc.parent)))
        want = min(dm / um if um > 0 else np.inf for dm, um in zip(dmin, umax))
        tau = ob.cell_advection_timescale(mb)
        assert abs(tau - want) <= 1e-12 * want, (name, tau, want)
        wiz = ob.TimeStepWizard(cfl=0.5, max_change=1.2, min_change=0.5, max_Δt=10.0)
        old = cfg["dt"]
        new = wiz.new_time_step(old, mb)
        expect = min(max(min(1.2 * old, 0.5 * want), 0.5 * old), 10.0)
        assert abs(new - expect) <= 1e-12 * expect
    # a NaN in a velocity is reported as NaN (NaNChecker)
    u = mb.velocities["u"]
    a = u.interior().copy()
    a[0, 0, 0] = np.nan
    u.set(a)
    assert np.isnan(ob.max_abs_velocities(mb)[0])


# ---- several models in one process: handles own their streams, events and tensor maps ------------------------------------
def test_two_models_of_different_sizes_interleaved_and_recreated(ob):
    """create two models of different sizes, step them alternately, destroy one, create a third of yet another size (its
    buffers may reuse the freed addresses: stale tensor maps would fault or corrupt), and check all against the oracle"""
    import gc
    from ocean_b200._lib import lib

    def pair(size, seed):
        cfg = dict(size=size, topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5", tracers=("b",), buoyancy=True,
                   ts="RungeKutta3", dt=2e-3)
        mo, mb = build_models(ob, cfg, np.float64)
        init_state(mo, mb, ob, seed)
        return mo, mb
    a_o, a_b = pair((32, 16, 16), 41)
    b_o, b_b = pair((64, 12, 8), 42)
    for _ in range(2):
        a_o.time_step(2e-3); ob.time_step(a_b, 2e-3)
        b_o.time_step(2e-3); ob.time_step(b_b, 2e-3)
    compare_fields(a_o, a_b, 1e-12, "model A")
    compare_fields(b_o, b_b, 1e-12, "model B")
    maps_before = lib.ob200_debug_cached_tensor_maps()
    assert maps_before > 0                    # both took the TMA-staged fused kernel
    a_b.destroy()
    del a_b
    gc.collect()
    assert lib.ob200_debug_cached_tensor_maps() < maps_before       # the maps over A's buffers were evicted
    c_o, c_b = pair((32, 20, 16), 43)
    for _ in range(2):
        c_o.time_step(2e-3); ob.time_step(c_b, 2e-3)
        b_o.time_step(2e-3); ob.time_step(b_b, 2e-3)
    compare_fields(c_o, c_b, 1e-12, "model C (after A was destroyed)")
    compare_fields(b_o, b_b, 1e-12, "model B (second round)")


# ---- output path: on-device slices / averages, checkpoints (SURVEY.md 8(f) rank 4) ------------------------------------------
def test_on_device_slices_and_averages(ob):
    rng = np.random.default_rng(41)
    for topo, FT in (((O.Periodic, O.Bounded, O.Bounded), np.float64), ((O.Periodic, O.Periodic, O.Periodic), np.float32)):
        _, gb = make_pair(ob, FT, (12, 9, 7), topo, extent=(1, 1, 1))
        for loc in (("Center", "Center", "Center"), ("Center", "Face", "Face")):
            f = ob.Field(loc, gb)
            p = rng.uniform(-1, 1, f.parent_size).astype(FT)
            f.set_parent(p)
            H, n = gb.H, f.size()
            # an xy plane with halos, a yz plane without, a single column, the whole parent
            for sl in (ob.FieldSlicer(k=3, with_halos=True), ob.FieldSlicer(i=5), ob.FieldSlicer(i=2, j=(2, 4)),
                       ob.FieldSlicer(with_halos=True), ob.FieldSlicer(i=(3, 9), j=(1, n[1]), k=(2, 2))):
                lo, hi = sl.box(f)
                want = p[tuple(slice(H[d] + lo[d] - 1, H[d] + hi[d]) for d in range(3))]
                assert np.array_equal(ob.fetch_output(f, sl), want)
            inter = p[tuple(slice(H[d], H[d] + n[d]) for d in range(3))].astype(np.float64)
            tol = 1e-13 if FT == np.float64 else 1e-6
            for dims in ((1, 2), (3,), (1,), (1, 2, 3), (2, 3)):
                want = inter.mean(axis=tuple(d - 1 for d in dims), keepdims=True)
                got = f.average(dims)
                assert got.shape == want.shape and np.max(np.abs(got - want)) < tol * max(1.0, np.max(np.abs(want)))
            assert np.allclose(ob.horizontal_average(f), inter.mean(axis=(0, 1)), rtol=0, atol=tol)
    with pytest.raises(ob.B200Error):
        f.slice((0, 1, 1), (99, 1, 1))


@pytest.mark.parametrize("name", ["c2_periodic_weno_rk3", "c3_fused_js_ab2_no_closure", "smagorinsky_bounded_b"])
def test_checkpoint_resume_is_bitwise(ob, name, tmp_path):
    """Checkpointer (checkpointer.jl:64-95) + set!(model, filepath) (:201-262): 3 steps, checkpoint, restore into a NEW model,
    3 more steps == 6 steps straight, bit for bit (fields, G^n / G^-, clock; AB2 keeps its history and its previous time step)"""
    cfg = CONFIGS[name]
    mo, m1 = build_models(ob, cfg, np.float64)
    init_state(mo, m1, ob, 43)
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
    path = ob.Checkpointer(m1, dir=str(tmp_path), prefix="ck").write()
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
    _, m2 = build_models(ob, cfg, np.float64)
    ob.Checkpointer.restore(m2, path)
    assert m2.clock.iteration == 3
    for _ in range(3):
        ob.time_step(m2, cfg["dt"])
    assert m2.clock.iteration == m1.clock.iteration and m2.clock.time == m1.clock.time
    for n in m1.names:
        assert np.array_equal(m1.fields[n].parent(), m2.fields[n].parent()), n


@pytest.mark.parametrize("name", ["c3_fused_js_ab2_no_closure", "c3_fused_stretched_weno_rk3", "c2_periodic_weno_rk3",
                                  "ppb_regular_fused_weno_rk3"])
def test_two_identical_models_agree_bit_for_bit(ob, name):
    """no result may depend on the history or the memory of a solver / model instance: the Fourier-tridiagonal solve pins the
    singular horizontal-mean column instead of dividing rounding noise by rounding noise, and the mean is summed in a fixed
    order (no atomics).  Two models built and initialised alike agree in every bit of every field, tendency and pressure."""
    cfg = CONFIGS[name]
    mo, m1 = build_models(ob, cfg, np.float64)
    init_state(mo, m1, ob, 48)
    for _ in range(2):                   # freed memory of a model with a history is what the next two are allocated from
        ob.time_step(m1, cfg["dt"])
    m1.destroy()
    _, m2 = build_models(ob, cfg, np.float64)
    _, m3 = build_models(ob, cfg, np.float64)
    init_state(mo, m2, ob, 47)
    ob.time_step(m2, cfg["dt"])          # m2's solver has solved before; m3's has not
    init_state(mo, m2, ob, 47)
    m2.set_clock(0.0, 0)
    init_state(mo, m3, ob, 47)
    for step in range(3):
        ob.time_step(m2, cfg["dt"])
        ob.time_step(m3, cfg["dt"])
        for n in m2.names:
            assert np.array_equal(m2.fields[n].parent(), m3.fields[n].parent()), (step, n)
        assert np.array_equal(m2.pressures["pNHS"].interior(), m3.pressures["pNHS"].interior()), step


def test_fourier_tridiagonal_solve_is_history_free_and_well_conditioned(ob):
    """a right-hand side that violates the discrete compatibility condition (zero unweighted mean on a stretched grid): the
    reference's elimination divides by a pivot that is rounding noise and returns a solution quantised at eps * 1e12; here the
    singular column is pinned, two solver instances and repeated solves agree bit for bit, the solution has zero mean and solves
    the equations of every non-singular mode (compared with the oracle on the compatible part)"""
    for size in ((32, 12, 8), (32, 16, 8)):              # general path (Ny not a power of two), half-spectrum path
        kw = dict(size=size, x=(0, 2), y=(0, 1), z=_zf(size[2]), topology=("Periodic", "Periodic", "Bounded"))
        go, gb1 = O.RectilinearGrid(np.float64, **kw), ob.RectilinearGrid(ob.arch, np.float64, **kw)
        gb2 = ob.RectilinearGrid(ob.arch, np.float64, **kw)
        rng = np.random.default_rng(1)
        rhs = rng.uniform(-1, 1, size)
        rhs -= rhs.mean()
        s1, s2 = ob.FourierTridiagonalPoissonSolver(gb1), ob.FourierTridiagonalPoissonSolver(gb2)
        p1, p2 = ob.CenterField(gb1), ob.CenterField(gb2)
        ob.solve(p1, s1, rhs)
        a = p1.interior().copy()
        ob.solve(p1, s1, 0.5 * rhs)                      # history
        ob.solve(p1, s1, rhs)
        ob.solve(p2, s2, rhs)
        assert np.array_equal(a, p1.interior()) and np.array_equal(a, p2.interior())
        assert abs(a.mean()) < 1e-15 and len(np.unique(a)) > 0.99 * a.size
        # compatible right-hand side: remove the Δz-weighted mean; then the oracle (the reference's algorithm) is well conditioned
        dz = np.diff(_zf(size[2])).reshape(1, 1, -1)
        rc = rhs - (rhs * dz).sum() / (dz.sum() * size[0] * size[1])
        po = O.Field(go, auxiliary=True)
        O.FourierTridiagonalPoissonSolver(go).solve(po, rc)
        ob.solve(p1, s1, rc)
        assert relerr(p1.interior(), po.interior) < 1e-11


@pytest.mark.parametrize("form,ν,κ,want", [("ThreeDimensional", 0.3, 0.7, dict(T=2 * 0.7, u=2 * 0.3, v=4 * 0.3, w=6 * 0.3)),
                                           ("Horizontal", 0.3, 0.7, dict(T=8 * 0.7, u=2 * 0.3, v=4 * 0.3, w=6 * 0.3)),
                                           ("Vertical", 0.1, 0.5, dict(T=10 * 0.5, u=4 * 0.1, v=6 * 0.1, w=8 * 0.1))])
def test_closure_flux_divergence_known_answers_on_cuda(ob, form, ν, κ, want):
    """the reference's hand-computed closure flux divergences (test/test_turbulence_closures.jl:26-101: -2κ, -2ν, -4ν, -6ν for the
    isotropic closure; -8κh, -10κz, ... for the horizontal / vertical ones) as the TENDENCIES of a model with nothing but the
    closure, through the CUDA path; independent of the oracle"""
    gb = ob.RectilinearGrid(ob.arch, np.float64, size=(3, 1, 4), extent=(3, 1, 4), topology=("Periodic", "Periodic", "Bounded"))
    m = ob.NonhydrostaticModel(gb, advection=None, closure=ob.ScalarDiffusivity(form, ν=ν, κ=κ), tracers=("T",))
    if form == "ThreeDimensional":
        lines = {n: {k: [0, c, 0] for k in (1, 2, 3, 4)} for n, c in (("u", -0.5), ("v", -2), ("w", -3), ("T", -1))}
    else:
        lines = {n: {2: [0, 1, 0], 3: [0, c, 0], 4: [0, 1, 0]} for n, c in (("u", -1), ("v", -2), ("w", -3), ("T", -4))}
    for n, prof in lines.items():
        f = m.fields[n]
        a = np.zeros(f.size())
        for k, line in prof.items():
            a[:, 0, k - 1] = line
        f.set(a)                                  # no projection: the reference test sets the arrays directly
    ob.update_state(m)
    ob.calculate_tendencies(m)
    for n, val in want.items():
        got = m.Gn[n].interior()[1, 0, 2]         # Julia (2, 1, 3); tendency = -(flux divergence)
        assert abs(got - val) <= 4e-16 * abs(val), (n, got, val)
