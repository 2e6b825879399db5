"""Background fields (background_fields.jl) on the CUDA path against the oracle with the same backgrounds
(background_reference.py): configurations that reach every tendency path with backgrounds (the background-only shared-face
pass + the fused kernel's accumulate form, periodic and Bounded z; after the AMD closure split; with the relaxation pass; the
general kernels on Flat and tilted grids and with vertically implicit diffusion; the per-field fallback of a second tracer),
the fused path against the general kernels, the linear-stratification known answer, replacing a background between steps,
checkpoint / resume, Float32 and the mirror's rejections."""
import numpy as np
import pytest

import oracle as O
from background_reference import BackgroundNonhydrostaticModel, table
from test_gpu_parity import CONFIGS, _zf, compare_fields, init_state, make_pair, relerr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ob():
    import ocean_b200 as ob
    ob.arch = ob.B200()
    return ob


def build_bg(ob, cfg, FT, bg, forcing=None):
    """both models of `cfg` with background_fields = `bg` ({name: func(x, y, z, t)}) and Relaxation `forcing`; `ob` may be the
    oracle-only stand-in of test_gpu_float32.py"""
    go, gb = make_pair(ob, FT, cfg["size"], cfg["topology"], coords=cfg.get("coords"), extent=cfg.get("extent"))
    adv = cfg["adv"]
    if adv == "WENO5":
        ao, ab = O.WENO5(FT), ob.WENO5(FT)
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
    if cfg.get("amd") is not None:
        clo_o, clo_b = O.AnisotropicMinimumDissipation(**cfg["amd"]), ob.AnisotropicMinimumDissipation(**cfg["amd"])
    cor_o = O.FPlane(cfg["f"]) if cfg.get("f") else None
    cor_b = ob.FPlane(cfg["f"]) if cfg.get("f") else None
    bu_o = O.Buoyancy(O.BuoyancyTracer(), cfg.get("tilt")) if cfg.get("buoyancy") else None
    bu_b = ob.Buoyancy(ob.BuoyancyTracer(), cfg.get("tilt")) if cfg.get("buoyancy") else None
    bcs_o = bcs_b = None
    if cfg.get("bcs"):
        bcs_o = {n: {s: O.BoundaryCondition(*kv) for s, kv in d.items()} for n, d in cfg["bcs"].items()}
        bcs_b = {n: {s: ob.BoundaryCondition(*kv) for s, kv in d.items()} for n, d in cfg["bcs"].items()}
    frc = {}
    for n, (rate, mask, target) in (forcing or {}).items():
        m = None if mask is None else ob.GaussianMask(*mask)
        t = ob.LinearTarget(*target) if isinstance(target, tuple) else target
        frc[n] = ob.Relaxation(rate, mask=m, target=t)
    mo = BackgroundNonhydrostaticModel(go, background_fields=bg, forcing=frc, advection=ao, closure=clo_o, coriolis=cor_o,
                                       buoyancy=bu_o, tracers=cfg["tracers"], timestepper=cfg["ts"], boundary_conditions=bcs_o)
    mb = ob.NonhydrostaticModel(gb, advection=ab, closure=clo_b, coriolis=cor_b, buoyancy=bu_b, tracers=cfg["tracers"],
                                timestepper=cfg["ts"], boundary_conditions=bcs_b, forcing=frc or None, background_fields=bg)
    return mo, mb


N2 = 2.0
STRAT = lambda x, y, z, t: N2 * z
SHEAR = lambda x, y, z, t: 0.3 * np.tanh((z + 0.5) / 0.15)
HEADLINE = dict(size=(32, 12, 16), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5", tracers=("b",), buoyancy=True,
                ts="RungeKutta3", dt=2e-3)
C3 = CONFIGS["c3_fused_stretched_weno_rk3"]
SPONGE = lambda rate: (rate, ("z", -0.9, 0.1), None)
THETA = 0.2
CASES = {
    # B = N² z on the triply periodic headline: the background pass + the fused periodic kernel's accumulate form
    "headline_strat": (HEADLINE, {"b": STRAT}, None),
    # C3 physics with U(z), B(z): the fused Bounded-z kernel
    "c3_shear_strat": (C3, {"u": SHEAR, "b": STRAT}, None),
    # AMD: closure-only kernel, then the background pass adding onto it
    "amd_c3_split": (CONFIGS["amd_c3_fused_split"], {"u": SHEAR, "b": STRAT}, None),
    # background pass + relaxation pass + accumulate form
    "c3_sponge": (C3, {"u": SHEAR, "b": STRAT}, {"u": SPONGE(20.0), "b": (20.0, ("z", -0.9, 0.1), ("z", 0.0, 0.5))}),
    # vertically implicit diffusion: the general shared-face kernel with the background fluxes
    "vitd_c3": (CONFIGS["vitd_c3_stretched_weno"], {"u": SHEAR, "b": STRAT}, None),
    # 2-D Kelvin-Helmholtz (Flat y): the general kernel
    "kh_2d_flat_y": (dict(size=(32, 16), topology=(O.Periodic, O.Flat, O.Bounded), extent=(2, 1), adv="WENO5", tracers=("b",),
                          buoyancy=True, ts="RungeKutta3", dt=2e-3),
                     {"u": lambda x, y, z, t: np.tanh((z + 0.5) / 0.1), "b": lambda x, y, z, t: 0.5 * np.tanh((z + 0.5) / 0.1)},
                     None),
    # tilted gravity, Periodic x, B = N² (x sin θ + z cos θ): not periodic in x, its halos unwrapped
    "tilted_periodic_x": (dict(size=(32, 8, 16), topology=(O.Periodic, O.Periodic, O.Bounded), extent=(1, 1, 1), adv="WENO5",
                               tracers=("b",), buoyancy=True, tilt=(np.sin(THETA), 0.0, np.cos(THETA)), ts="RungeKutta3", dt=2e-3),
                          {"b": lambda x, y, z, t: N2 * (x * np.sin(THETA) + z * np.cos(THETA))}, None),
    # every velocity and a second tracer with its own background: per-field general kernels for tracer c
    "all_velocities_two_tracers": (dict(HEADLINE, tracers=("b", "c")),
                                   {"u": lambda x, y, z, t: 0.2 * np.sin(2 * np.pi * z), "v": lambda x, y, z, t: 0.1 + 0 * x,
                                    "w": lambda x, y, z, t: 0.05 * np.cos(2 * np.pi * y), "b": STRAT,
                                    "c": lambda x, y, z, t: np.sin(2 * np.pi * y)}, None),
    # AB2 on the fused Bounded-z kernel, JS weights, two tracers
    "ab2_c3_js": (CONFIGS["c3_fused_js_ab2_no_closure"], {"b": STRAT, "c": lambda x, y, z, t: 0.3 * z ** 2}, None),
}


@pytest.mark.parametrize("name", list(CASES))
def test_background_tendencies_and_steps_match_oracle_f64(ob, name):
    cfg, bg, forcing = CASES[name]
    mo, mb = build_bg(ob, cfg, np.float64, bg, forcing)
    init_state(mo, mb, ob, 81)
    mo.calculate_tendencies()
    ob.calculate_tendencies(mb)
    g = mo.grid
    for n in mo.names:
        Go = mo.Gn[n][O.R(1, g.Nx), O.R(1, g.Ny), O.R(1, g.Nz)]
        assert relerr(mb.Gn[n].interior()[:g.Nx, :g.Ny, :g.Nz], Go) < 1e-12, f"tendency {n}"
    for step in range(4):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        compare_fields(mo, mb, 1e-12, f"step {step + 1}")


@pytest.mark.parametrize("name", ["headline_strat", "c3_shear_strat", "amd_c3_split", "all_velocities_two_tracers"])
def test_fused_path_agrees_with_general_kernels(ob, name):
    cfg, bg, forcing = CASES[name]
    mo, m1 = build_bg(ob, cfg, np.float64, bg, forcing)
    _, m2 = build_bg(ob, cfg, np.float64, bg, forcing)
    m2.use_fast_kernels(False)
    init_state(mo, m1, ob, 83)
    init_state(mo, m2, ob, 83)
    ob.calculate_tendencies(m1)
    ob.calculate_tendencies(m2)
    for n in m1.names:
        assert relerr(m1.Gn[n].interior(), m2.Gn[n].interior()) < 1e-13, f"tendency {n}"
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert relerr(m1.fields[n].interior(), m2.fields[n].interior()) < 1e-13, n


@pytest.mark.parametrize("periodic", [True, False])
def test_linear_stratification_known_answer_on_cuda(ob, periodic):
    """Gb(with B = N² z) - Gb(without) = -N² (w[k] + w[k+1]) / 2 on a divergence-free state, on the fused path (triply periodic:
    B's halos unwrapped) and on a regular Bounded z"""
    topo = ("Periodic",) * 3 if periodic else ("Periodic", "Periodic", "Bounded")
    ms = []
    for bg in (None, {"b": STRAT}):
        gb = ob.RectilinearGrid(ob.arch, np.float64, size=(32, 16, 16), extent=(1, 1, 1), topology=topo)
        m = ob.NonhydrostaticModel(gb, advection=ob.WENO5(), tracers=("b",), timestepper="RungeKutta3", background_fields=bg)
        rng = np.random.default_rng(5)
        st = {n: rng.uniform(-1, 1, m.fields[n].size()) for n in "uvwb"}
        if not periodic:
            st["w"][:, :, [0, -1]] = 0
        ob.set_model(m, **st)
        ob.calculate_tendencies(m)
        ms.append(m)
    w = ms[1].fields["w"].interior()
    wk1 = np.concatenate([w[:, :, 1:], w[:, :, :1]], axis=2) if periodic else w[:, :, 1:]
    want = -N2 * (w[:, :, :16] + wk1[:, :, :16]) / 2
    d = ms[1].Gn["b"].interior() - ms[0].Gn["b"].interior()
    assert np.max(np.abs(d - want)) <= 1e-10 * N2 * np.max(np.abs(w))


def test_replacing_background_between_steps_matches_oracle(ob):
    cfg, bg, _ = CASES["c3_shear_strat"]
    mo, mb = build_bg(ob, cfg, np.float64, bg)
    init_state(mo, mb, ob, 85)
    for _ in range(2):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
    new = lambda x, y, z, t: 1.5 * N2 * z + 0.1 * np.sin(2 * np.pi * x)
    mo.set_background("b", new)
    ob.set_background(mb, "b", new)
    assert np.array_equal(mb.background_fields["b"].parent(), mo.bg["b"].parent)
    for step in range(3):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        compare_fields(mo, mb, 1e-12, f"after replacement, step {step + 1}")


def test_background_checkpoint_resume_is_bitwise(ob, tmp_path):
    cfg, bg, forcing = CASES["c3_sponge"]
    mo, m1 = build_bg(ob, cfg, np.float64, bg, forcing)
    init_state(mo, m1, ob, 86)
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
    path = ob.Checkpointer(m1, dir=str(tmp_path), prefix="ck").write()
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
    _, m2 = build_bg(ob, cfg, np.float64, bg, forcing)
    ob.Checkpointer.restore(m2, path)
    for _ in range(3):
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert np.array_equal(m1.fields[n].parent(), m2.fields[n].parent()), n


@pytest.mark.parametrize("name", ["headline_strat", "c3_shear_strat", "kh_2d_flat_y", "all_velocities_two_tracers"])
def test_background_float32_against_float64(ob, name):
    """the Float32 CUDA model against the oracle in Float64 on the same Float32-rounded inputs, backgrounds included, within the
    yardstick of test_gpu_float32.py (4 x the Float32 oracle's error + eps32; states also <= 1e-5)"""
    from test_gpu_float32 import f32, run_model_case
    cfg, bg, forcing = CASES[name]

    def build(M, c, FT):
        fbg = bg if FT == np.float32 else {n: (lambda f: lambda *a: f32(f(*a)))(f) for n, f in bg.items()}
        return build_bg(M, c, FT, fbg, forcing)
    run_model_case(ob, f"background/{name}", build, cfg, 87)


def test_mirror_rejects_bad_backgrounds(ob):
    gb = ob.RectilinearGrid(ob.arch, np.float64, size=(32, 8, 8), extent=(1, 1, 1), topology=("Periodic",) * 3)
    for bad in ({"q": STRAT}, {"b": 3.0}, {"b": lambda x, y, z, t: np.zeros((2, 2, 2))}, [("b", STRAT)]):
        with pytest.raises(ValueError):
            ob.NonhydrostaticModel(gb, advection=ob.WENO5(), tracers=("b",), background_fields=bad)
    m = ob.NonhydrostaticModel(gb, advection=ob.WENO5(), tracers=("b",),
                               background_fields={"b": ob.BackgroundField(lambda x, y, z, t, p: p * z, parameters=N2)})
    assert np.array_equal(m.background_fields["b"].parent(), table(O.RectilinearGrid(np.float64, size=(32, 8, 8), extent=(1, 1, 1),
                                                                                         topology=(O.Periodic,) * 3),
                                                                  ("c", "c", "c"), STRAT))
    with pytest.raises(ValueError):
        ob.set_background(m, "u", STRAT)


def test_background_on_two_gpus_matches_oracle():
    """runs tests/dist_background_check.py under torchrun when the box has >= 2 GPUs (skipped otherwise)"""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29536",
                          os.path.join(root, "tests", "dist_background_check.py")], capture_output=True, text=True, timeout=600)
    assert "DIST_BACKGROUND_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
