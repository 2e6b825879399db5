"""Relaxation forcing (src/Forcings/relaxation.jl) on the CUDA path against the oracle with the same forcing
(relaxation_reference.py): forced versions of the parity configurations that reach every tendency kernel (the fused persistent
kernel periodic and Bounded-z, its accumulate form after the closure split, the per-field fallback of a second tracer to the
general kernels, the general kernels in a channel, in 2-D and with vertically implicit diffusion), the fused kernel against the
general ones, the RK3 known answer, checkpoint / resume and the mirror's rejections."""
import numpy as np
import pytest

import oracle as O
from relaxation_reference import ForcedNonhydrostaticModel
from test_gpu_parity import CONFIGS, _zf, compare_fields, init_state, make_pair, relerr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ob():
    import ocean_b200 as ob
    ob.arch = ob.B200()
    return ob


def build_forced(ob, cfg, FT, forcing):
    """build_models of test_gpu_parity.py with `forcing` = {name: (rate, mask args or None, target)} given to both models;
    mask args = (dim, center, width); target = None, a number or (dim, intercept, gradient)"""
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
    bu_o = O.Buoyancy(O.BuoyancyTracer(), None) if cfg.get("buoyancy") else None
    bu_b = ob.Buoyancy(ob.BuoyancyTracer(), None) if cfg.get("buoyancy") else None
    bcs_o = bcs_b = None
    if cfg.get("bcs"):
        bcs_o = {n: {s: O.BoundaryCondition(*kv) for s, kv in d.items()} for n, d in cfg["bcs"].items()}
        bcs_b = {n: {s: ob.BoundaryCondition(*kv) for s, kv in d.items()} for n, d in cfg["bcs"].items()}
    frc = {}
    for n, (rate, mask, target) in forcing.items():
        m = None if mask is None else ob.GaussianMask(*mask)
        t = ob.LinearTarget(*target) if isinstance(target, tuple) else target
        frc[n] = ob.Relaxation(rate, mask=m, target=t)
    mo = ForcedNonhydrostaticModel(go, forcing=frc, advection=ao, closure=clo_o, coriolis=cor_o, buoyancy=bu_o,
                                   tracers=cfg["tracers"], timestepper=cfg["ts"], boundary_conditions=bcs_o)
    mb = ob.NonhydrostaticModel(gb, advection=ab, closure=clo_b, coriolis=cor_b, buoyancy=bu_b, tracers=cfg["tracers"],
                                timestepper=cfg["ts"], boundary_conditions=bcs_b, forcing=frc)
    return mo, mb


HEADLINE = dict(size=(32, 12, 16), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5", tracers=("b",), buoyancy=True,
                ts="RungeKutta3", dt=2e-3)
SPONGE = lambda rate: (rate, ("z", -0.9, 0.1), None)            # bottom sponge toward rest
CASES = {
    # b restored to a linear profile, u damped with a mask along x (fused periodic kernel)
    "headline_forced": (HEADLINE, {"b": (5.0, None, ("z", 0.1, 0.5)), "u": (8.0, ("x", 0.5, 0.15), None)}),
    # C3 physics with a bottom sponge on u, v, w and b (fused Bounded-z kernel)
    "c3_fused_sponge": (CONFIGS["c3_fused_stretched_weno_rk3"],
                        {"u": SPONGE(20.0), "v": SPONGE(20.0), "w": SPONGE(20.0), "b": (20.0, ("z", -0.9, 0.1), ("z", 0.0, 0.5))}),
    # AMD: closure-only general kernel + accumulate form of the fused kernel
    "amd_c3_split_sponge": (CONFIGS["amd_c3_fused_split"], {"u": SPONGE(20.0), "b": (10.0, ("z", -0.9, 0.1), ("z", 0.0, 0.5))}),
    # a second forced tracer: the per-field kernels hand it to the general kernels
    "second_tracer": (dict(HEADLINE, tracers=("b", "c"), ts="QuasiAdamsBashforth2"),
                      {"c": (3.0, ("y", 0.5, 0.2), 0.25), "b": (2.0, None, ("z", 0.0, 0.5))}),
    "channel_y_mask": (CONFIGS["channel_bounded_yz_weno"], {"u": (6.0, ("y", 0.1, 0.1), 0.3), "v": (6.0, ("y", 0.9, 0.1), None)}),
    "c1_2d_x_mask": (CONFIGS["c1_2d_flat_weno_ab2"], {"u": (4.0, ("x", 1.0, 0.5), None), "v": (2.0, None, 0.1)}),
    "vitd_c3_sponge": (CONFIGS["vitd_c3_stretched_weno"], {"u": SPONGE(20.0), "b": (10.0, ("z", -0.9, 0.1), ("z", 0.0, 0.5))}),
}


@pytest.mark.parametrize("name", list(CASES))
def test_forced_tendencies_and_steps_match_oracle_f64(ob, name):
    cfg, forcing = CASES[name]
    mo, mb = build_forced(ob, cfg, np.float64, forcing)
    init_state(mo, mb, ob, 61)
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


@pytest.mark.parametrize("name", ["headline_forced", "c3_fused_sponge"])
def test_forced_steps_match_oracle_f32(ob, name):
    cfg, forcing = CASES[name]
    mo, mb = build_forced(ob, cfg, np.float32, forcing)
    init_state(mo, mb, ob, 62)
    for step in range(3):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        compare_fields(mo, mb, 1e-5, f"f32 step {step + 1}")


@pytest.mark.parametrize("size,stretched", [((64, 40, 48), True), ((64, 13, 7), True), ((32, 12, 33), False)])
def test_forced_fused_kernel_agrees_with_general_kernels(ob, size, stretched):
    cfg = dict(CONFIGS["c3_fused_stretched_weno_rk3"], size=size)
    if stretched:
        cfg["coords"] = dict(x=(0, 2), y=(0, 1.5), z=_zf(size[2]))
    else:
        cfg.pop("coords")
        cfg["extent"], cfg["adv"] = (1, 1, 1), "WENO5"
    forcing = CASES["c3_fused_sponge"][1]
    mo, m1 = build_forced(ob, cfg, np.float64, forcing)
    _, m2 = build_forced(ob, cfg, np.float64, forcing)
    m2.use_fast_kernels(False)
    init_state(mo, m1, ob, 63)
    init_state(mo, m2, ob, 63)
    ob.calculate_tendencies(m1)
    ob.calculate_tendencies(m2)
    for n in m1.names:
        assert relerr(m1.Gn[n].interior(), m2.Gn[n].interior()) < 1e-12, f"tendency {n}"
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert relerr(m1.fields[n].interior(), m2.fields[n].interior()) < 1e-12, n


def test_rk3_relaxation_known_answer_on_cuda(ob):
    """a tracer at rest relaxing toward LinearTarget{:z} under GaussianMask{:z} on a stretched Bounded z: one RK3 step gives
    c₁ - T = (1 + z + z²/2 + z³/6)(c₀ - T), z = -rate mask Δt"""
    gb = ob.RectilinearGrid(ob.arch, np.float64, size=(32, 4, 16), x=(0, 1), y=(0, 1), z=_zf(16),
                            topology=("Periodic", "Periodic", "Bounded"))
    r = ob.Relaxation(2.0, mask=ob.GaussianMask("z", -0.7, 0.2), target=ob.LinearTarget("z", 1.5, 0.8))
    m = ob.NonhydrostaticModel(gb, advection=None, tracers=("c",), timestepper="RungeKutta3", forcing={"c": r})
    rng = np.random.default_rng(3)
    c0 = rng.uniform(-1, 1, m.fields["c"].size())
    ob.set_model(m, c=c0)
    z = gb.nodes(("Center",) * 3)[2]
    T = 1.5 + 0.8 * z
    x = -(2.0 * np.exp(-(z + 0.7) ** 2 / (2 * 0.2 ** 2))) * 0.3
    ob.time_step(m, 0.3)
    got = m.fields["c"].interior() - T
    assert np.max(np.abs(got - (1 + x + x ** 2 / 2 + x ** 3 / 6) * (c0 - T))) <= 1e-13 * np.max(np.abs(c0 - T))


def test_forced_checkpoint_resume_is_bitwise(ob, tmp_path):
    cfg, forcing = CASES["c3_fused_sponge"]
    mo, m1 = build_forced(ob, cfg, np.float64, forcing)
    init_state(mo, m1, ob, 64)
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
    path = ob.Checkpointer(m1, dir=str(tmp_path), prefix="ck").write()
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
    _, m2 = build_forced(ob, cfg, np.float64, forcing)
    ob.Checkpointer.restore(m2, path)
    for _ in range(3):
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert np.array_equal(m1.fields[n].parent(), m2.fields[n].parent()), n


def test_mirror_rejects_unsupported_forcing(ob):
    gb = ob.RectilinearGrid(ob.arch, np.float64, size=(32, 8), extent=(1, 1), topology=("Periodic", "Periodic", "Flat"))
    ok = ob.Relaxation(1.0)
    for bad in ({"u": lambda x, y, z, t: 0.0}, {"u": object()}, {"q": ok}, {"u": ob.Relaxation(1.0, mask=ob.GaussianMask("z", 0, 1))},
                {"v": ob.Relaxation(1.0, target=ob.LinearTarget("z", 0, 1))}):
        with pytest.raises(ValueError):
            ob.NonhydrostaticModel(gb, advection=ob.WENO5(), forcing=bad)
    with pytest.raises(ValueError):
        ob.Relaxation("1.0")
    ob.NonhydrostaticModel(gb, advection=ob.WENO5(), forcing={"u": ok})


def test_forcing_on_two_gpus_matches_oracle():
    """runs tests/dist_forcing_check.py under torchrun when the box has >= 2 GPUs (skipped otherwise)"""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29534",
                          os.path.join(root, "tests", "dist_forcing_check.py")], capture_output=True, text=True, timeout=600)
    assert "DIST_FORCING_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
