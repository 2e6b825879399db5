"""Array-valued Flux / Value / Gradient boundary conditions on the CUDA path against the oracle with the same arrays
(bc_array_reference.py): halo fills (and, filled with a constant, bit for bit against the constant condition), model steps on the configurations that reach every tendency path (fused Bounded-z
kernel, its accumulate form after the closure split, a second tracer on the general kernels, implicit vertical diffusion, y sides,
all six sides, a Flat tangential dimension, Relaxation forcing), the fused kernel against the general ones, the launch count of the
boundary-plane pass, constant-filled arrays against constants, values changed between steps, the flux-budget known answer and
checkpoint / resume."""
import numpy as np
import pytest

import oracle as O
from bc_array_reference import array_bc, set_values, tangential_shape
from relaxation_reference import ForcedNonhydrostaticModel
from test_gpu_parity import CONFIGS, _zf, compare_fields, init_state, make_pair, relerr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ob():
    import ocean_b200 as ob
    ob.arch = ob.B200()
    return ob


def random_arrays(go, spec, seed):
    """spec = {name: {side: (kind, amplitude)}} -> {name: {side: (kind, Q)}} with Q uniform in ±amplitude around amplitude / 2"""
    rng = np.random.default_rng(seed)
    return {n: {s: (k, amp * (0.5 + rng.uniform(-1, 1, tangential_shape(go, s)))) for s, (k, amp) in d.items()}
            for n, d in spec.items()}


def build(ob, cfg, FT, arrays, forcing=None):
    """the models of test_gpu_parity.build_models with `arrays` = {name: {side: (kind, Q)}} on top of cfg's constant conditions,
    and Relaxation `forcing` as in test_gpu_forcing.build_forced"""
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
    if cfg.get("smagorinsky") is not None:
        clo_o, clo_b = O.SmagorinskyLilly(**cfg["smagorinsky"]), ob.SmagorinskyLilly(**cfg["smagorinsky"])
    if cfg.get("amd") is not None:
        clo_o, clo_b = O.AnisotropicMinimumDissipation(**cfg["amd"]), ob.AnisotropicMinimumDissipation(**cfg["amd"])
    cor_o = O.FPlane(cfg["f"]) if cfg.get("f") else None
    cor_b = ob.FPlane(cfg["f"]) if cfg.get("f") else None
    bu_o = O.Buoyancy(O.BuoyancyTracer(), None) if cfg.get("buoyancy") else None
    bu_b = ob.Buoyancy(ob.BuoyancyTracer(), None) if cfg.get("buoyancy") else None
    bcs_o = {n: {s: O.BoundaryCondition(*kv) for s, kv in d.items()} for n, d in cfg.get("bcs", {}).items()}
    bcs_b = {n: {s: ob.BoundaryCondition(*kv) for s, kv in d.items()} for n, d in cfg.get("bcs", {}).items()}
    for n, d in arrays.items():
        for s, (kind, Q) in d.items():
            bcs_o.setdefault(n, {})[s] = array_bc(kind, Q, s)
            bcs_b.setdefault(n, {})[s] = ob.BoundaryCondition(kind, Q)
    frc = {}
    for n, (rate, mask, target) in (forcing or {}).items():
        m = None if mask is None else ob.GaussianMask(*mask)
        t = ob.LinearTarget(*target) if isinstance(target, tuple) else target
        frc[n] = ob.Relaxation(rate, mask=m, target=t)
    mo = ForcedNonhydrostaticModel(go, forcing=frc, advection=ao, closure=clo_o, coriolis=cor_o, buoyancy=bu_o,
                                   tracers=cfg["tracers"], timestepper=cfg["ts"], boundary_conditions=bcs_o)
    mb = ob.NonhydrostaticModel(gb, advection=ab, closure=clo_b, coriolis=cor_b, buoyancy=bu_b, tracers=cfg["tracers"],
                                timestepper=cfg["ts"], boundary_conditions=bcs_b, forcing=frc)
    return mo, mb


C3 = CONFIGS["c3_fused_stretched_weno_rk3"]
C3_ARRAYS = {"u": {"top": ("Flux", -1e-2)}, "v": {"top": ("Flux", 5e-3)}, "b": {"top": ("Flux", 1e-3), "bottom": ("Gradient", 1e-1)}}
SPONGE = (20.0, ("z", -0.9, 0.1), None)
CASES = {
    # the fused Bounded-z kernel + the pass
    "c3_fused": (C3, C3_ARRAYS, None),
    # AB2; the second tracer c goes to the general kernels; a Value array on v
    "c3_js_ab2_second_tracer": (CONFIGS["c3_fused_js_ab2_no_closure"],
                                {"b": {"bottom": ("Flux", -2e-3)}, "c": {"top": ("Flux", 3e-3), "bottom": ("Gradient", 0.1)},
                                 "v": {"top": ("Value", 0.1)}}, None),
    # closure split: closure-only general kernel, then the accumulate form of the fused kernel
    "amd_split": (CONFIGS["amd_c3_fused_split"], C3_ARRAYS, None),
    # the pass before the implicit vertical diffusion step
    "vitd": (CONFIGS["vitd_c3_stretched_weno"], C3_ARRAYS, None),
    # y sides (v is normal there)
    "channel_y_sides": (CONFIGS["channel_bounded_yz_weno"],
                        {"u": {"south": ("Flux", 1e-2), "north": ("Value", 0.2)}, "w": {"north": ("Gradient", 0.3)},
                         "b": {"south": ("Flux", -2e-3), "north": ("Gradient", 0.1), "top": ("Flux", 1e-3)}}, None),
    # all six sides, x included
    "box_all_sides": (CONFIGS["box_bbb_upwind5_vertical"],
                      {"b": {"west": ("Flux", 2e-3), "east": ("Value", 0.3), "south": ("Gradient", -0.2), "north": ("Flux", -1e-3),
                             "bottom": ("Flux", 1e-3), "top": ("Gradient", 0.1)},
                       "u": {"south": ("Flux", 1e-2), "top": ("Flux", -1e-2)}, "v": {"west": ("Flux", 5e-3), "bottom": ("Value", 0.1)},
                       "w": {"east": ("Gradient", 0.2), "north": ("Flux", 2e-3)}}, None),
    # a Flat tangential dimension: y sides of a (Periodic, Bounded, Flat) grid take (Nx, 1) arrays
    "flat_2d": (CONFIGS["smagorinsky_2d_flat"], {"c": {"south": ("Flux", 1e-2), "north": ("Value", 0.5)}, "u": {"north": ("Flux", -1e-2)}},
                None),
    # with Relaxation forcing on the same fields
    "c3_fused_sponge": (C3, C3_ARRAYS, {"u": SPONGE, "v": SPONGE, "b": (20.0, ("z", -0.9, 0.1), ("z", 0.0, 0.5))}),
}


@pytest.mark.parametrize("name", list(CASES))
def test_bc_arrays_tendencies_and_steps_match_oracle_f64(ob, name):
    cfg, spec, forcing = CASES[name]
    go = make_pair(ob, np.float64, cfg["size"], cfg["topology"], coords=cfg.get("coords"), extent=cfg.get("extent"))[0]
    mo, mb = build(ob, cfg, np.float64, random_arrays(go, spec, 71), forcing)
    init_state(mo, mb, ob, 72)
    compare_fields(mo, mb, 1e-12, "after set!")
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


@pytest.mark.parametrize("name", ["c3_fused", "box_all_sides"])
def test_bc_arrays_steps_match_oracle_f32(ob, name):
    cfg, spec, forcing = CASES[name]
    go = make_pair(ob, np.float32, cfg["size"], cfg["topology"], coords=cfg.get("coords"), extent=cfg.get("extent"))[0]
    mo, mb = build(ob, cfg, np.float32, random_arrays(go, spec, 73), forcing)
    init_state(mo, mb, ob, 74)
    for step in range(4):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        compare_fields(mo, mb, 1e-5, f"f32 step {step + 1}")


# ---- halo fills ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("FT", [np.float64, np.float32])
@pytest.mark.parametrize("stretched", [False, True])
def test_value_gradient_array_halo_fills(ob, FT, stretched):
    """all six sides of a (Bounded, Bounded, Bounded) box, Center and Face fields (every side not normal to the Face location):
    random arrays against the oracle to the rounding of the extrapolation (the CUDA fill contracts cI + grad * Δ into one FMA,
    as it does for constants: test_gpu_parity.test_fill_halo_value_gradient_bcs), every cell the fill does not write bit for
    bit, and arrays filled with a constant bit for bit against the constant condition on the CUDA path"""
    coords = dict(x=(0, 1.3), y=(-1, 1), z=_zf(7) if stretched else (-0.7, 0))
    go, gb = make_pair(ob, FT, (9, 6, 7), (O.Bounded,) * 3, coords=coords, halo=(3, 2, 2))
    rng = np.random.default_rng(75)
    sides = ("west", "east", "south", "north", "bottom", "top")
    tol = 4 * np.finfo(FT).eps
    for loc in (("c", "c", "c"), ("f", "c", "c"), ("c", "f", "c"), ("c", "c", "f")):
        L = tuple({"c": "Center", "f": "Face"}[l] for l in loc)
        bo, bb, bconst, bfill = {}, {}, {}, {}
        for s_i, s in enumerate(sides):
            if loc[s_i // 2] == "f":
                continue
            kind = ("Value", "Gradient")[(s_i + len(bo)) % 2]
            Q = rng.uniform(-1, 1, tangential_shape(go, s))
            bo[s], bb[s] = array_bc(kind, Q, s), ob.BoundaryCondition(kind, Q)
            v = float(Q[0, 0])
            bconst[s], bfill[s] = ob.BoundaryCondition(kind, v), ob.BoundaryCondition(kind, np.full(Q.shape, v))
        fo = O.Field(go, loc, O.FieldBoundaryConditions(go, loc, **bo))
        fb, fc, ff = ob.Field(L, gb, bb), ob.Field(L, gb, bconst), ob.Field(L, gb, bfill)
        a = rng.uniform(-1, 1, fo.parent.shape).astype(FT)
        fo.parent[...] = a
        for f in (fb, fc, ff):
            f.set_parent(a)
        O.fill_halo_regions(fo)
        ob.fill_halo_regions([fb, fc, ff])
        got = fb.parent()
        assert relerr(got, fo.parent) < tol, loc
        written = fo.parent != a
        assert written.any() and np.array_equal(got[~written], a[~written]), loc
        assert np.array_equal(ff.parent(), fc.parent()), loc


# ---- paths ------------------------------------------------------------------------------------------------------------------------
def test_bc_arrays_fused_kernel_agrees_with_general_kernels(ob):
    cfg = CASES["c3_fused"][0]
    go = make_pair(ob, np.float64, cfg["size"], cfg["topology"], coords=cfg.get("coords"))[0]
    arrays = random_arrays(go, C3_ARRAYS, 76)
    mo, m1 = build(ob, cfg, np.float64, arrays)
    _, m2 = build(ob, cfg, np.float64, arrays)
    m2.use_fast_kernels(False)
    init_state(mo, m1, ob, 77)
    init_state(mo, m2, ob, 77)
    ob.calculate_tendencies(m1)
    ob.calculate_tendencies(m2)
    for n in m1.names:
        assert relerr(m1.Gn[n].interior(), m2.Gn[n].interior()) < 1e-13, f"tendency {n}"
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert relerr(m1.fields[n].interior(), m2.fields[n].interior()) < 1e-13, n


def _constant_pair(ob, fast):
    """C3 with the constant top Flux of u and b, once as constants and once as arrays filled with them"""
    cfg = CASES["c3_fused"][0]
    go = make_pair(ob, np.float64, cfg["size"], cfg["topology"], coords=cfg.get("coords"))[0]
    filled = {n: {s: (k, np.full(tangential_shape(go, s), v)) for s, (k, v) in d.items()} for n, d in cfg["bcs"].items()}
    mo, mc = build(ob, cfg, np.float64, {})
    _, ma = build(ob, cfg, np.float64, filled)
    for m in (mc, ma):
        m.use_fast_kernels(fast)
        init_state(mo, m, ob, 78)
    return cfg, mc, ma


def test_launch_count_grows_by_one_pass_per_stage(ob):
    """the fused path is still taken: one RK3 step launches exactly 3 kernels more (one boundary-plane pass per stage)"""
    cfg, mc, ma = _constant_pair(ob, True)
    counts = []
    for m in (mc, ma):
        ob.time_step(m, cfg["dt"])          # first step: one-time set-up outside the count
        ob.sync()
        n0 = ob.launch_count()
        ob.time_step(m, cfg["dt"])
        ob.sync()
        counts.append(ob.launch_count() - n0)
    assert counts[1] == counts[0] + 3, counts


def test_constant_filled_arrays_match_constant_bcs(ob):
    """general kernels: G^n and the state bit for bit; fused path: within 1e-12 (the constant is added inside the kernel there)"""
    cfg, mc, ma = _constant_pair(ob, False)
    ob.calculate_tendencies(mc)
    ob.calculate_tendencies(ma)
    for n in mc.names:
        assert np.array_equal(mc.Gn[n].parent(), ma.Gn[n].parent()), f"tendency {n}"
    for _ in range(3):
        ob.time_step(mc, cfg["dt"])
        ob.time_step(ma, cfg["dt"])
    for n in mc.names:
        assert np.array_equal(mc.fields[n].parent(), ma.fields[n].parent()), n
    cfg, mc, ma = _constant_pair(ob, True)
    for _ in range(3):
        ob.time_step(mc, cfg["dt"])
        ob.time_step(ma, cfg["dt"])
    for n in mc.names:
        assert relerr(ma.fields[n].interior(), mc.fields[n].interior()) <= 1e-12, n


def test_values_changed_between_steps(ob):
    """new values set between steps (a callback's `bc.condition .= Q`) take effect from the next step on, as on the oracle updated
    the same way"""
    cfg = CASES["c3_fused"][0]
    go = make_pair(ob, np.float64, cfg["size"], cfg["topology"], coords=cfg.get("coords"))[0]
    mo, mb = build(ob, cfg, np.float64, random_arrays(go, C3_ARRAYS, 79))
    init_state(mo, mb, ob, 80)
    for step in range(4):
        if step in (1, 3):
            new = random_arrays(go, C3_ARRAYS, 81 + step)
            for n, d in new.items():
                for s, (_, Q) in d.items():
                    set_values(mo.fields[n], s, Q)
                    ob.set_boundary_condition_values(mb.fields[n], s, Q)
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        compare_fields(mo, mb, 1e-12, f"step {step + 1}")


def test_flux_budget_known_answer_on_cuda(ob):
    """no advection, no closure, a tracer at rest with a top Flux array: one forward-Euler step changes Σ c V by -Δt Σ Q A"""
    go, gb = make_pair(ob, np.float64, (32, 8, 12), (O.Periodic, O.Periodic, O.Bounded), coords=dict(x=(0, 2), y=(0, 1), z=_zf(12)))
    rng = np.random.default_rng(85)
    Q = rng.uniform(-1, 1, (32, 8))
    m = ob.NonhydrostaticModel(gb, advection=None, tracers=("c",), boundary_conditions={"c": {"top": ob.FluxBoundaryCondition(Q)}})
    ob.set_model(m, c=rng.uniform(-1, 1, (32, 8, 12)))
    i, j, k = O.R(1, 32), O.R(1, 8), O.R(1, 12)
    V = np.broadcast_to(go.V(i, j, k, "c", "c", "c"), (32, 8, 12))
    A = np.broadcast_to(go.Az(i, j, O.R(13), "c", "c", "f"), (32, 8, 1))[:, :, 0]
    before = np.sum(m.fields["c"].interior() * V)
    dt = 0.1
    ob.time_step(m, dt, euler=True)
    after = np.sum(m.fields["c"].interior() * V)
    want = -dt * np.sum(Q * A)
    assert abs((after - before) - want) <= 1e-13 * max(abs(before), abs(want))


def test_bc_arrays_checkpoint_resume_is_bitwise(ob, tmp_path):
    """the Checkpointer does not store boundary conditions (as in the reference): the restored model is built with the same arrays"""
    cfg = CASES["c3_fused"][0]
    go = make_pair(ob, np.float64, cfg["size"], cfg["topology"], coords=cfg.get("coords"))[0]
    arrays = random_arrays(go, C3_ARRAYS, 86)
    mo, m1 = build(ob, cfg, np.float64, arrays)
    init_state(mo, m1, ob, 87)
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
    path = ob.Checkpointer(m1, dir=str(tmp_path), prefix="ck").write()
    for _ in range(3):
        ob.time_step(m1, cfg["dt"])
    _, m2 = build(ob, cfg, np.float64, arrays)
    ob.Checkpointer.restore(m2, path)
    for _ in range(3):
        ob.time_step(m2, cfg["dt"])
    for n in m1.names:
        assert np.array_equal(m1.fields[n].parent(), m2.fields[n].parent()), n


def test_library_rejects_unsupported_sides(ob):
    """ob200_field_set_boundary_values fails with a message for a Periodic side, an Open side and the wall side of a Face field"""
    import ctypes
    gb = ob.RectilinearGrid(ob.arch, np.float64, size=(8, 6, 4), extent=(1, 1, 1), topology=("Periodic", "Bounded", "Bounded"))
    Q = np.zeros((8, 6))
    c = ob.CenterField(gb)
    w = ob.ZFaceField(gb)
    for f, side in ((c, 0), (w, 5), (w, 4)):
        with pytest.raises(ob.B200Error):
            ob._lib.check(ob.lib.ob200_field_set_boundary_values(f.handle, side, Q.ctypes.data_as(ctypes.c_void_p)))
    ob._lib.check(ob.lib.ob200_field_set_boundary_values(c.handle, 5, Q.ctypes.data_as(ctypes.c_void_p)))
    ob._lib.check(ob.lib.ob200_field_set_boundary_values(c.handle, 5, None))
