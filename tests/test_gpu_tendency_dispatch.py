"""Which tendency kernels each model configuration launches.  One time step runs under torch.profiler with CUDA activities, and
the multiset of tendency-related kernels it launched (tendency_*, relaxation_pass_kernel, boundary_flux_kernel; demangled
names with their template arguments, without the parameter list) must equal the literal list of the configuration.  The
parity tests compare results, which agree to 1e-12 whichever kernel computed them; this file pins the choice itself: the
fused kernel and its instantiation, the closure-only and background-only pre-passes, the relaxation pass, and the per-field
TMA, 2-D direct-load, shared-face and one-cell kernels.  Counts are per time step: three stages for RK3, one for AB2."""
import collections
import json

import numpy as np
import pytest

import oracle as O
from test_gpu_advection_walls import CASES as WALLS
from test_gpu_background import SHEAR, STRAT, build_bg
from test_gpu_parity import CONFIGS, init_state

pytestmark = pytest.mark.gpu

KEPT = ("tendency_", "relaxation_pass_kernel", "boundary_flux_kernel")


@pytest.fixture(scope="module")
def ob():
    import ocean_b200 as ob
    ob.arch = ob.B200()
    return ob


def kernel_name(name):
    """'void ob::k<double, 1>(ob::Args<double>)' -> 'ob::k<double, 1>'"""
    if name.startswith("void "):
        name = name[len("void "):]
    depth = 0
    for i, ch in enumerate(name):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            return name[:i]
    return name


def launched_kernels(ob, model, dt, trace_path):
    """the tendency-related kernels of one time step, after one step outside the profiler"""
    from torch.profiler import ProfilerActivity, profile
    ob.time_step(model, dt)
    ob.sync()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        ob.time_step(model, dt)
        ob.sync()
    prof.export_chrome_trace(str(trace_path))
    with open(trace_path) as f:
        events = json.load(f)["traceEvents"]
    names = (kernel_name(e["name"]) for e in events if e.get("cat") == "kernel")
    return collections.Counter(n for n in names if any(k in n for k in KEPT))


HEADLINE = dict(size=(32, 16, 16), topology=(O.Periodic,) * 3, extent=(1, 1, 1), adv="WENO5", tracers=("b",), buoyancy=True,
                ts="RungeKutta3", dt=2e-3)
SPONGE = (20.0, ("z", -0.9, 0.1), ("z", 0.0, 0.5))
TILT = 0.2
FLAT_Z = CONFIGS["c1_2d_flat_weno_ab2"]
C3 = CONFIGS["c3_fused_stretched_weno_rk3"]
AMD_C3 = CONFIGS["amd_c3_fused_split"]
# w with a non-zero constant Flux on the top wall: the fused Bounded-z kernel does not apply it, so the model takes the general
# kernels for every field, and the closure-only pre-pass of AMD is not launched either
AMD_C3_W_FLUX = dict(AMD_C3, bcs=dict(AMD_C3["bcs"], w={"top": ("Flux", 1e-4)}))


# name: (configuration, background_fields, forcing, float type, use_fast_kernels, expected kernels per time step)
CASES = {
    # triply periodic, one tracer: the fused kernel computes everything (stage 1 without G^-)
    "headline": (HEADLINE, None, None, np.float64, True, {
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, false, false, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, true, false, 12, false>": 2}),
    "headline_f32": (HEADLINE, None, None, np.float32, True, {
        "ob::fz::tendency_fused_kernel<float, true, 0, 1, false, false, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<float, true, 0, 1, true, false, 12, false>": 2}),
    # no tracer: the three-field variant
    "no_tracer": (dict(HEADLINE, tracers=(), buoyancy=False), None, None, np.float64, True, {
        "ob::fz::tendency_fused_kernel<double, true, 0, 0, false, false, 8, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 0, 0, true, false, 8, false>": 2}),
    # tracers beyond the first: the per-field TMA kernel (Ny % 8 == 0) ...
    "three_tracers_ny16": (dict(HEADLINE, tracers=("b", "c", "d")), None, None, np.float64, True, {
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, false, false, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, true, false, 12, false>": 2,
        "ob::tma::tendency_tma_kernel<double, true, 3>": 6}),
    "three_tracers_ny16_f32": (dict(HEADLINE, tracers=("b", "c", "d")), None, None, np.float32, True, {
        "ob::fz::tendency_fused_kernel<float, true, 0, 1, false, false, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<float, true, 0, 1, true, false, 12, false>": 2,
        "ob::tma::tendency_tma_kernel<float, true, 3>": 6}),
    # ... or the shared-face general kernel (Ny = 9)
    "three_tracers_ny9": (dict(HEADLINE, size=(32, 9, 16), tracers=("b", "c", "d")), None, None, np.float64, True, {
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, false, false, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, true, false, 12, false>": 2,
        "ob::tendency_shared_kernel<double, 3, 0, 0, 0>": 6}),
    # Flat z: the 2-D direct-load kernel per field; with a closure the one-cell general kernel
    "flat_z": (FLAT_Z, None, None, np.float64, True, {
        "ob::fast::tendency_fast_kernel<double, true, 0>": 1,
        "ob::fast::tendency_fast_kernel<double, true, 1>": 1,
        "ob::fast::tendency_fast_kernel<double, true, 2>": 1}),
    "flat_z_closure": (dict(FLAT_Z, closure=("ThreeDimensional", 1e-3, 1e-3)), None, None, np.float64, True, {
        "ob::tendency_general_kernel<double, 0, false>": 1,
        "ob::tendency_general_kernel<double, 1, false>": 1,
        "ob::tendency_general_kernel<double, 2, false>": 1}),
    # C3 class: Bounded stretched z, ScalarDiffusivity computed by the fused Bounded-z variant itself
    "c3": (C3, None, None, np.float64, True, {
        "ob::fz::tendency_fused_kernel<double, true, 1, 1, false, false, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 1, 1, true, false, 12, false>": 2}),
    # AMD: the closure-only pre-pass (C3-class shared-face kernel), then the accumulate form
    "c3_amd": (AMD_C3, None, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 1, 1, 0>": 3,
        "ob::tendency_shared_kernel<double, 1, 1, 1, 0>": 3,
        "ob::tendency_shared_kernel<double, 2, 1, 1, 0>": 3,
        "ob::tendency_shared_kernel<double, 3, 1, 1, 0>": 3,
        "ob::fz::tendency_fused_kernel<double, true, 1, 1, false, true, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 1, 1, true, true, 12, false>": 2}),
    # any closure on the triply periodic variant: the closure-only pre-pass of the generic shared-face kernel
    "periodic_scalar_diffusivity": (CONFIGS["scalar3d_periodic_fused_split"], None, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 0, 1, 0>": 3,
        "ob::tendency_shared_kernel<double, 1, 0, 1, 0>": 3,
        "ob::tendency_shared_kernel<double, 2, 0, 1, 0>": 3,
        "ob::tendency_shared_kernel<double, 3, 0, 1, 0>": 3,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, false, true, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, true, true, 12, false>": 2}),
    # backgrounds on u and b: the background-only pre-pass, then the accumulate form
    "background": (HEADLINE, {"u": SHEAR, "b": STRAT}, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 0, 0, 2>": 3,
        "ob::tendency_shared_kernel<double, 1, 0, 0, 2>": 3,
        "ob::tendency_shared_kernel<double, 2, 0, 0, 2>": 3,
        "ob::tendency_shared_kernel<double, 3, 0, 0, 2>": 3,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, false, true, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, true, true, 12, false>": 2}),
    # a background without a tracer: the three-field variant has no accumulate form, so every field takes the general kernel
    "background_no_tracer": (dict(HEADLINE, tracers=(), buoyancy=False), {"u": SHEAR}, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 0, 0, 1>": 3,
        "ob::tendency_shared_kernel<double, 1, 0, 0, 1>": 3,
        "ob::tendency_shared_kernel<double, 2, 0, 0, 1>": 3}),
    # relaxation of b: in Float64 the pointwise pass and the accumulate form, in Float32 the FRC instantiation
    "relaxation_b": (HEADLINE, None, {"b": SPONGE}, np.float64, True, {
        "ob::fz::relaxation_pass_kernel<double>": 3,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, false, true, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, true, true, 12, false>": 2}),
    "relaxation_b_f32": (HEADLINE, None, {"b": SPONGE}, np.float32, True, {
        "ob::fz::tendency_fused_kernel<float, true, 0, 1, false, false, 12, true>": 1,
        "ob::fz::tendency_fused_kernel<float, true, 0, 1, true, false, 12, true>": 2}),
    # a forced third tracer: the general kernel for it, the TMA kernel for the unforced second one
    "forced_third_tracer": (dict(HEADLINE, tracers=("b", "c", "d")), None, {"d": SPONGE}, np.float64, True, {
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, false, false, 12, false>": 1,
        "ob::fz::tendency_fused_kernel<double, true, 0, 1, true, false, 12, false>": 2,
        "ob::tma::tendency_tma_kernel<double, true, 3>": 3,
        "ob::tendency_shared_kernel<double, 3, 0, 0, 0>": 3}),
    # tilted gravity and vertically implicit diffusion: the shared-face kernel for every field
    "tilted_gravity": (dict(HEADLINE, size=(32, 8, 16), topology=(O.Periodic, O.Periodic, O.Bounded),
                            tilt=(np.sin(TILT), 0.0, np.cos(TILT))), None, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 1, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 2, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 3, 0, 0, 0>": 3}),
    "vertically_implicit": (CONFIGS["vitd_c3_stretched_weno"], None, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 1, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 2, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 3, 0, 0, 0>": 3}),
    # the headline after use_fast_kernels(False)
    "headline_general": (HEADLINE, None, None, np.float64, False, {
        "ob::tendency_shared_kernel<double, 0, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 1, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 2, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 3, 0, 0, 0>": 3}),
    "c3_amd_w_flux": (AMD_C3_W_FLUX, None, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 1, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 1, 1, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 2, 1, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 3, 1, 0, 0>": 3}),
    # the wall cases of test_gpu_advection_walls.py: a Bounded x at the seam size (several x, y tiles and z chunks) and any
    # scheme but the uniform WENO5 take the generic shared-face kernel, a 2-D Flat-z grid with a Bounded x the one-cell kernel
    "walls_weno_bounded_x_seam": (WALLS["WENO5-BPP-seam"][0], None, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 1, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 2, 0, 0, 0>": 3,
        "ob::tendency_shared_kernel<double, 3, 0, 0, 0>": 3}),
    "walls_upwind1_bounded_z": (WALLS["U1-PPB-seam"][0], None, None, np.float64, True, {
        "ob::tendency_shared_kernel<double, 0, 0, 0, 0>": 1,
        "ob::tendency_shared_kernel<double, 1, 0, 0, 0>": 1,
        "ob::tendency_shared_kernel<double, 2, 0, 0, 0>": 1,
        "ob::tendency_shared_kernel<double, 3, 0, 0, 0>": 1}),
    "walls_upwind3_bounded_x_flat_z": (WALLS["U3-BPF-seam"][0], None, None, np.float64, True, {
        "ob::tendency_general_kernel<double, 0, false>": 1,
        "ob::tendency_general_kernel<double, 1, false>": 1,
        "ob::tendency_general_kernel<double, 2, false>": 1,
        "ob::tendency_general_kernel<double, 3, false>": 1}),
    # ... and (P, P, B) with the uniform WENO5 at Nx = 32 the fused Bounded-z kernel, in both precisions
    "walls_weno_bounded_z_fused": (WALLS["WENO5-PPB-fused"][0], None, None, np.float64, True, {
        "ob::fz::tendency_fused_kernel<double, true, 1, 1, true, false, 12, false>": 1}),
    "walls_weno_bounded_z_fused_f32": (WALLS["WENO5-PPB-fused"][0], None, None, np.float32, True, {
        "ob::fz::tendency_fused_kernel<float, true, 1, 1, true, false, 12, false>": 1}),
}


@pytest.mark.parametrize("name", list(CASES))
def test_tendency_kernels_per_step(ob, name, tmp_path):
    cfg, bg, forcing, FT, fast, want = CASES[name]
    mo, mb = build_bg(ob, cfg, FT, bg, forcing)
    init_state(mo, mb, ob, 91)
    if not fast:
        mb.use_fast_kernels(False)
    got = launched_kernels(ob, mb, cfg["dt"], tmp_path / "trace.json")
    assert dict(got) == want, f"{name}: launched {dict(sorted(got.items()))}"
