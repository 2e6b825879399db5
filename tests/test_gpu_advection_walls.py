"""Every advection scheme of the C ABI at every kind of Bounded wall, and across the tile seams of the general tendency kernels,
against the oracle.

Next to a Bounded wall every reconstruction wider than second order falls back to second order
(topologically_conditional_interpolation.jl:19-80).  Which faces fall back depends on the scheme's buffer width Nᴮ, on the side
(the left- and right-biased predicates differ by one) and on the staggering.  A wrong buffer width or an off-by-one predicate
changes the tendency only in the one or two planes next to a wall, and only for the schemes that share that width, so besides
the whole-field comparison each case compares the Nᴮ + 1 planes next to every wall against their own scale and names the
wall that differs.

Two sizes per scheme and grid: 9 x 8 x 7 has fallback faces and high-order faces in every Bounded dimension; 40 x 17 x 37
crosses every seam of tendency_shared_kernel, whose 32 x 8 thread blocks finish 31 x 7 cells (two x tiles, the second one
ragged; three y tiles, the last one ragged) and which walks z in chunks of 32 levels (32 + 5).  (P, P, B) with the uniform
WENO5 also runs at Nx = 32, which the fused Bounded-z kernel takes in both precisions (at Nx = 40 the general kernel runs).

No closure: the advective fluxes are the only terms near a wall that differ between schemes.  Float64 is held to 1e-12, as
in test_gpu_parity.py; Float32 to the conditioning yardstick of test_gpu_float32.py."""
import os
import re

import numpy as np
import pytest

import oracle as O
from test_gpu_float32 import FACTOR, run_model_case
from test_gpu_parity import _zf, build_models, compare_fields, init_state, relerr

B, P, F = O.Bounded, O.Periodic, O.Flat


def abi_schemes():
    """every OB200_ADV_* of the C header, in order, as a scheme name of the builders (None for no advection; WENO5 with Z and
    with JS weights).  Read from the header rather than from the library, so that collecting this file needs no build; a scheme
    added to the ABI appears here under its header name and fails loudly until the builders know it."""
    header = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "ocean_b200.h")
    with open(header) as f:
        abi = sorted((int(v), n) for n, v in re.findall(r"OB200_ADV_(\w+)\s*=\s*(\d+)", f.read()))
    known = {"NONE": [None], "CENTERED2": ["CenteredSecondOrder"], "CENTERED4": ["CenteredFourthOrder"],
             "UPWIND1": ["UpwindBiasedFirstOrder"], "UPWIND3": ["UpwindBiasedThirdOrder"], "UPWIND5": ["UpwindBiasedFifthOrder"],
             "WENO5": ["WENO5", "WENO5js"]}
    return [s for _, n in abi for s in known.get(n, [n])]


SCHEMES = abi_schemes()
SHORT = {None: "none", "CenteredSecondOrder": "C2", "CenteredFourthOrder": "C4", "UpwindBiasedFirstOrder": "U1",
         "UpwindBiasedThirdOrder": "U3", "UpwindBiasedFifthOrder": "U5", "WENO5": "WENO5", "WENO5js": "WENO5js",
         "WENO5grid": "WENO5grid", "WENO5grid_js": "WENO5grid_js"}
# name: (topology, stretched z)
GRIDS = {"BPP": ((B, P, P), False), "PBP": ((P, B, P), False), "PPB": ((P, P, B), False), "PPB_stretched": ((P, P, B), True),
         "BBB": ((B, B, B), False), "BPF": ((B, P, F), False), "BBF": ((B, B, F), False)}
SIZES = {"small": (9, 8, 7), "seam": (40, 17, 37)}
EXTENT = (1.0, 0.75, 0.5)         # unequal spacings, so that a dimension mixed up with another shows; exact in Float32


def config(scheme, grid, size, ts):
    topo, stretched = GRIDS[grid]
    n = tuple(size[:2]) if topo[2] == F else tuple(size)
    cfg = dict(size=n, topology=topo, adv=scheme, tracers=("b",), buoyancy=True, f=0.3, ts=ts, dt=2e-3)
    if stretched:
        cfg["coords"] = dict(x=(0, EXTENT[0]), y=(0, EXTENT[1]), z=EXTENT[2] * _zf(n[2]))
    else:
        cfg["extent"] = EXTENT[:len(n)]
    return cfg


def _cases():
    """name: (configuration, seed); RK3 and AB2 alternate over schemes and grids"""
    out = {}
    for si, scheme in enumerate(SCHEMES):
        for gi, grid in enumerate(GRIDS):
            ts = ("RungeKutta3", "QuasiAdamsBashforth2")[(si + gi) % 2]
            for size in SIZES:
                out[f"{SHORT.get(scheme, scheme)}-{grid}-{size}"] = (config(scheme, grid, SIZES[size], ts), 100 + 10 * si + gi)
    for si, scheme in enumerate(("WENO5grid", "WENO5grid_js")):
        ts = ("RungeKutta3", "QuasiAdamsBashforth2")[si]
        for size in SIZES:
            out[f"{scheme}-PPB_stretched-{size}"] = (config(scheme, "PPB_stretched", SIZES[size], ts), 200 + si)
    for si, scheme in enumerate(("WENO5", "WENO5js")):
        ts = ("QuasiAdamsBashforth2", "RungeKutta3")[si]
        out[f"{scheme}-PPB-fused"] = (config(scheme, "PPB", (32, 17, 37), ts), 210 + si)
    return out


CASES = _cases()


@pytest.fixture(scope="module")
def ob():
    import ocean_b200 as ob
    ob.arch = ob.B200()
    return ob


def buffer_width(model):
    """Nᴮ of the model's scheme (0 for no advection)"""
    return getattr(model.advection, "buffer", 0)


def check_wall_slabs(name, Gb, Go, topology, NB):
    """the Nᴮ + 1 planes next to each side of every Bounded dimension, relative to their own maximum (floored at 1e-3 of the
    field's): an error confined to the fallback faces is not hidden by the scale of the whole field"""
    floor = 1e-3 * np.max(np.abs(Go))
    for d in range(3):
        if topology[d] != B:
            continue
        for side, sl in (("low", slice(0, NB + 1)), ("high", slice(-(NB + 1), None))):
            ix = [slice(None)] * 3
            ix[d] = sl
            a, b = Gb[tuple(ix)], Go[tuple(ix)]
            scale = max(np.max(np.abs(b)), floor, 1e-300)
            e = float(np.max(np.abs(a - b)) / scale)
            assert e < 1e-12, f"tendency {name}: {'xyz'[d]} {side} wall, {NB + 1} planes: rel err {e:.3e}"


def check_walls_closed(mb, topology, what):
    """the wall-normal velocity is exactly zero on both walls (Face indices 1 and N + 1) of every Bounded dimension"""
    for d in range(3):
        if topology[d] != B:
            continue
        n = "uvw"[d]
        a = mb.fields[n].interior()
        for side, i in (("low", 0), ("high", -1)):
            worst = float(np.max(np.abs(np.take(a, i, axis=d))))
            assert worst == 0, f"{what}: {n} on the {'xyz'[d]} {side} wall is {worst:.3e}, not 0"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_advection_walls_f64(ob, name):
    cfg, seed = CASES[name]
    mo, mb = build_models(ob, cfg, np.float64)
    init_state(mo, mb, ob, seed)
    mo.calculate_tendencies()
    ob.calculate_tendencies(mb)
    g = mo.grid
    NB = buffer_width(mo)
    worst_G = worst_state = 0.0
    for n in mo.names:
        Go = mo.Gn[n][O.R(1, g.Nx), O.R(1, g.Ny), O.R(1, g.Nz)]
        Gb = mb.Gn[n].interior()[:g.Nx, :g.Ny, :g.Nz]
        check_wall_slabs(n, Gb, Go, g.topology, NB)
        e = relerr(Gb, Go)
        assert e < 1e-12, f"tendency {n}: rel err {e:.3e}"
        worst_G = max(worst_G, e)
    for step in range(1, 4):
        mo.time_step(cfg["dt"])
        ob.time_step(mb, cfg["dt"])
        worst_state = max(worst_state, compare_fields(mo, mb, 1e-12, f"step {step}"))
        assert relerr(mb.pressures["pNHS"].interior(), mo.pNHS.interior) < 1e-9, f"pNHS, step {step}"
        check_walls_closed(mb, g.topology, f"step {step}")
    assert mb.diagnostics()["max_abs_div"] < 1e-10
    print(f"F64 walls/{name}: tendencies {worst_G:.3e} states {worst_state:.3e}")


# Float32 checks over the relative bound on a B200, by case: {check: finding}.  Only these checks are exempt from it (states keep
# the absolute 1e-5), at least one of them must still exceed it, and every other check of the case is asserted.  None of them is
# a wall-fallback error: Float64 agrees to 1e-14 on the same cases, wall planes included.
#  * (P, P, B) stretched at 40 x 17 x 37: the largest Float32 errors of the projected w and of the tendencies sit in the top
#    levels, where the stretched spacing is finest, for every scheme and on most seeds (set/w 4.4 - 6.2x, tendencies up
#    to 7.4x, the stepped states with them); the absolute 1e-5 on states and the pNHS bound stay asserted; open.
#  * the FFT solve of (B, P, Flat) at 40 x 17 (transform lengths that are not powers of two) gives pNHS 6.2x on this seed
#    (1.4 - 4.2x on others).
#  * the two Z-WENO tendencies exceed on this seed only (1.2 - 1.5x on three others), in the interior, not next to a wall; IEEE
#    divisions in the Float32 reconstruction (4.5x) and no FMA contraction (4.9x) do not change that.
STRETCHED_CHECKS = ("set/w",) + tuple(f"{s}/{n}" for s in ("G", "step1", "step2", "step3") for n in "uvwb")
STRETCHED_TOP = "Float32 stretched z at 40 x 17 x 37: largest errors in the finest top levels"
F32_OPEN = {
    "C4-PPB_stretched-seam": dict.fromkeys(STRETCHED_CHECKS, STRETCHED_TOP),
    "U3-PPB_stretched-seam": dict.fromkeys(STRETCHED_CHECKS, STRETCHED_TOP),
    "WENO5js-PPB_stretched-seam": dict.fromkeys(STRETCHED_CHECKS, STRETCHED_TOP),
    "WENO5grid-PPB_stretched-seam": dict.fromkeys(STRETCHED_CHECKS, STRETCHED_TOP),
    "WENO5-BPF-seam": {"step1/pNHS": "Float32 FFT solve at 40 x 17, non-power-of-two lengths"},
    "WENO5-PBP-seam": {"G/w": "Z-WENO tendency, interior, this seed"},
    "WENO5-BBB-seam": {"G/v": "Z-WENO tendency, interior, this seed"},
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_advection_walls_f32(ob, name):
    cfg, seed = CASES[name]
    open_checks = F32_OPEN.get(name, {})
    ratios = run_model_case(ob, f"walls/{name}", build_models, cfg, seed, expected_over=open_checks)
    over = {c: r for c, r in ratios.items() if r > FACTOR}
    if open_checks:
        assert over, f"{name}: every exempt check is within the bound now ({ratios}); it is no longer an open finding"
        pytest.xfail("; ".join(f"{c}: {r:.2f}x the Float32 yardstick ({open_checks[c]})" for c, r in over.items()))
