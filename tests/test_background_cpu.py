"""Background fields (src/Models/NonhydrostaticModels/background_fields.jl) without a device: the mirror's tabulation of a
background over the whole parent (halos, the extra Face point, Flat dimensions, the `parameters` form) against the reference's
pointwise evaluation, its rejections, the C layout of the new `background` member against ctypes, and two known answers of the
oracle with backgrounds (background_reference.py)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import oracle as O
from background_reference import BackgroundNonhydrostaticModel, table

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MLOC = {"c": "Center", "f": "Face"}


def _zf(n, p=1.5):
    return -np.linspace(1, 0, n + 1) ** p


class _MirrorView:
    """an oracle grid seen through the attributes background_table reads (topology, N, H, FT, F, C with .span)"""

    def __init__(self, g):
        from ocean_b200.grids import _OV
        self.topology = tuple({O.Periodic: "Periodic", O.Bounded: "Bounded", O.Flat: "Flat"}[t] for t in g.topology)
        self.N, self.H, self.FT = g.N, g.H, g.FT
        self.F = [_OV(v.parent, v.first) for v in g.nodesF]
        self.C = [_OV(v.parent, v.first) for v in g.nodesC]


GRIDS = {
    "ppb_stretched": dict(size=(6, 5, 8), x=(0, 2), y=(0, 1), z=_zf(8), topology=(O.Periodic, O.Periodic, O.Bounded)),
    "bbb": dict(size=(5, 4, 6), x=(0, 1), y=(-1, 1), z=(-2, 0), topology=(O.Bounded,) * 3),
    "flat_y": dict(size=(8, 6), x=(0, 1), z=(-1, 0), topology=(O.Periodic, O.Flat, O.Bounded)),
}
LOCS = [("f", "c", "c"), ("c", "f", "c"), ("c", "c", "f"), ("c", "c", "c")]


@pytest.mark.parametrize("FT", [np.float64, np.float32])
@pytest.mark.parametrize("grid", list(GRIDS))
def test_mirror_table_matches_pointwise_evaluation(grid, FT):
    from ocean_b200.model import BackgroundField, background_table
    g = O.RectilinearGrid(FT, **GRIDS[grid])
    f = lambda x, y, z, t, p: p["a"] * np.tanh((z + 0.5) / 0.1) + np.sin(3 * x) * np.cos(2 * y) + p["b"] * t
    for loc in LOCS:
        want = table(g, loc, f, parameters=dict(a=0.3, b=2.0), time=0.25)
        got = background_table(_MirrorView(g), tuple(MLOC[l] for l in loc),
                               BackgroundField(f, parameters=dict(a=0.3, b=2.0)), time=0.25)
        assert got.shape == g.parent_size(loc) and got.dtype == FT
        assert np.array_equal(got, want), loc


def test_table_covers_halos_face_point_and_flat():
    """B = z on a (Periodic, Flat, Bounded) grid: z halos are the function's values (no periodic wrap, no fill), a z-Face field
    has Nz + 1 interior faces, the Flat dimension has extent 1 and the bare-callable form equals the BackgroundField form"""
    from ocean_b200.model import background_table
    g = O.RectilinearGrid(np.float64, size=(4, 5), x=(0, 1), z=(-1, 0), topology=(O.Periodic, O.Flat, O.Bounded), halo=(3, 3))
    V = _MirrorView(g)
    t = background_table(V, ("Center", "Center", "Face"), lambda x, y, z, t: z)
    assert t.shape == (4 + 6, 1, 5 + 6 + 1)
    zF = np.array(g.nodesF[2].slice(-2, 5 + 4))
    assert np.array_equal(t[0, 0, :], zF)
    assert zF[0] < -1 and zF[-1] > 0                       # halos below the bottom and above the top, linearly extended
    x = background_table(V, ("Face", "Center", "Center"), lambda x, y, z, t: x)
    assert np.array_equal(x[:, 0, 0], np.array(g.nodesF[0].slice(-2, 4 + 3)))     # periodic x halos: node values, not wrapped
    assert x[0, 0, 0] < 0 and x[-1, 0, 0] >= 1


def test_table_rejections():
    from ocean_b200.model import BackgroundField, background_table
    g = _MirrorView(O.RectilinearGrid(np.float64, **GRIDS["bbb"]))
    with pytest.raises(ValueError):
        BackgroundField(3.0)
    with pytest.raises(ValueError):
        background_table(g, ("Center",) * 3, lambda x, y, z, t: np.zeros((2, 3, 4)))


def test_model_desc_background_offset_matches_header(tmp_path):
    """sizeof(ob200_model_desc) and offsetof(..., background) / (..., forcing) from the C header against _lib.ModelDesc"""
    from ocean_b200 import _lib as L
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ocean_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(ob200_model_desc), offsetof(ob200_model_desc, background),'
                   ' offsetof(ob200_model_desc, forcing), sizeof(((ob200_model_desc*)0)->background)); return 0; }\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [ctypes.sizeof(L.ModelDesc), L.ModelDesc.background.offset, L.ModelDesc.forcing.offset,
                   ctypes.sizeof(ctypes.c_void_p) * (3 + L.MAX_TRACERS)]


def _stratified_pair(grid_kw, adv_of, N2=3.0, seed=1):
    """two oracle models on the same projected state, one with B = N² z: returns (without, with)"""
    g = O.RectilinearGrid(np.float64, **grid_kw)
    out = []
    for bg in ({}, {"b": lambda x, y, z, t: N2 * z}):
        m = BackgroundNonhydrostaticModel(g, background_fields=bg, advection=adv_of(g), tracers=("b",))
        rng = np.random.default_rng(seed)
        st = {n: rng.uniform(-1, 1, m.fields[n].size()) for n in "uvwb"}
        if g.topology[2] == O.Bounded:
            st["w"][:, :, [0, -1]] = 0                     # no flow through the walls
        m.set(**st)
        m.calculate_tendencies()
        out.append(m)
    return out


ADV = {"WENO5": lambda g: O.WENO5(grid=g) if not all(g.regular) else O.WENO5(), "Centered2": lambda g: O.CenteredSecondOrder()}


@pytest.mark.parametrize("adv", list(ADV))
@pytest.mark.parametrize("grid", ["periodic", "bounded_z"])
def test_linear_stratification_known_answer_oracle(grid, adv):
    """with B = N² z and a divergence-free state, Gb(with B) - Gb(without) = -N² (w[k] + w[k+1]) / 2.  The triply periodic grid
    needs B's halos unwrapped (a wrapped N² z would jump at the top and bottom)"""
    kw = dict(size=(8, 6, 12), x=(0, 1), y=(0, 1), z=(-1, 0),
              topology=(O.Periodic,) * 3 if grid == "periodic" else (O.Periodic, O.Periodic, O.Bounded))
    N2 = 3.0
    m0, m1 = _stratified_pair(kw, ADV[adv], N2)
    i, j, k = m0._box()
    w = m1.fields["w"]
    d = m1.Gn["b"][i, j, k] - m0.Gn["b"][i, j, k]
    want = -N2 * (w[i, j, k] + w[i, j, k + 1]) / 2
    assert np.max(np.abs(d - want)) <= 1e-10 * N2 * np.max(np.abs(w.interior))
    for n in "uvw":                                        # a tracer background enters no velocity tendency
        assert np.array_equal(m1.Gn[n].parent, m0.Gn[n].parent)


def test_linear_stratification_known_answer_oracle_stretched_weno():
    """the same on a stretched Bounded z with WENO5(grid): exact wherever the reconstruction keeps its full stencil.  Within two
    cells of a wall the reference falls back to lower-order reconstructions, which do not reproduce a linear profile between
    unevenly spaced centres, so those levels are excluded"""
    kw = dict(size=(8, 6, 12), x=(0, 1), y=(0, 1), z=_zf(12), topology=(O.Periodic, O.Periodic, O.Bounded))
    N2 = 3.0
    m0, m1 = _stratified_pair(kw, ADV["WENO5"], N2)
    i, j, _ = m0._box()
    k = O.R(3, 12 - 3)
    w = m1.fields["w"]
    d = m1.Gn["b"][i, j, k] - m0.Gn["b"][i, j, k]
    want = -N2 * (w[i, j, k] + w[i, j, k + 1]) / 2
    assert np.max(np.abs(d - want)) <= 1e-10 * N2 * np.max(np.abs(w.interior))


def _linearity(topo, adv, bg, total, buoyancy, steps=5, dt=1e-2):
    """model A steps the total fields, model B the perturbations about the backgrounds `bg`; returns the largest difference of
    A - background and B over every step, relative to the perturbation scale"""
    g = O.RectilinearGrid(np.float64, size=(8, 6, 10), x=(0, 1), y=(0, 1), z=(-1, 0), topology=topo)
    kw = dict(advection=adv, tracers=("b",), buoyancy=O.BuoyancyTracer() if buoyancy else None, timestepper="RungeKutta3")
    mA = BackgroundNonhydrostaticModel(g, **kw)
    mB = BackgroundNonhydrostaticModel(g, background_fields=bg, **kw)
    rng = np.random.default_rng(5)
    st = {n: 0.1 * rng.uniform(-1, 1, mB.fields[n].size()) for n in "uvwb"}
    if topo[2] == O.Bounded:
        st["w"][:, :, [0, -1]] = 0
    mB.set(**st)
    pert = {n: mB.fields[n].interior.copy() for n in "uvwb"}
    nodes = {n: mA.grid.nodes(mA.fields[n].loc) for n in "uvwb"}
    offs = {n: (total[n](*nodes[n], 0.0) + np.zeros(pert[n].shape)) if n in total else 0 for n in "uvwb"}
    mA.set(enforce_incompressibility=False, **{n: pert[n] + offs[n] for n in "uvwb"})
    worst = 0.0
    for _ in range(steps):
        mA.time_step(dt)
        mB.time_step(dt)
        for n in "uvwb":
            worst = max(worst, np.max(np.abs(mA.fields[n].interior - offs[n] - mB.fields[n].interior)) / 0.1)
    return worst


def test_linearity_known_answer_oracle_stratified_c2():
    """b = N² z + b', u = U₀ + u' against backgrounds B = N² z, U = U₀ with perturbations b', u' (CenteredSecondOrder, Bounded
    z, BuoyancyTracer): the centred flux is bilinear, and N² z changes pHY' by a function of z alone, so the two agree for 5
    RK3 steps to rounding"""
    N2, U0 = 2.0, 0.7
    bg = {"b": lambda x, y, z, t: N2 * z, "u": lambda x, y, z, t: U0 + 0 * x}
    assert _linearity((O.Periodic, O.Periodic, O.Bounded), O.CenteredSecondOrder(), bg, bg, True) <= 1e-12


@pytest.mark.parametrize("adv", ["CenteredSecondOrder", "CenteredFourthOrder"])
def test_linearity_known_answer_oracle_periodic(adv):
    """the same for both centred schemes on a triply periodic grid with a periodic tracer background and a uniform U₀ (no
    buoyancy: a background enters no buoyancy term, so only a passive b is linear in it).  On a Bounded z the fourth-order
    stencil reads the halos next to the walls, where the total field's no-flux fill and the background's function values
    differ, so that case is not linear"""
    U0 = 0.7          # along x, across which B does not vary: the term div(U_bg, B) the reference drops is exactly zero
    bg = {"b": lambda x, y, z, t: 0.5 * np.sin(2 * np.pi * y) * np.cos(2 * np.pi * z), "u": lambda x, y, z, t: U0 + 0 * x}
    assert _linearity((O.Periodic,) * 3, getattr(O, adv)(), bg, bg, False) <= 1e-12
