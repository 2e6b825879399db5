"""Array-valued Flux / Value / Gradient boundary conditions without a device: on the oracle, an array filled with the constant
reproduces the constant condition bit for bit (halo fills and flux terms, every side of a (Bounded, Bounded, Bounded) grid, regular
and stretched z); the flux-budget known answer of one forward-Euler step; the mirror's checks of the arrays (boundary_values,
set_boundary_condition_values) and its rejections."""
import types

import numpy as np
import pytest

import oracle as O
from oracle.fields import apply_flux_bcs
from bc_array_reference import SIDES, array_bc, normal_dim, tangential_shape


def _zf(n, p=1.5):
    return -np.linspace(1, 0, n + 1) ** p


def _bbb(FT, stretched):
    kw = dict(size=(5, 4, 6), topology=(O.Bounded,) * 3, x=(0, 1.3), y=(-1, 1))
    kw["z"] = _zf(6) if stretched else (-0.7, 0)
    return O.RectilinearGrid(FT, halo=(2, 2, 2), **kw)


LOCS = [("c", "c", "c"), ("f", "c", "c"), ("c", "f", "c"), ("c", "c", "f")]
CONST = {"Flux": 3.25e-2, "Value": -0.75, "Gradient": 1.5}


def _allowed(loc, side):
    return loc[normal_dim(side)] == "c"          # the side normal to a Face location is the wall


@pytest.mark.parametrize("FT", [np.float64, np.float32])
@pytest.mark.parametrize("stretched", [False, True])
@pytest.mark.parametrize("kind", ["Flux", "Value", "Gradient"])
def test_constant_filled_array_matches_constant_oracle(FT, stretched, kind):
    g = _bbb(FT, stretched)
    rng = np.random.default_rng(7)
    v = CONST[kind]
    for loc in LOCS:
        sides = [s for s in SIDES if _allowed(loc, s)]
        bc_c = O.FieldBoundaryConditions(g, loc, **{s: O.BoundaryCondition(kind, v) for s in sides})
        bc_a = O.FieldBoundaryConditions(g, loc, **{s: array_bc(kind, np.full(tangential_shape(g, s), v), s) for s in sides})
        fc, fa = O.Field(g, loc, bc_c), O.Field(g, loc, bc_a)
        p = rng.uniform(-1, 1, fc.parent.shape).astype(FT)
        fc.parent[...] = p
        fa.parent[...] = p
        O.fill_halo_regions(fc)
        O.fill_halo_regions(fa)
        assert fa.parent.dtype == fc.parent.dtype and np.array_equal(fa.parent, fc.parent), loc
        Gc, Ga = O.Field(g, loc), O.Field(g, loc)
        G0 = rng.uniform(-1, 1, Gc.parent.shape).astype(FT)
        Gc.parent[...] = G0
        Ga.parent[...] = G0
        apply_flux_bcs(Gc, fc)
        apply_flux_bcs(Ga, fa)
        assert np.array_equal(Ga.parent, Gc.parent), loc
        if kind == "Flux":
            assert not np.array_equal(Gc.parent, G0)


def test_array_varies_per_boundary_point_on_the_oracle():
    """a non-uniform array: each boundary point takes its own value (Q[j, k], Q[i, k], Q[i, j]), and the Value fill is the
    constant fill with that point's value"""
    g = _bbb(np.float64, True)
    rng = np.random.default_rng(8)
    for side in SIDES:
        d = normal_dim(side)
        Q = rng.uniform(-1, 1, tangential_shape(g, side))
        f = O.Field(g, ("c", "c", "c"), O.FieldBoundaryConditions(g, ("c", "c", "c"), **{side: array_bc("Value", Q, side)}))
        f.parent[...] = rng.uniform(-1, 1, f.parent.shape)
        O.fill_halo_regions(f)
        a, b = [e for e in range(3) if e != d]
        for ia, ib in ((1, 1), (g.N[a], 2), (2, g.N[b])):
            f1 = O.Field(g, ("c", "c", "c"), O.FieldBoundaryConditions(g, ("c", "c", "c"),
                                                                       **{side: O.BoundaryCondition("Value", Q[ia - 1, ib - 1])}))
            f1.parent[...] = f.parent
            O.fill_halo_regions(f1)
            idx = [None] * 3
            idx[d] = 0 if side in ("west", "south", "bottom") else g.N[d] + 1
            idx[a], idx[b] = ia, ib
            assert f[tuple(idx)] == f1[tuple(idx)], (side, ia, ib)


@pytest.mark.parametrize("side,sign", [("top", -1), ("bottom", 1)])
def test_flux_budget_known_answer_oracle(side, sign):
    """no advection, no closure, a tracer with a Flux array on one side: one forward-Euler AB2 step changes Σ c V by
    ∓ Δt Σ Q A over that side (the array form of test/test_boundary_conditions_integration.jl:26-50)"""
    g = O.RectilinearGrid(np.float64, size=(6, 5, 8), x=(0, 2), y=(0, 1), z=_zf(8), topology=(O.Periodic, O.Periodic, O.Bounded))
    rng = np.random.default_rng(9)
    Q = rng.uniform(-1, 1, tangential_shape(g, side))
    m = O.NonhydrostaticModel(g, advection=None, tracers=("c",), boundary_conditions={"c": {side: array_bc("Flux", Q, side)}})
    m.set(c=rng.uniform(-1, 1, m.fields["c"].size()))
    i, j, k = m._box()
    V = np.broadcast_to(g.V(i, j, k, "c", "c", "c"), (g.Nx, g.Ny, g.Nz))
    before = np.sum(m.fields["c"][i, j, k] * V)
    dt = 0.1
    m.time_step(dt, euler=True)
    after = np.sum(m.fields["c"][i, j, k] * V)
    kk = O.R(g.Nz + 1) if side == "top" else O.R(1)
    A = np.broadcast_to(g.Az(i, j, kk, "c", "c", "f"), (g.Nx, g.Ny, 1))[:, :, 0]
    want = sign * dt * np.sum(Q * A)
    assert abs((after - before) - want) <= 1e-13 * max(abs(before), abs(want))


# ---- the mirror: pure checks, no library call ---------------------------------------------------------------------------------
def _mirror():
    import ocean_b200.model as M
    return M


def test_mirror_accepts_the_tangential_shapes():
    M = _mirror()
    g = O.RectilinearGrid(np.float32, size=(6, 5, 4), extent=(1, 1, 1), topology=(O.Bounded,) * 3)
    C, F = M.Center, M.Face
    for side, shape in (("west", (5, 4)), ("east", (5, 4)), ("south", (6, 4)), ("north", (6, 4)), ("bottom", (6, 5)),
                        ("top", (6, 5))):
        for kind in ("Flux", "Value", "Gradient"):
            t = M.boundary_values(g, (C, C, C), side, M.BoundaryCondition(kind, np.arange(np.prod(shape), dtype=np.float64)
                                                                          .reshape(shape)))
            assert t.shape == shape and t.dtype == np.float32 and t.flags.f_contiguous
            assert np.array_equal(t, np.arange(np.prod(shape)).reshape(shape).astype(np.float32))
    # tangential sides of Face fields, integer arrays
    assert M.boundary_values(g, (F, C, C), "top", M.FluxBoundaryCondition(np.ones((6, 5), dtype=np.int64))).dtype == np.float32
    assert M.boundary_values(g, (C, C, F), "west", M.ValueBoundaryCondition(np.ones((5, 4)))).shape == (5, 4)
    # a Flat tangential dimension counts as 1
    g2 = O.RectilinearGrid(np.float64, size=(16, 12), extent=(1, 1), topology=(O.Periodic, O.Bounded, O.Flat))
    assert M.boundary_values(g2, (C, C, C), "south", M.FluxBoundaryCondition(np.zeros((16, 1)))).shape == (16, 1)
    g3 = O.RectilinearGrid(np.float64, size=(16, 12), extent=(1, 1), topology=(O.Flat, O.Bounded, O.Bounded))
    assert M.boundary_values(g3, (C, C, C), "top", M.GradientBoundaryCondition(np.zeros((1, 16)))).shape == (1, 16)


def test_mirror_rejects_unsupported_arrays():
    M = _mirror()
    C, F = M.Center, M.Face
    g = O.RectilinearGrid(np.float64, size=(6, 5, 4), extent=(1, 1, 1), topology=(O.Periodic, O.Bounded, O.Bounded))
    ok = np.zeros((6, 5))
    cases = [
        (g, (C, C, C), "top", M.FluxBoundaryCondition(np.zeros((5, 6)))),           # transposed
        (g, (C, C, C), "top", M.FluxBoundaryCondition(np.zeros((6, 4)))),          # too small
        (g, (C, C, C), "west", M.FluxBoundaryCondition(np.zeros((5, 4)))),          # Periodic dimension
        (g, (C, C, F), "top", M.FluxBoundaryCondition(ok)),                          # normal to w: the wall
        (g, (C, F, C), "south", M.ValueBoundaryCondition(np.zeros((6, 4)))),         # normal to v
        (g, (C, C, C), "top", M.BoundaryCondition("Open", ok)),
        (g, (C, C, C), "top", M.BoundaryCondition(None, ok)),
        (g, (C, C, C), "top", M.FluxBoundaryCondition(0.5)),                         # not an array
    ]
    for grid, loc, side, bc in cases:
        with pytest.raises(ValueError):
            M.boundary_values(grid, loc, side, bc)
    slab = types.SimpleNamespace(topology=(O.Periodic, "FullyConnected", O.Bounded), N=(6, 5, 4), FT=np.float64)
    with pytest.raises(ValueError, match="slab-decomposed"):
        M.boundary_values(slab, (C, C, C), "top", M.FluxBoundaryCondition(ok))
    g2 = O.RectilinearGrid(np.float64, size=(16, 12), extent=(1, 1), topology=(O.Periodic, O.Bounded, O.Flat))
    with pytest.raises(ValueError):
        M.boundary_values(g2, (C, C, C), "south", M.FluxBoundaryCondition(np.zeros((16, 2))))       # Flat counts as 1
    for bad in (np.zeros(6), np.zeros((6, 5, 1)), np.zeros((6, 5), dtype=bool), np.zeros((6, 5), dtype=complex),
                np.array([["a"] * 5] * 6)):
        with pytest.raises(ValueError):
            M.FluxBoundaryCondition(bad)
    # the time-varying setter checks the same things before touching the library (no handle here)
    fake = types.SimpleNamespace(grid=g, loc=(C, C, C), handle=None,
                                 boundary_conditions={"top": M.FluxBoundaryCondition(ok), "bottom": M.BoundaryCondition("Open"),
                                                      "west": M.BoundaryCondition("Periodic")})
    for side, values in (("top", np.zeros((5, 6))), ("top", [[0.0] * 5] * 6), ("bottom", ok), ("west", np.zeros((5, 4))),
                         ("up", ok)):
        with pytest.raises(ValueError):
            M.set_boundary_condition_values(fake, side, values)


def test_mirror_constant_conditions_unchanged():
    """a number, None and a 0-d array still cross as the constant `value` of ob200_bc"""
    M = _mirror()
    g = types.SimpleNamespace(topology=("Periodic", "Bounded", "Bounded"), N=(4, 4, 4), FT=np.float64)
    arr = M._bc_array(g, ("Center",) * 3, {"top": M.FluxBoundaryCondition(1e-4), "bottom": M.GradientBoundaryCondition(np.float64(2.0)),
                                           "north": M.ValueBoundaryCondition(np.array(0.5))})
    got = [(arr[s].kind, arr[s].value) for s in range(6)]
    L = M.L
    assert got == [(L.BC_PERIODIC, 0.0), (L.BC_PERIODIC, 0.0), (L.BC_FLUX, 0.0), (L.BC_VALUE, 0.5),
                   (L.BC_GRADIENT, 2.0), (L.BC_FLUX, 1e-4)]
    arr = M._bc_array(g, ("Center",) * 3, {"top": M.FluxBoundaryCondition(np.ones((4, 4)))})
    assert (arr[5].kind, arr[5].value) == (L.BC_FLUX, 0.0)
