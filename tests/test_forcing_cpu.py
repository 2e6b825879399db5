"""Relaxation forcing (src/Forcings/relaxation.jl) without a device: known answers of one time step on the oracle with the
forcing as the only tendency, the host table builder of the mirror against the pointwise forcing evaluation, the mirror's
rejections and the C layout of the forcing descriptor against its ctypes mirror."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import oracle as O
from relaxation_reference import ForcedNonhydrostaticModel, relaxation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _zf(n, p=1.5):
    return -np.linspace(1, 0, n + 1) ** p


def _rk3_poly(z):
    return 1 + z + z ** 2 / 2 + z ** 3 / 6


def _tracer_model(ts):
    from ocean_b200.model import Relaxation, GaussianMask, LinearTarget
    g = O.RectilinearGrid(np.float64, size=(4, 3, 16), x=(0, 1), y=(0, 1), z=_zf(16), topology=(O.Periodic, O.Periodic, O.Bounded))
    r = Relaxation(rate=2.0, mask=GaussianMask("z", center=-0.7, width=0.2), target=LinearTarget("z", intercept=1.5, gradient=0.8))
    m = ForcedNonhydrostaticModel(g, forcing={"c": r}, advection=None, tracers=("c",), timestepper=ts)
    rng = np.random.default_rng(3)
    m.set(c=rng.uniform(-1, 1, m.fields["c"].size()))
    z = g.nodes(("c", "c", "c"))[2]
    lam = -(2.0 * np.exp(-(z + 0.7) ** 2 / (2 * 0.2 ** 2)))
    return m, r, 1.5 + 0.8 * z, lam


def _box(m, name):
    g = m.grid
    return m.fields[name][O.R(1, g.Nx), O.R(1, g.Ny), O.R(1, g.Nz)].copy()


def test_rk3_relaxation_known_answer_oracle():
    """one RK3 step of dc/dt = λ (c - T): c₁ - T = (1 + z + z²/2 + z³/6)(c₀ - T), z = λ Δt (exact for the Le-Moin coefficients)"""
    m, _, T, lam = _tracer_model("RungeKutta3")
    dt = 0.3
    c0 = _box(m, "c")
    m.time_step(dt)
    want = _rk3_poly(lam * dt) * (c0 - T)
    assert np.max(np.abs((_box(m, "c") - T) - want)) <= 1e-13 * np.max(np.abs(c0 - T))


def test_ab2_relaxation_known_answer_oracle():
    """AB2: a forward-Euler first step (1 + z), then e_{n+1} = e_n + z ((3/2 + χ) e_n - (1/2 + χ) e_{n-1}), χ = 0.1"""
    m, _, T, lam = _tracer_model("QuasiAdamsBashforth2")
    dt = 0.2
    z = lam * dt
    e = [_box(m, "c") - T]
    e.append((1 + z) * e[0])
    for _ in range(3):
        e.append(e[-1] + z * (1.6 * e[-1] - 0.6 * e[-2]))
    for n in range(1, 5):
        m.time_step(dt)
        got = _box(m, "c") - T
        assert np.max(np.abs(got - e[n])) <= 1e-13 * np.max(np.abs(e[0])), n


def test_velocity_relaxation_known_answer_oracle():
    """u(z) relaxed toward a linear profile under a bottom sponge in a (Periodic, Periodic, Bounded) box: u stays a function of z,
    the flow stays divergence free and one RK3 step follows the same polynomial"""
    from ocean_b200.model import Relaxation, GaussianMask, LinearTarget
    g = O.RectilinearGrid(np.float64, size=(4, 4, 12), x=(0, 1), y=(0, 1), z=_zf(12), topology=(O.Periodic, O.Periodic, O.Bounded))
    r = Relaxation(rate=3.0, mask=GaussianMask("z", center=-1.0, width=0.3), target=LinearTarget("z", intercept=0.2, gradient=-0.5))
    m = ForcedNonhydrostaticModel(g, forcing={"u": r}, advection=None, timestepper="RungeKutta3")
    z = g.nodes(("f", "c", "c"))[2]
    u0 = np.broadcast_to(np.sin(3 * z), m.fields["u"].size())
    m.set(u=u0)
    T = 0.2 - 0.5 * z
    lam = -(3.0 * np.exp(-(z + 1.0) ** 2 / (2 * 0.3 ** 2)))
    dt = 0.25
    m.time_step(dt)
    u1 = _box(m, "u")
    want = T + _rk3_poly(lam * dt) * (u0 - T)
    assert np.max(np.abs(u1 - want)) <= 1e-13 * np.max(np.abs(u0 - T))
    assert m.max_divergence() < 1e-14
    assert np.max(np.abs(_box(m, "v"))) < 1e-15 and np.max(np.abs(_box(m, "w"))) < 1e-15


@pytest.mark.parametrize("FT", [np.float64, np.float32])
@pytest.mark.parametrize("stretched", [False, True])
def test_host_relaxation_tables_match_oracle(FT, stretched):
    """the mirror's table builder (relaxation_tables) equals the pointwise forcing evaluation bit for bit, at all four field
    locations, for masks and targets along each dimension"""
    from ocean_b200.model import Relaxation, GaussianMask, LinearTarget, relaxation_tables
    kw = dict(size=(6, 5, 7), topology=(O.Bounded, O.Periodic, O.Bounded), x=(-1, 2), y=(0, 3))
    kw["z"] = _zf(7) if stretched else (-1, 0)
    g = O.RectilinearGrid(FT, **kw)
    cases = [Relaxation(1 / 7, mask=GaussianMask(d, center=0.3, width=0.45), target=LinearTarget(e, intercept=0.1, gradient=1 / 3))
             for d in "xyz" for e in "xyz"]
    cases += [Relaxation(0.25), Relaxation(2, target=0.75), Relaxation(1e-3, mask=GaussianMask("z", -0.5, 0.1))]
    rng = np.random.default_rng(5)
    for loc in (("c", "c", "c"), ("f", "c", "c"), ("c", "f", "c"), ("c", "c", "f")):
        x, y, z = g.nodes(loc)
        psi = rng.uniform(-1, 1, (x.shape[0], y.shape[1], z.shape[2])).astype(FT)
        for r in cases:
            md, M, td, T = relaxation_tables(r, loc, g)
            want = relaxation(r, x, y, z, psi)
            Mb = M if md < 0 else np.asarray(M).reshape([len(M) if d == md else 1 for d in range(3)])
            Tb = T if td < 0 else np.asarray(T).reshape([len(T) if d == td else 1 for d in range(3)])
            got = Mb * (Tb - psi)
            assert got.dtype == want.dtype and np.array_equal(got, want), (loc, md, td)
            for d, t in ((md, M), (td, T)):
                if d >= 0:
                    n = g.N[d] + (1 if loc[d] == "f" and g.topology[d] == O.Bounded else 0)
                    assert len(t) == n


def test_mirror_rejects_unsupported_forcings():
    from ocean_b200.model import Relaxation, GaussianMask, LinearTarget, relaxation_tables
    with pytest.raises(ValueError):
        Relaxation(rate="fast")
    with pytest.raises(ValueError):
        Relaxation(rate=lambda x: x)
    with pytest.raises(ValueError):
        Relaxation(rate=1.0, mask=lambda x, y, z: 1.0)
    with pytest.raises(ValueError):
        Relaxation(rate=1.0, target=lambda x, y, z, t: 0.0)
    with pytest.raises(ValueError):
        GaussianMask("q", 0.0, 1.0)
    with pytest.raises(ValueError):
        LinearTarget("x", "a", 1.0)
    g = O.RectilinearGrid(np.float64, size=(8, 6), extent=(1, 1), topology=(O.Periodic, O.Periodic, O.Flat))
    with pytest.raises(ValueError, match="Flat"):
        relaxation_tables(Relaxation(1.0, mask=GaussianMask("z", 0.0, 1.0)), ("c", "c", "c"), g)
    with pytest.raises(ValueError, match="Flat"):
        relaxation_tables(Relaxation(1.0, target=LinearTarget("z", 0.0, 1.0)), ("c", "c", "c"), g)


def test_forcing_descriptor_layout_matches_ctypes(tmp_path):
    """sizeof / offsetof of ob200_model_desc, its forcing array and ob200_forcing from the C header against _lib's structures"""
    import ocean_b200._lib as L
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ocean_b200.h"\nint main(void) {\n'
                   'printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(ob200_model_desc), offsetof(ob200_model_desc, forcing),'
                   ' offsetof(ob200_model_desc, closure_vertically_implicit), sizeof(ob200_forcing),'
                   ' offsetof(ob200_forcing, mask_dim), offsetof(ob200_forcing, rate), offsetof(ob200_forcing, mask),'
                   ' offsetof(ob200_forcing, target_dim), offsetof(ob200_forcing, target_value), offsetof(ob200_forcing, target),'
                   ' sizeof(((ob200_model_desc*)0)->forcing));\nreturn 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    F, D = L.Forcing, L.ModelDesc
    want = [ctypes.sizeof(D), D.forcing.offset, D.closure_vertically_implicit.offset, ctypes.sizeof(F), F.mask_dim.offset,
            F.rate.offset, F.mask.offset, F.target_dim.offset, F.target_value.offset, F.target.offset,
            ctypes.sizeof(F) * (3 + L.MAX_TRACERS)]
    assert got == want
