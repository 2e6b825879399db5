"""Background fields on the oracle's NonhydrostaticModel (test infrastructure).

The reference's `background_fields` (src/Models/NonhydrostaticModels/background_fields.jl) enter every tendency as two terms
right after the advection of the field by the model velocities (nonhydrostatic_tendency_kernel_functions.jl):

    Gψ = - div_𝐯ψ(advection, U, ψ) - div_𝐯ψ(advection, U_bg, ψ) - div_𝐯ψ(advection, U, ψ_bg) - ...      (velocities)
    Gc = - div_Uc(advection, U, c)  - div_Uc(advection, U_bg, c)  - div_Uc(advection, U, c_bg)  - ...      (tracers)

A missing background is a ZeroField, whose terms are exactly zero.  A background is a FunctionField: its value at every parent
index, halos included, is the function at that node, and its halos are never filled.  `BackgroundNonhydrostaticModel` holds each
background as a parent-shaped array and evaluates the two terms with the oracle's own div_Uu / div_Uc, in place of the oracle's
`- zero - zero` slots.  They are added after the oracle's other terms (and after the boundary fluxes and the Relaxation forcing
it adds inside its tendency step), which differs from the reference's order by rounding only.  Without backgrounds the model is
the oracle's.
"""
import numpy as np

import oracle as O
from oracle.advection import div_Uu, div_Uc
from relaxation_reference import ForcedNonhydrostaticModel


def parent_nodes(grid, loc):
    """x, y, z at every parent index of a field at `loc` on an oracle grid (halos, the extra Face point of a Bounded dimension,
    the Flat coordinate), broadcast-shaped, in double"""
    out = []
    for d in range(3):
        src = grid.nodesF[d] if loc[d] == O.Face else grid.nodesC[d]
        n = grid.parent_size(loc)[d]
        lo = 1 - grid.H[d]
        a = np.asarray(src.slice(lo, lo + n - 1), dtype=np.float64)
        shape = [1, 1, 1]
        shape[d] = n
        out.append(a.reshape(shape))
    return out


def table(grid, loc, func, parameters=None, time=0.0):
    """FunctionField(loc, func, grid; clock, parameters) as a parent array: func(x, y, z, t[, parameters]) at every node,
    evaluated in double, rounded once to the grid's float type"""
    x, y, z = parent_nodes(grid, loc)
    v = func(x, y, z, np.float64(time)) if parameters is None else func(x, y, z, np.float64(time), parameters)
    return np.asfortranarray(np.broadcast_to(np.asarray(v, dtype=np.float64), grid.parent_size(loc)).astype(grid.FT))


class BackgroundNonhydrostaticModel(ForcedNonhydrostaticModel):
    """oracle NonhydrostaticModel(grid; background_fields = {name: parent array or func(x, y, z, t)}, forcing = ..., kwargs...)"""

    def __init__(self, grid, background_fields=None, **kw):
        super().__init__(grid, **kw)
        self.bg = {}
        for n, v in (background_fields or {}).items():
            if n not in self.names:
                raise ValueError(f"{n} is not a prognostic field")
            self.set_background(n, v)

    def set_background(self, name, value):
        loc = self.fields[name].loc
        f = self.bg.get(name) or O.Field(self.grid, loc)
        f.parent[...] = table(self.grid, loc, value) if callable(value) else np.asarray(value, dtype=self.grid.FT)
        self.bg[name] = f

    def background_terms(self):
        """- div(U_bg, ψ) - div(U, ψ_bg) of every field with a non-zero term, over the interior cells"""
        g = self.grid
        i, j, k = self._box()
        adv = self.advection
        U = tuple(self.velocities[n] for n in "uvw")
        has_U = any(n in self.bg for n in "uvw")
        Ubg = tuple(self.bg[n] if n in self.bg else O.Field(g, self.velocities[n].loc) for n in "uvw")     # ZeroField
        out = {}
        for q, n in enumerate(self.names):
            if not has_U and n not in self.bg:
                continue
            psi = self.fields[n]
            G = g.FT(0)
            if n in "uvw":
                if has_U:
                    G = G - div_Uu(q, i, j, k, g, adv, Ubg, psi)
                if n in self.bg:
                    G = G - div_Uu(q, i, j, k, g, adv, U, self.bg[n])
            else:
                if has_U:
                    G = G - div_Uc(i, j, k, g, adv, Ubg, psi)
                if n in self.bg:
                    G = G - div_Uc(i, j, k, g, adv, U, self.bg[n])
            out[n] = G
        return out

    def calculate_tendencies(self):
        B = self.background_terms()
        super().calculate_tendencies()
        i, j, k = self._box()
        for n, t in B.items():
            self.Gn[n][i, j, k] = self.Gn[n][i, j, k] + t
