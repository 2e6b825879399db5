"""Relaxation forcing on the oracle's NonhydrostaticModel (test infrastructure).

The reference's Relaxation(; rate, mask, target), GaussianMask{D} and LinearTarget{D} (src/Forcings/relaxation.jl) written
out pointwise, evaluated at the forced field's own nodes (xnode(LX, i, grid) etc.: `regularize_forcing` wraps the Relaxation in
a ContinuousForcing of the field itself, and interpolating a field to its own location is the identity):

    rate * mask(x, y, z) * (target(x, y, z, t) - field)

with the parameters and the float-type nodes in their promoted type.  `ForcedNonhydrostaticModel` adds this term to each
forced tendency of the oracle model, in place of the oracle's trailing `+ zero`.  The oracle adds the boundary-flux
contributions inside its tendency step, so here the forcing follows them: at cells with a non-trivial Flux boundary
condition the sum differs from the reference's order by rounding only.  Without forcing the model is the oracle's.
"""
import numpy as np

import oracle as O

DIMS = {"x": 0, "y": 1, "z": 2}


def _p(v):
    """a Python float is a Float64 parameter (it promotes Float32 nodes); anything else as given"""
    return np.float64(v) if isinstance(v, float) else v


def gaussian_mask(mask, x, y, z):
    """(g::GaussianMask{D})(x, y, z) = exp(-(ξ - g.center)^2 / (2 * g.width^2)), ξ the coordinate along D"""
    xi = (x, y, z)[DIMS[mask.dim]]
    return np.exp(-(xi - _p(mask.center)) ** 2 / (2 * _p(mask.width) ** 2))


def linear_target(target, x, y, z):
    """(p::LinearTarget{D})(x, y, z, t) = p.intercept + p.gradient * ξ"""
    xi = (x, y, z)[DIMS[target.dim]]
    return _p(target.intercept) + _p(target.gradient) * xi


def relaxation(r, x, y, z, field):
    """(f::Relaxation)(x, y, z, t, field) = f.rate * f.mask(x, y, z) * (f.target(x, y, z, t) - field); onefunction /
    zerofunction for a missing mask / target, and the Number-target method for a number"""
    mask = 1 if r.mask is None else gaussian_mask(r.mask, x, y, z)
    if r.target is None:
        target = 0
    elif isinstance(r.target, (int, float, np.integer, np.floating)):
        target = _p(r.target)
    else:
        target = linear_target(r.target, x, y, z)
    return _p(r.rate) * mask * (target - field)


class ForcedNonhydrostaticModel(O.NonhydrostaticModel):
    """oracle NonhydrostaticModel(grid; forcing = {name: Relaxation}, kwargs...)"""

    def __init__(self, grid, forcing=None, **kw):
        self.forcing = dict(forcing or {})
        super().__init__(grid, **kw)
        for n in self.forcing:
            if n not in self.names:
                raise ValueError(f"{n} is not a prognostic field")

    def forcing_term(self, name):
        """the Relaxation of field `name` over its interior cells 1..N"""
        f = self.fields[name]
        g = self.grid
        x, y, z = g.nodes(f.loc)
        i, j, k = self._box()
        x, y, z = x[:g.Nx], y[:, :g.Ny], z[:, :, :g.Nz]       # a Face field on a Bounded dimension has one node more
        return relaxation(self.forcing[name], x, y, z, f[i, j, k])

    def calculate_tendencies(self):
        F = {n: self.forcing_term(n) for n in self.forcing}
        super().calculate_tendencies()
        i, j, k = self._box()
        for n, t in F.items():
            self.Gn[n][i, j, k] = self.Gn[n][i, j, k] + t
