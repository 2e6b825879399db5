"""Array-valued boundary conditions on the oracle (test infrastructure).

The reference indexes an array condition by the grid's interior indices along the side's two tangential dimensions,
getbc(bc::BC{<:Any,<:AbstractArray}, i, j, grid, args...) = bc.condition[i, j] (src/BoundaryConditions/boundary_condition.jl):
Q[j, k] on x sides, Q[i, k] on y sides, Q[i, j] on z sides, a Flat dimension counting as 1.  The oracle's halo fills and flux
terms (oracle/fields.py) work on whole boundary planes of the grid's interior extent with the condition as `FT(condition)`; given
the (N_a, N_b) array with a unit axis inserted along the side's normal dimension, that expression is the array in the grid's
float type and broadcasts over the plane point by point.  So the oracle itself is unchanged and its constant path untouched.
"""
import numpy as np

import oracle as O

SIDES = ("west", "east", "south", "north", "bottom", "top")


def normal_dim(side):
    return SIDES.index(side) // 2


def tangential_shape(grid, side):
    """(N_a, N_b) of the side's tangential dimensions in x, y, z order, Flat = 1"""
    d = normal_dim(side)
    return tuple(1 if grid.topology[e] == O.Flat else grid.N[e] for e in range(3) if e != d)


def oracle_condition(Q, side):
    """the (N_a, N_b) array as the oracle's condition: a unit axis along the side's normal dimension"""
    Q = np.asarray(Q)
    assert Q.ndim == 2
    return np.expand_dims(Q, normal_dim(side))


def array_bc(kind, Q, side):
    """FluxBoundaryCondition(Q) / ValueBoundaryCondition(Q) / GradientBoundaryCondition(Q) on the oracle"""
    return O.BoundaryCondition(kind, oracle_condition(Q, side))


def set_values(field, side, Q):
    """bc.condition .= Q on an oracle field, as a callback does between steps"""
    bc = getattr(field.bcs, side)
    bc.condition = oracle_condition(Q, side)
