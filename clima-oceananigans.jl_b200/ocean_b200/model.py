"""Host-side mirror of the reference's operator interface for the NonhydrostaticModel path on the
`B200()` architecture: Field, fill_halo_regions!, FFTBasedPoissonSolver /
FourierTridiagonalPoissonSolver / BatchedTridiagonalSolver + solve!, NonhydrostaticModel, set!,
update_state!, time_step!.  Names, argument meaning and error behaviour follow the reference
(files cited per class); all arithmetic happens in libocean_b200.so."""
import ctypes as C

import numpy as np

from . import _lib as L
from ._lib import lib, check, B200Error
from .grids import RectilinearGrid, Periodic, Bounded, Flat, Center, Face

_LOC = {Center: L.CENTER, Face: L.FACE}
_BCK = {"Periodic": L.BC_PERIODIC, "Flux": L.BC_FLUX, "Value": L.BC_VALUE, "Gradient": L.BC_GRADIENT,
        "Open": L.BC_OPEN, None: L.BC_NONE}


# ---- boundary conditions (src/BoundaryConditions/boundary_condition.jl) ----------------------
class BoundaryCondition:
    """`condition` is None, a number or a 2-D numpy array (getbc(bc::BC{<:Any,<:AbstractArray}, i, j, grid) = bc.condition[i, j]):
    indexed by the grid's interior indices along the side's two tangential dimensions, Flat counting as 1."""

    def __init__(self, kind, condition=None):
        if callable(condition):
            raise ValueError("function-valued boundary conditions cannot cross the C ABI of the B200 "
                             "architecture (SURVEY.md 8(b)); use constants or 2-D arrays")
        if isinstance(condition, np.ndarray) and condition.ndim != 0 and not _is_real_matrix(condition):
            raise ValueError(f"an array boundary condition must be a 2-D real numeric array, got a {condition.ndim}-D "
                             f"{condition.dtype} array")
        self.kind, self.condition = kind, condition

    @property
    def is_array(self):
        return isinstance(self.condition, np.ndarray) and self.condition.ndim != 0


def _is_real_matrix(a):
    return (isinstance(a, np.ndarray) and a.ndim == 2 and a.dtype != bool and
            (np.issubdtype(a.dtype, np.integer) or np.issubdtype(a.dtype, np.floating)))


def FluxBoundaryCondition(v):
    return BoundaryCondition("Flux", v)


def ValueBoundaryCondition(v):
    return BoundaryCondition("Value", v)


def GradientBoundaryCondition(v):
    return BoundaryCondition("Gradient", v)


_SIDES = ("west", "east", "south", "north", "bottom", "top")


def _default_bc(topo, loc, auxiliary=False):
    """default_prognostic_bc / default_auxiliary_bc (field_boundary_conditions.jl:13-34)."""
    if topo in (Periodic, "FullyConnected"):
        return BoundaryCondition("Periodic")
    if topo == Flat:
        return BoundaryCondition(None)
    if loc == Center:
        return BoundaryCondition("Flux", None)
    return BoundaryCondition(None) if auxiliary else BoundaryCondition("Open", None)


def _resolve_bcs(grid, loc, user=None, auxiliary=False):
    """{side: BoundaryCondition} with the defaults filled in"""
    user = user or {}
    return {name: user.get(name) or _default_bc(grid.topology[s // 2], loc[s // 2], auxiliary) for s, name in enumerate(_SIDES)}


def _bc_array(grid, loc, user=None, auxiliary=False):
    """the ob200_bc[6] of a field; an array condition crosses as its kind with value 0 and is pushed after creation"""
    arr = (L.BC * 6)()
    for s, (name, bc) in enumerate(_resolve_bcs(grid, loc, user, auxiliary).items()):
        arr[s].kind = _BCK[bc.kind]
        arr[s].value = 0.0 if (bc.condition is None or bc.is_array) else float(bc.condition)
    return arr


def boundary_values(grid, loc, side, bc):
    """The table of an array boundary condition `bc` on `side` of a field at `loc` (anything with .topology, .N and .FT): the
    array cast to the grid's float type, column-major, after checking it against the grid and the side.  No library call.
    The shape is (N_a, N_b) of the side's two tangential dimensions in x, y, z order, a Flat dimension counting as 1: the
    reference's BC kernels run over the grid's interior size, not the field's (fill_halo_regions.jl:163-170)."""
    if side not in _SIDES:
        raise ValueError(f"unknown side {side!r}; sides are {_SIDES}")
    s = _SIDES.index(side)
    d = s // 2
    if "FullyConnected" in tuple(grid.topology):
        raise ValueError("array boundary conditions are not supported on a slab-decomposed (FullyConnected) grid")
    if grid.topology[d] != Bounded:
        raise ValueError(f"array boundary condition on the {side} side of a {grid.topology[d]} dimension: only Bounded "
                         "dimensions have boundary conditions of that kind")
    if bc.kind not in ("Flux", "Value", "Gradient"):
        raise ValueError(f"array boundary conditions must be Flux, Value or Gradient conditions, not {bc.kind}")
    if loc[d] == Face:
        raise ValueError(f"the {side} side of a field located on the {'xyz'[d]}-faces is the impenetrable wall; it takes no "
                         "array boundary condition")
    q = bc.condition
    if not _is_real_matrix(q):
        raise ValueError("an array boundary condition must be a 2-D real numeric numpy array")
    shape = tuple(1 if grid.topology[e] == Flat else int(grid.N[e]) for e in range(3) if e != d)
    if q.shape != shape:
        raise ValueError(f"the array boundary condition on the {side} side has shape {q.shape}; the grid needs {shape} "
                         f"(interior size along {', '.join('xyz'[e] for e in range(3) if e != d)}, Flat = 1)")
    return np.asfortranarray(q, dtype=grid.FT)


def _array_tables(grid, loc, bcs):
    """{side index: table} of every array condition among the resolved `bcs`, checked before any library call"""
    return {_SIDES.index(n): boundary_values(grid, loc, n, bc) for n, bc in bcs.items() if bc is not None and bc.is_array}


def _push_boundary_values(handle, tables):
    for s, t in tables.items():
        check(lib.ob200_field_set_boundary_values(handle, s, t.ctypes.data_as(C.c_void_p)))


def set_boundary_condition_values(field, side, values):
    """Replace the values of the array boundary condition on `side` of `field` (a Field or a model field such as
    model.tracers["b"]), as `bc.condition .= values` in a callback does in the reference.  The copy is ordered after every step
    enqueued so far, so it takes effect from the next step on.  Raises ValueError before any library call if the side cannot
    take an array (see boundary_values) or the shape is wrong."""
    if side not in _SIDES:
        raise ValueError(f"unknown side {side!r}; sides are {_SIDES}")
    bc = field.boundary_conditions[side]
    if not _is_real_matrix(values):
        raise ValueError("boundary condition values must be a 2-D real numeric numpy array")
    t = boundary_values(field.grid, field.loc, side, BoundaryCondition(bc.kind, values))
    _push_boundary_values(field.handle, {_SIDES.index(side): t})
    field.boundary_conditions[side] = BoundaryCondition(bc.kind, t)


# ---- Field (src/Fields/field.jl:16-31) ---------------------------------------------------------
class Field:
    def __init__(self, loc, grid, boundary_conditions=None, _handle=None, auxiliary=False):
        self.grid, self.loc = grid, tuple(loc)
        self._owned = _handle is None
        # the resolved boundary conditions; a model sets those of its fields itself
        self.boundary_conditions = _resolve_bcs(grid, self.loc, boundary_conditions, auxiliary)
        if _handle is None:
            tables = _array_tables(grid, self.loc, self.boundary_conditions)
            h = C.c_void_p()
            locs = (C.c_int32 * 3)(*[_LOC[l] for l in self.loc])
            check(lib.ob200_field_create(grid.handle, locs, _bc_array(grid, self.loc, boundary_conditions, auxiliary),
                                         C.byref(h)))
            _handle = h
            _push_boundary_values(h, tables)
        self.handle = _handle
        ps = (C.c_int32 * 3)()
        check(lib.ob200_field_parent_size(self.handle, ps))
        self.parent_size = tuple(ps)

    def size(self):
        g = self.grid
        return tuple(g.N[d] + (1 if (self.loc[d] == Face and g.topology[d] == Bounded) else 0) for d in range(3))

    def parent(self):
        """Array(parent(field)) -- reference layout incl. halos, column-major."""
        a = np.zeros(self.parent_size, dtype=self.grid.FT, order="F")
        check(lib.ob200_field_get_parent(self.handle, a.ctypes.data_as(C.c_void_p)))
        return a

    def set_parent(self, a):
        a = np.asfortranarray(a, dtype=self.grid.FT)
        if a.shape != self.parent_size:
            raise ValueError(f"parent array has shape {a.shape}, expected {self.parent_size}")
        check(lib.ob200_field_set_parent(self.handle, a.ctypes.data_as(C.c_void_p)))

    def _islice(self):
        n, H = self.size(), self.grid.H
        return tuple(slice(H[d], H[d] + n[d]) for d in range(3))

    def interior(self):
        return self.parent()[self._islice()]

    def set(self, value):
        """set!(field, value) (src/Fields/set!.jl:20-65): array or function of (x, y, z)."""
        n = self.size()
        if callable(value):
            x, y, z = self.grid.nodes(self.loc)
            value = value(x, y, z) + np.zeros(n)
        p = self.parent()
        p[self._islice()] = np.asarray(value, dtype=self.grid.FT).reshape(n)
        self.set_parent(p)

    def slice(self, lo, hi, out=None, sync=True):
        """dense copy of the index box lo..hi (Julia indices, 1-based, inclusive; halo indices allowed), gathered on the device:
        only the box travels to the host (fetch_output with a FieldSlicer, OutputWriters/fetch_output.jl:24-36).  With
        sync=False the array is valid after sync() / ob200_sync_downloads."""
        shape = tuple(int(h) - int(l) + 1 for l, h in zip(lo, hi))
        if out is None:
            out = np.empty(shape, dtype=self.grid.FT, order="F")
        check(lib.ob200_field_slice_async(self.handle, (C.c_int32 * 3)(*[int(x) for x in lo]),
                                          (C.c_int32 * 3)(*[int(x) for x in hi]), out.ctypes.data_as(C.c_void_p)))
        if sync:
            check(lib.ob200_sync())
        return out

    def average(self, dims, out=None, sync=True):
        """mean(field, dims=...) over the interior, reduced on the device (AveragedField); dims: 1-based dimension numbers as in
        the reference, e.g. (1, 2) for a horizontal average.  Averaged dimensions keep extent 1."""
        flags = [1 if (d + 1) in tuple(dims) else 0 for d in range(3)]
        n = self.size()
        shape = tuple(1 if flags[d] else n[d] for d in range(3))
        if out is None:
            out = np.empty(shape, dtype=self.grid.FT, order="F")
        check(lib.ob200_field_average_async(self.handle, (C.c_int32 * 3)(*flags), out.ctypes.data_as(C.c_void_p)))
        if sync:
            check(lib.ob200_sync())
        return out

    def reduce(self):
        s, s2, mx, nan = C.c_double(), C.c_double(), C.c_double(), C.c_int32()
        check(lib.ob200_field_reduce(self.handle, C.byref(s), C.byref(s2), C.byref(mx), C.byref(nan)))
        return dict(sum=s.value, sumsq=s2.value, maxabs=mx.value, has_nan=bool(nan.value))

    def __del__(self):
        try:
            if self._owned and self.handle:
                lib.ob200_field_destroy(self.handle)
        except Exception:
            pass


def CenterField(grid, boundary_conditions=None):
    return Field((Center, Center, Center), grid, boundary_conditions)


def XFaceField(grid, boundary_conditions=None):
    return Field((Face, Center, Center), grid, boundary_conditions)


def YFaceField(grid, boundary_conditions=None):
    return Field((Center, Face, Center), grid, boundary_conditions)


def ZFaceField(grid, boundary_conditions=None):
    return Field((Center, Center, Face), grid, boundary_conditions)


def fill_halo_regions(fields):
    """fill_halo_regions!(fields) (src/BoundaryConditions/fill_halo_regions.jl:34-82,
    src/Fields/field_tuples.jl:51-77)."""
    if isinstance(fields, Field):
        fields = [fields]
    fields = list(fields.values()) if isinstance(fields, dict) else list(fields)
    arr = (C.c_void_p * len(fields))(*[f.handle for f in fields])
    check(lib.ob200_fill_halo_regions(arr, len(fields)))


# ---- solvers (src/Solvers) -----------------------------------------------------------------------
class _PoissonSolver:
    KIND = L.SOLVER_AUTO

    def __init__(self, grid):
        self.grid = grid
        h = C.c_void_p()
        check(lib.ob200_poisson_create(grid.handle, self.KIND, C.byref(h)))
        self.handle = h

    def __del__(self):
        try:
            lib.ob200_poisson_destroy(self.handle)
        except Exception:
            pass


class FFTBasedPoissonSolver(_PoissonSolver):
    """src/Solvers/fft_based_poisson_solver.jl:50-72."""
    KIND = L.SOLVER_FFT


class FourierTridiagonalPoissonSolver(_PoissonSolver):
    """src/Solvers/fourier_tridiagonal_poisson_solver.jl:30-72."""
    KIND = L.SOLVER_FT


def solve(phi, solver, rhs):
    """solve!(ϕ, solver, rhs): rhs is the real source term, an (Nx, Ny, Nz) array
    (fft_based_poisson_solver.jl:93-120; fourier_tridiagonal_poisson_solver.jl:74-118)."""
    g = solver.grid
    rhs = np.asfortranarray(rhs, dtype=g.FT)
    if rhs.shape != g.N:
        raise ValueError("rhs must have the grid's interior size")
    check(lib.ob200_poisson_solve(solver.handle, phi.handle, rhs.ctypes.data_as(C.c_void_p)))
    return phi


def solve_for_pressure(pressure, solver, dt, U):
    """solve_for_pressure!(pressure, solver, Δt, U★) (solve_for_pressure.jl:55-89)."""
    check(lib.ob200_solve_for_pressure(solver.handle, pressure.handle, float(dt), U["u"].handle, U["v"].handle,
                                       U["w"].handle))


class BatchedTridiagonalSolver:
    """src/Solvers/batched_tridiagonal_solver.jl:10-72 (array coefficients)."""

    def __init__(self, grid, lower_diagonal, diagonal, upper_diagonal):
        self.grid = grid
        Nx, Ny, Nz = grid.N
        self.a = np.ascontiguousarray(lower_diagonal, dtype=np.float64)
        self.c = np.ascontiguousarray(upper_diagonal, dtype=np.float64)
        b = np.asarray(diagonal, dtype=np.float64)
        if b.ndim == 1:
            b = np.broadcast_to(b.reshape(1, 1, Nz), (Nx, Ny, Nz))
        self.b = np.asfortranarray(b)

    def solve(self, rhs):
        g = self.grid
        Nx, Ny, Nz = g.N
        cplx = np.iscomplexobj(rhs)
        dt = (np.complex64 if g.FT == np.float32 else np.complex128) if cplx else g.FT
        rhs = np.asfortranarray(np.broadcast_to(rhs, (Nx, Ny, Nz)) if np.ndim(rhs) == 3 else
                                np.broadcast_to(np.asarray(rhs).reshape(1, 1, Nz), (Nx, Ny, Nz)), dtype=dt)
        out = np.zeros((Nx, Ny, Nz), dtype=dt, order="F")
        P = lambda a: a.ctypes.data_as(C.c_void_p)
        check(lib.ob200_batched_tridiagonal_solve(L.F32 if g.FT == np.float32 else L.F64, int(cplx), Nx, Ny, Nz,
                                                  P(self.a), P(self.b), P(self.c), P(rhs), P(out)))
        return out


# ---- model components -----------------------------------------------------------------------------
class _Adv:
    name = "none"
    required_halo = 1


class CenteredSecondOrder(_Adv):
    name, required_halo = "CenteredSecondOrder", 1


class CenteredFourthOrder(_Adv):
    name, required_halo = "CenteredFourthOrder", 2


class UpwindBiasedFirstOrder(_Adv):
    name, required_halo = "UpwindBiasedFirstOrder", 2


class UpwindBiasedThirdOrder(_Adv):
    name, required_halo = "UpwindBiasedThirdOrder", 2


class UpwindBiasedFifthOrder(_Adv):
    name, required_halo = "UpwindBiasedFifthOrder", 3


def _eno_weights(r, x, i):
    """interp_weights(r, coord, i, 0, -) (src/Advection/weno_fifth_order.jl:740-772)."""
    out = []
    for j in range(3):
        c = 0
        for m in range(j + 1, 4):
            num = 0
            for l in range(4):
                if l == m:
                    continue
                pr = 1
                for q in range(4):
                    if q != m and q != l:
                        pr *= x[i] - x[i - (r - q + 1)]
                num += pr
            den = 1
            for l in range(4):
                if l != m:
                    den *= x[i - (r - m + 1)] - x[i - (r - l + 1)]
            c += num / den
        out.append(c * (x[i - (r - j)] - x[i - (r - j + 1)]))
    return out


class WENO5(_Adv):
    """WENO5(FT; grid=nothing, zweno=true) (src/Advection/weno_fifth_order.jl:164-180).  With
    `grid`, stretched dimensions get the ENO coefficient tables of :182-209,562-584."""
    name, required_halo = "WENO5", 3

    def __init__(self, FT=None, grid=None, zweno=True, stretched_smoothness=False):
        if stretched_smoothness:
            raise ValueError("stretched_smoothness=true is outside the B200 path's supported set")
        self.FT = grid.FT if grid is not None else (np.dtype(FT).type if FT is not None else np.float64)
        self.zweno = bool(zweno)
        self.tables = {}
        if grid is not None:
            g4 = grid.with_halo((4, 4, 4))
            for d in range(3):
                if g4.regular[d]:
                    continue
                for li, nodes in ((0, g4.F[d]), (1, g4.C[d])):
                    n2 = g4.N[d] + 2
                    t = np.zeros((4, n2, 3))
                    for ri, r in enumerate((-1, 0, 1, 2)):
                        for i in range(n2):
                            t[ri, i] = [float(self.FT(w)) for w in _eno_weights(r, nodes, i)]
                    self.tables[(d, li)] = np.ascontiguousarray(t)


class ScalarDiffusivity:
    """ScalarDiffusivity(formulation; ν, κ) (scalar_diffusivity.jl:60-76), constants only."""
    required_halo = 1

    def __init__(self, formulation="ThreeDimensional", ν=0.0, κ=0.0, nu=None, kappa=None, time_discretization="Explicit"):
        ν = nu if nu is not None else ν
        κ = kappa if kappa is not None else κ
        if time_discretization not in ("Explicit", "VerticallyImplicit"):
            raise ValueError("time_discretization must be 'Explicit' or 'VerticallyImplicit'")
        if time_discretization == "VerticallyImplicit" and formulation == "Horizontal":
            raise ValueError("VerticallyImplicitTimeDiscretization is not supported for HorizontalScalarDiffusivity")
        self.time_discretization = time_discretization
        if callable(ν) or callable(κ) or isinstance(ν, np.ndarray):
            raise ValueError("only constant ν, κ are supported on the B200 architecture")
        if formulation not in L.CLOSURE:
            raise ValueError(f"unsupported formulation {formulation}")
        self.formulation, self.ν, self.κ = formulation, ν, κ


class SmagorinskyLilly:
    """SmagorinskyLilly(FT; C=0.16, Cb=1.0, Pr=1.0) (src/TurbulenceClosures/turbulence_closure_implementations/
    smagorinsky_lilly.jl:6-72), explicit time discretisation; Pr is a number or a dict {tracer name: number}."""
    required_halo = 1
    formulation = "ThreeDimensional"

    def __init__(self, C=0.16, Cb=1.0, Pr=1.0):
        self.C, self.Cb, self.Pr = C, Cb, Pr

    def prandtl(self, name):
        return self.Pr[name] if isinstance(self.Pr, dict) else self.Pr


class AnisotropicMinimumDissipation:
    """AnisotropicMinimumDissipation(FT; C=1/12, Cν=nothing, Cκ=nothing, Cb=nothing) (src/TurbulenceClosures/
    turbulence_closure_implementations/anisotropic_minimum_dissipation.jl:96-105); constant Poincaré constants (Cκ a
    number or a dict per tracer), explicit time discretisation."""
    required_halo = 1
    formulation = "ThreeDimensional"

    def __init__(self, C=1 / 12, Cν=None, Cκ=None, Cb=None):
        self.Cν = C if Cν is None else Cν
        self.Cκ = C if Cκ is None else Cκ
        self.Cb = Cb
        for v in (self.Cν, self.Cκ):
            if callable(v):
                raise ValueError("only constant Poincaré constants are supported on the B200 architecture")

    def Ck(self, name):
        return self.Cκ[name] if isinstance(self.Cκ, dict) else self.Cκ


def VerticalScalarDiffusivity(**kw):
    return ScalarDiffusivity("Vertical", **kw)


def HorizontalScalarDiffusivity(**kw):
    return ScalarDiffusivity("Horizontal", **kw)


class FPlane:
    def __init__(self, f):
        self.f = f


class BuoyancyTracer:
    pass


class LinearEquationOfState:
    """LinearEquationOfState(FT; thermal_expansion=1.67e-4, haline_contraction=7.80e-4)
    (src/BuoyancyModels/linear_equation_of_state.jl:6-30)"""

    def __init__(self, thermal_expansion=1.67e-4, haline_contraction=7.80e-4):
        self.thermal_expansion, self.haline_contraction = thermal_expansion, haline_contraction


class SeawaterBuoyancy:
    """SeawaterBuoyancy(FT; gravitational_acceleration=g_Earth, equation_of_state=LinearEquationOfState(FT),
    constant_temperature=nothing, constant_salinity=nothing) (src/BuoyancyModels/seawater_buoyancy.jl:61-73).
    Only the linear equation of state crosses the C ABI."""
    g_Earth = 9.80665            # BuoyancyModels.jl:20

    def __init__(self, gravitational_acceleration=None, equation_of_state=None, constant_temperature=None,
                 constant_salinity=None):
        self.gravitational_acceleration = self.g_Earth if gravitational_acceleration is None else gravitational_acceleration
        self.equation_of_state = equation_of_state or LinearEquationOfState()
        if not isinstance(self.equation_of_state, LinearEquationOfState):
            raise ValueError("only LinearEquationOfState is supported on the B200 architecture")
        self.constant_temperature = 0.0 if constant_temperature is True else constant_temperature
        self.constant_salinity = 0.0 if constant_salinity is True else constant_salinity
        if self.constant_temperature is not None and self.constant_salinity is not None:
            raise ValueError("temperature and salinity cannot both be constant")

    def required_tracers(self):
        if self.constant_salinity is not None:
            return ("T",)
        if self.constant_temperature is not None:
            return ("S",)
        return ("T", "S")


class Buoyancy:
    def __init__(self, model=None, gravity_unit_vector=None):
        self.model = model or BuoyancyTracer()
        if not isinstance(self.model, (BuoyancyTracer, SeawaterBuoyancy)):
            raise ValueError("only BuoyancyTracer and SeawaterBuoyancy(LinearEquationOfState) are supported on the B200 architecture")
        self.g = gravity_unit_vector


# ---- forcing (src/Forcings/relaxation.jl) ------------------------------------------------------------
_DIMS = {"x": 0, "y": 1, "z": 2}


def _param(v):
    """a parameter as Julia would hold it: a Python float is a Float64 (it promotes Float32 nodes), everything else as given"""
    return np.float64(v) if isinstance(v, float) else v


def _is_number(v):
    return isinstance(v, (int, float, np.integer, np.floating)) and not isinstance(v, bool)


class GaussianMask:
    """GaussianMask{D}(center, width) (relaxation.jl): exp(-(ξ - center)² / (2 width²)) along dimension D = "x", "y" or "z"."""

    def __init__(self, dim, center, width):
        if dim not in _DIMS:
            raise ValueError(f"GaussianMask dimension must be one of 'x', 'y', 'z', got {dim!r}")
        if not (_is_number(center) and _is_number(width)):
            raise ValueError("GaussianMask center and width must be numbers")
        self.dim, self.center, self.width = dim, center, width

    def __call__(self, xi):
        c, w = _param(self.center), _param(self.width)
        return np.exp(-(xi - c) ** 2 / (2 * w ** 2))


class LinearTarget:
    """LinearTarget{D}(intercept, gradient) (relaxation.jl): intercept + gradient ξ along dimension D, independent of time."""

    def __init__(self, dim, intercept, gradient):
        if dim not in _DIMS:
            raise ValueError(f"LinearTarget dimension must be one of 'x', 'y', 'z', got {dim!r}")
        if not (_is_number(intercept) and _is_number(gradient)):
            raise ValueError("LinearTarget intercept and gradient must be numbers")
        self.dim, self.intercept, self.gradient = dim, intercept, gradient

    def __call__(self, xi):
        return _param(self.intercept) + _param(self.gradient) * xi


class Relaxation:
    """Relaxation(; rate, mask=onefunction, target=zerofunction) (src/Forcings/relaxation.jl): the forcing
    rate * mask(x, y, z) * (target(x, y, z, t) - ψ) of the field ψ it is given for.  mask: None (onefunction) or a
    GaussianMask; target: None (zerofunction), a number or a LinearTarget."""

    def __init__(self, rate, mask=None, target=None):
        if not _is_number(rate):
            raise ValueError(f"Relaxation rate must be a number, got {type(rate).__name__}")
        if mask is not None and not isinstance(mask, GaussianMask):
            raise ValueError("Relaxation mask must be None (onefunction) or a GaussianMask on the B200 architecture")
        if target is not None and not (_is_number(target) or isinstance(target, LinearTarget)):
            raise ValueError("Relaxation target must be None (zerofunction), a number or a LinearTarget on the B200 architecture")
        self.rate, self.mask, self.target = rate, mask, target


def relaxation_tables(relaxation, loc, grid):
    """Host tables of a Relaxation for a field at `loc` of `grid` (anything with .topology and .nodes(loc), the interior nodes
    broadcast-shaped): (mask_dim, M, target_dim, T) with M = rate * mask at the field's nodes along mask_dim (-1: M is the
    number rate) and T = the target there (-1: the number target).  Evaluated as the reference evaluates the forcing at a point:
    parameters and nodes in their promoted type, rate * mask first.  No library call."""
    def nodes(d, what):
        if grid.topology[d] == Flat:
            raise ValueError(f"Relaxation {what} along the Flat dimension {'xyz'[d]}")
        return np.asarray(grid.nodes(loc)[d]).ravel()
    rate = _param(relaxation.rate)
    m = relaxation.mask
    if m is None:
        md, M = -1, rate
    else:
        md = _DIMS[m.dim]
        M = rate * m(nodes(md, "mask"))
    t = relaxation.target
    if isinstance(t, LinearTarget):
        td = _DIMS[t.dim]
        T = t(nodes(td, "target"))
    else:
        td, T = -1, (0 if t is None else _param(t))
    return md, M, td, T


# ---- background fields (src/Models/NonhydrostaticModels/background_fields.jl) ----------------------------
class BackgroundField:
    """BackgroundField(func; parameters=nothing) (background_fields.jl): a steady field U(x, y, z, t) that the model's velocities
    or tracers are perturbations about.  The B200 path tabulates it ONCE, at the clock time of construction: a time-dependent
    background is updated by the caller, e.g. `set_background(model, "b", func_or_array, time=t)` in a callback."""

    def __init__(self, func, parameters=None):
        if not callable(func):
            raise ValueError(f"a BackgroundField needs a callable, got {type(func).__name__}")
        self.func, self.parameters = func, parameters


def _parent_nodes(grid, loc):
    """x, y, z of every node of the parent array of a field at `loc` (halos included; the extra Face point on Bounded dimensions;
    the Flat coordinate along Flat dimensions), broadcast-shaped, in double"""
    out = []
    for d in range(3):
        src = grid.F[d] if loc[d] == Face else grid.C[d]
        if grid.topology[d] == Flat:
            a = np.asarray(src.span(1, 1))
        else:
            n = grid.N[d] + 2 * grid.H[d] + (1 if (loc[d] == Face and grid.topology[d] == Bounded) else 0)
            a = np.asarray(src.span(1 - grid.H[d], n - grid.H[d]))
        shape = [1, 1, 1]
        shape[d] = len(a)
        out.append(a.astype(np.float64).reshape(shape))
    return out


def background_table(grid, loc, background, time=0.0):
    """The parent-shaped table of a background (a BackgroundField or a bare callable) for a field at `loc`: the function at every
    node of the parent, halos included, as the reference's FunctionField evaluates it (its halos are never filled, not even along
    a Periodic dimension), called as func(x, y, z, t) or func(x, y, z, t, parameters), evaluated in double and rounded once to the
    grid's float type.  No library call."""
    bf = background if isinstance(background, BackgroundField) else BackgroundField(background)
    x, y, z = _parent_nodes(grid, loc)
    t = np.float64(time)
    v = bf.func(x, y, z, t) if bf.parameters is None else bf.func(x, y, z, t, bf.parameters)
    shape = tuple(len(a) for a in (x.ravel(), y.ravel(), z.ravel()))
    try:
        v = np.broadcast_to(np.asarray(v, dtype=np.float64), shape)
    except ValueError:
        raise ValueError(f"the background function returned shape {np.shape(v)}, which does not broadcast to the field's "
                         f"parent {shape}") from None
    return np.asfortranarray(v.astype(grid.FT))


def set_background(model, name, value, time=None):
    """Replace the background of field `name` (one the model was built with): `value` is a parent-shaped array or a function /
    BackgroundField, evaluated as at construction at `time` (default: the model's clock).  The copy is ordered after every step
    enqueued so far, so it takes effect from the next step on; this is how a time-dependent background is advanced."""
    if name not in model.background_fields:
        raise ValueError(f"{name} has no background field; backgrounds: {tuple(model.background_fields)}")
    f = model.background_fields[name]
    if callable(value) or isinstance(value, BackgroundField):
        value = background_table(model.grid, f.loc, value, model.clock.time if time is None else time)
    f.set_parent(value)


class Clock:
    def __init__(self, model):
        self._m = model

    @property
    def time(self):
        t = C.c_double()
        check(lib.ob200_model_clock(self._m.handle, C.byref(t), None))
        return t.value

    @property
    def iteration(self):
        it = C.c_int64()
        check(lib.ob200_model_clock(self._m.handle, None, C.byref(it)))
        return it.value


class NonhydrostaticModel:
    """NonhydrostaticModel(; grid, advection, closure, coriolis, buoyancy, tracers, timestepper,
    boundary_conditions) (src/Models/NonhydrostaticModels/nonhydrostatic_model.jl:102-203).
    Defaults as in the reference: advection = CenteredSecondOrder(), timestepper =
    :QuasiAdamsBashforth2.  `forcing` = {field name: Relaxation(...)}.  `background_fields` = {field name: BackgroundField(...)
    or a callable}: evaluated once, at time 0, over each field's whole parent (background_table); model.background_fields holds
    the resulting fields and set_background replaces their values.  Unsupported pieces (function-valued forcings, function BCs,
    immersed boundaries, particles, closures other than ScalarDiffusivity / SmagorinskyLilly / AnisotropicMinimumDissipation)
    raise ArgumentError-like ValueErrors."""

    def __init__(self, grid, advection="default", closure=None, coriolis=None, buoyancy=None, tracers=(),
                 timestepper="QuasiAdamsBashforth2", boundary_conditions=None, forcing=None,
                 background_fields=None, particles=None, immersed_boundary=None, stokes_drift=None,
                 pressure_solver=None, chi=0.1):
        for name, v in (("particles", particles),
                        ("immersed_boundary", immersed_boundary), ("stokes_drift", stokes_drift)):
            if v:
                raise ValueError(f"`{name}` is not supported on the B200 architecture (SURVEY.md 8(b))")
        if not isinstance(grid, RectilinearGrid):
            raise ValueError("the B200 architecture supports RectilinearGrid only")
        if advection == "default":
            advection = CenteredSecondOrder()
        if timestepper not in L.TS:
            raise ValueError(f"unknown timestepper {timestepper}")
        if isinstance(buoyancy, (BuoyancyTracer, SeawaterBuoyancy)):
            buoyancy = Buoyancy(buoyancy)
        tracers = (tracers,) if isinstance(tracers, str) else tuple(tracers or ())
        if buoyancy is not None:          # validate_buoyancy (BuoyancyModels.jl:37-46)
            req = ("b",) if isinstance(buoyancy.model, BuoyancyTracer) else buoyancy.model.required_tracers()
            for n in req:
                if n not in tracers:
                    raise ValueError(f"{type(buoyancy.model).__name__} requires a tracer named :{n}")
        if len(tracers) > L.MAX_TRACERS:
            raise ValueError("too many tracers")
        if isinstance(advection, WENO5) and advection.FT != grid.FT:
            raise ValueError("WENO5 float type differs from the grid's; construct it as WENO5(grid.FT) or WENO5(grid=grid)")
        names = ("u", "v", "w") + tracers
        locs = [(Face, Center, Center), (Center, Face, Center), (Center, Center, Face)] + [(Center,) * 3] * len(tracers)
        # model_forcing (Forcings/model_forcing.jl): every name must be a prognostic field; the tables come from the interior
        # nodes, which halo inflation does not change
        frc = {}
        if forcing:
            if not isinstance(forcing, dict):
                raise ValueError("forcing must be a dict {field name: Relaxation(...)}")
            for n, fr in forcing.items():
                if n not in names:
                    raise ValueError(f"{n} is not a prognostic field of the model; forcing names must be among {names}")
                if not isinstance(fr, Relaxation):
                    raise ValueError(f"the forcing of {n} is a {type(fr).__name__}: only Relaxation crosses the C ABI of the B200 "
                                     "architecture (function-valued forcings are outside its supported set)")
                frc[names.index(n)] = relaxation_tables(fr, locs[names.index(n)], grid)
        if background_fields is not None and not isinstance(background_fields, dict):
            raise ValueError("background_fields must be a dict {field name: BackgroundField(...) or a function}")
        for n, bf in (background_fields or {}).items():
            if n not in names:
                raise ValueError(f"{n} is not a prognostic field of the model; background field names must be among {names}")
            if not (callable(bf) or isinstance(bf, BackgroundField)):
                raise ValueError(f"the background of {n} is a {type(bf).__name__}: it must be a BackgroundField or a function "
                                 "(x, y, z, t)")
        # halo inflation (nonhydrostatic_model.jl:140-148)
        H = list(grid.H)
        for term in (advection, closure):
            req = 1 if term is None else term.required_halo
            for d in range(3):
                H[d] = 0 if grid.topology[d] == Flat else max(req, H[d])
        if tuple(H) != grid.H:
            grid = grid.with_halo(H)
        self.grid, self.advection, self.closure, self.coriolis, self.buoyancy = grid, advection, closure, coriolis, buoyancy
        self.tracer_names, self.timestepper = tracers, timestepper
        d = L.ModelDesc()
        d.grid = grid.handle
        d.timestepper, d.chi = L.TS[timestepper], float(chi)
        d.advection = L.ADV[advection.name] if advection is not None else 0
        d.weno_zweno = int(getattr(advection, "zweno", True))
        self._keep = []
        if isinstance(advection, WENO5):
            for (dim, li), t in advection.tables.items():
                self._keep.append(t)
                d.weno_coeff[dim][li] = t.ctypes.data_as(C.POINTER(C.c_double))
        if isinstance(closure, AnisotropicMinimumDissipation):
            d.closure = L.CLOSURE["AnisotropicMinimumDissipation"]
            d.amd_Cnu = float(closure.Cν)
            d.amd_has_Cb, d.amd_Cb = int(closure.Cb is not None), float(closure.Cb or 0.0)
            for k, name in enumerate(tracers):
                d.amd_Ckappa[k] = float(closure.Ck(name))
        elif isinstance(closure, SmagorinskyLilly):
            d.closure = L.CLOSURE["SmagorinskyLilly"]
            d.smagorinsky_C, d.smagorinsky_Cb = float(closure.C), float(closure.Cb)
            for k, name in enumerate(tracers):
                d.prandtl[k] = float(closure.prandtl(name))
        else:
            d.closure = L.CLOSURE[closure.formulation] if closure is not None else 0
            if closure is not None:
                d.closure_vertically_implicit = int(closure.time_discretization == "VerticallyImplicit")
                d.nu = float(closure.ν)
                for k, name in enumerate(tracers):
                    d.kappa[k] = float(closure.κ[name] if isinstance(closure.κ, dict) else closure.κ)
        d.coriolis_fplane = int(coriolis is not None)
        if coriolis is not None:
            if not isinstance(coriolis, FPlane):
                raise ValueError("only FPlane is supported on the B200 architecture")
            d.f = float(coriolis.f)
        d.buoyancy_tracer, d.buoyancy_kind, d.temperature_tracer, d.salinity_tracer = -1, 0, -1, -1
        if buoyancy is not None and isinstance(buoyancy.model, SeawaterBuoyancy):
            sw = buoyancy.model
            d.buoyancy_kind = 1
            req = sw.required_tracers()
            d.temperature_tracer = tracers.index("T") if "T" in req else -1
            d.salinity_tracer = tracers.index("S") if "S" in req else -1
            d.gravitational_acceleration = float(sw.gravitational_acceleration)
            d.thermal_expansion = float(sw.equation_of_state.thermal_expansion)
            d.haline_contraction = float(sw.equation_of_state.haline_contraction)
        elif buoyancy is not None:
            d.buoyancy_tracer = tracers.index("b")
        d.gravity_tilted = int(buoyancy is not None and buoyancy.g is not None)
        g_hat = buoyancy.g if (buoyancy is not None and buoyancy.g is not None) else (0.0, 0.0, 1.0)
        for k in range(3):
            d.g_hat[k] = float(g_hat[k])
        d.ntracers = len(tracers)
        bcs = boundary_conditions or {}
        # array conditions: checked here, pushed once the model exists (set_model's update_state! then fills the halos with them)
        resolved = {n: _resolve_bcs(grid, loc, bcs.get(n)) for n, loc in zip(names, locs)}
        tables = {n: _array_tables(grid, loc, resolved[n]) for n, loc in zip(names, locs)}
        for q, (n, loc) in enumerate(zip(names, locs)):
            arr = _bc_array(grid, loc, bcs.get(n))
            for s in range(6):
                d.bcs[q][s].kind, d.bcs[q][s].value = arr[s].kind, arr[s].value
        d.pressure_solver = L.SOLVER_AUTO if pressure_solver is None else pressure_solver
        for q, (md, M, td, T) in frc.items():
            F = d.forcing[q]
            F.active, F.mask_dim, F.target_dim = 1, md, td
            if md < 0:
                F.rate = float(M)
            else:
                a = np.ascontiguousarray(M, dtype=np.float64)
                self._keep.append(a)
                F.mask = a.ctypes.data_as(C.POINTER(C.c_double))
            if td < 0:
                F.target_value = float(T)
            else:
                a = np.ascontiguousarray(T, dtype=np.float64)
                self._keep.append(a)
                F.target = a.ctypes.data_as(C.POINTER(C.c_double))
        self.forcing = dict(forcing or {})
        # backgrounds on the inflated grid (their halos are the function's values there), at the clock time of construction
        bgt = {n: background_table(grid, locs[names.index(n)], bf, 0.0) for n, bf in (background_fields or {}).items()}
        for n, t in bgt.items():
            self._keep.append(t)
            d.background[names.index(n)] = t.ctypes.data_as(C.c_void_p)
        h = C.c_void_p()
        check(lib.ob200_model_create(C.byref(d), C.byref(h)))
        self.handle = h
        self.names = names
        self.velocities = {n: self._field(n, n, locs[i]) for i, n in enumerate("uvw")}
        self.tracers = {n: self._field(f"c{k}", n, (Center,) * 3) for k, n in enumerate(tracers)}
        self.fields = {**self.velocities, **self.tracers}
        for n, f in self.fields.items():
            f.boundary_conditions = resolved[n]
            _push_boundary_values(f.handle, tables[n])
        self.pressures = {"pNHS": self._field("pNHS", "pNHS", (Center,) * 3)}
        if grid.topology[2] != Flat:
            self.pressures["pHY′"] = self._field("pHY", "pHY", (Center,) * 3)
        self.diffusivity_fields = {}
        if isinstance(closure, (SmagorinskyLilly, AnisotropicMinimumDissipation)):
            self.diffusivity_fields["νₑ"] = self._field("nu_e", "nu_e", (Center,) * 3)
        if isinstance(closure, AnisotropicMinimumDissipation):
            self.diffusivity_fields["κₑ"] = {n: self._field(f"kappa_e{k}", f"kappa_e_{n}", (Center,) * 3) for k, n in enumerate(tracers)}
        self.Gn = {n: self._field("Gn_" + (n if n in "uvw" else f"c{tracers.index(n)}"), n, locs[i])
                   for i, n in enumerate(names)}
        self.Gm = {n: self._field("Gm_" + (n if n in "uvw" else f"c{tracers.index(n)}"), n, locs[i])
                   for i, n in enumerate(names)}
        self.background_fields = {n: self._field("bg_" + (n if n in "uvw" else f"c{tracers.index(n)}"), n, locs[names.index(n)])
                                   for n in bgt}
        self.clock = Clock(self)

    def _field(self, cname, name, loc):
        h = C.c_void_p()
        check(lib.ob200_model_field(self.handle, cname.encode(), C.byref(h)))
        return Field(loc, self.grid, _handle=h)

    def use_fast_kernels(self, on=True):
        check(lib.ob200_model_use_fast_kernels(self.handle, int(on)))

    def diagnostics(self):
        a, b = C.c_double(), C.c_double()
        check(lib.ob200_model_diagnostics(self.handle, C.byref(a), C.byref(b)))
        return dict(max_abs_div=a.value, kinetic_energy=b.value)

    def set_clock(self, time=0.0, iteration=0, previous_Δt=float("inf")):
        """model.clock.time / .iteration = ...; previous_Δt = inf makes the next QuasiAdamsBashforth2 step a forward-Euler step
        with G^- cleared, as for a new model (quasi_adams_bashforth_2.jl:76-81)"""
        check(lib.ob200_model_set_clock(self.handle, float(time), int(iteration), float(previous_Δt)))

    def destroy(self):
        """release the library model now (device memory, streams, events, tensor maps); also done by the finalizer"""
        if getattr(self, "handle", None) is not None:
            lib.ob200_model_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def update_state(model):
    """update_state!(model) (update_nonhydrostatic_model_state.jl:14-37)."""
    check(lib.ob200_model_update_state(model.handle))


def calculate_tendencies(model):
    """calculate_tendencies!(model) (calculate_nonhydrostatic_tendencies.jl:12-36)."""
    check(lib.ob200_model_calculate_tendencies(model.handle))


def set_model(model, enforce_incompressibility=True, **kw):
    """set!(model; enforce_incompressibility=true, kwargs...) (set_nonhydrostatic_model.jl:32-59)."""
    for name, value in kw.items():
        if name not in model.fields:
            raise ValueError(f"name {name} not found in model.velocities or model.tracers.")
        model.fields[name].set(value)
    update_state(model)
    if enforce_incompressibility:
        check(lib.ob200_model_pressure_project(model.handle, 1.0))
        update_state(model)


def time_step(model, dt, euler=False):
    """time_step!(model, Δt; euler=false) (runge_kutta_3.jl:81-152, quasi_adams_bashforth_2.jl:70-104).
    Enqueues the whole step on the stream; does not synchronise."""
    check(lib.ob200_model_time_step(model.handle, float(dt), int(euler)))


def sync():
    check(lib.ob200_sync())
