# B200.jl -- the reference-side shim a maintainer adds to Oceananigans (a new src/B200/B200.jl, `include`d from
# src/Oceananigans.jl after the Models, plus the three one-line hooks listed in INTEGRATION.md).  It cannot be executed in
# this image (no Julia toolchain); it is written against Oceananigans v0.76.8 (the reference checkout) and against
# include/ocean_b200.h.  The Python package ocean_b200 is the executable stand-in the tests drive: every function below has
# its twin there (grid_handle <-> grids.py RectilinearGrid._create, model_desc <-> model.py NonhydrostaticModel._desc, ...).
#
# Everything is dispatch on the new architecture singleton; the reference's API is unchanged:
#     grid  = RectilinearGrid(B200(), size=(256,256,256), extent=(1,1,1), topology=(Periodic,Periodic,Periodic))
#     model = NonhydrostaticModel(; grid, advection=WENO5(), tracers=:b, buoyancy=BuoyancyTracer(),
#                                  timestepper=:RungeKutta3)
#     set!(model, u=..., v=...); run!(Simulation(model, Δt=..., stop_iteration=...))

module B200Arch

using OffsetArrays: OffsetArray
using Oceananigans
using Oceananigans.Architectures: AbstractArchitecture, AbstractMultiArchitecture, CPU
using Oceananigans.Grids: RectilinearGrid, Periodic, Bounded, Flat, FullyConnected, Center, Face,
                          topology, halo_size, total_length, offset_data, with_halo
using Oceananigans.Fields: Field, location, interior, VelocityFields, TracerFields, PressureFields, TendencyFields
using Oceananigans.BoundaryConditions: BoundaryCondition, FieldBoundaryConditions, Flux, Value, Gradient, Open,
                                       regularize_field_boundary_conditions
using Oceananigans.Advection: CenteredSecondOrder, CenteredFourthOrder, UpwindBiasedFirstOrder, UpwindBiasedThirdOrder,
                              UpwindBiasedFifthOrder, WENO5
using Oceananigans.TurbulenceClosures: ScalarDiffusivity, SmagorinskyLilly, AnisotropicMinimumDissipation, ThreeDimensionalFormulation, HorizontalFormulation,
                                       VerticalFormulation, ExplicitTimeDiscretization, VerticallyImplicitTimeDiscretization
using Oceananigans.Coriolis: FPlane
using Oceananigans.BuoyancyModels: Buoyancy, BuoyancyTracer, SeawaterBuoyancy, LinearEquationOfState, ZDirection, required_tracers
using Oceananigans.TimeSteppers: RungeKutta3TimeStepper, QuasiAdamsBashforth2TimeStepper, Clock
using Oceananigans.Solvers: FFTBasedPoissonSolver, FourierTridiagonalPoissonSolver, BatchedTridiagonalSolver
using Oceananigans.Models.NonhydrostaticModels: NonhydrostaticModel
using Oceananigans.Utils: tupleit
using Oceananigans.Forcings: Relaxation, GaussianMask, LinearTarget
using Oceananigans.Grids: xnodes, ynodes, znodes, topology

import Base: zeros, size, Array, copyto!
import Oceananigans.Architectures: device, array_type, arch_array, architecture, device_event, unsafe_free!
import Oceananigans.Grids: new_data
import Oceananigans.Fields: set!
import Oceananigans.TimeSteppers: time_step!, update_state!, calculate_tendencies!, calculate_pressure_correction!,
                                  pressure_correct_velocities!, store_tendencies!
import Oceananigans.BoundaryConditions: fill_halo_regions!
import Oceananigans.Solvers: solve!
import Oceananigans.Models.NonhydrostaticModels: PressureSolver, solve_for_pressure!
import Oceananigans.Utils: launch!

import Statistics
const lib = "libocean_b200.so"

"The new architecture singleton (src/Architectures.jl:68-75).  `device` selects the CUDA device of this process."
struct B200 <: AbstractArchitecture
    device :: Int32
end
B200() = B200(Int32(0))

function check(status::Int32)
    status == 0 && return nothing
    n = ccall((:ob200_last_error, lib), Csize_t, (Ptr{UInt8}, Csize_t), C_NULL, 0)
    buf = Vector{UInt8}(undef, n + 1)
    ccall((:ob200_last_error, lib), Csize_t, (Ptr{UInt8}, Csize_t), buf, n + 1)
    error(unsafe_string(pointer(buf)))                 # no CPU fallback: a failed call is an error, never a reroute
end

# ---- Architectures.jl:81-143 ------------------------------------------------------------------------------------
device(a::B200) = (check(ccall((:ob200_init, lib), Int32, (Int32,), a.device)); a.device)
launch!(::B200, args...; kw...) = error("B200(): KernelAbstractions kernels are not used on this architecture")
device_event(::B200) = nothing

"""
Device array of the B200 architecture (`array_type(::B200)`).  Two flavours:
  * raw: a library allocation (`ob200_malloc`), used for `zeros(FT, B200(), N...)` / `arch_array`;
  * field-backed: the parent array of a `Field`; it owns (or borrows from a model) an `ob200_field`, whose device storage
    is in the library's padded internal layout.  `Array(a)` / `copyto!(a, host)` convert to / from the reference's parent
    layout (`ob200_field_get_parent` / `ob200_field_set_parent`, Grids/new_data.jl:16-22).
"""
mutable struct B200Array{T, N} <: AbstractArray{T, N}
    ptr    :: Ptr{Cvoid}           # raw allocation (C_NULL if field-backed)
    field  :: Ptr{Cvoid}           # ob200_field* (C_NULL if raw)
    dims   :: NTuple{N, Int}
    owner  :: Any                  # keeps the grid / model that owns `field` alive
end
size(a::B200Array) = a.dims
Base.getindex(::B200Array, I...) = error("scalar indexing of a B200Array is not allowed; use Array(a)")
array_type(::B200) = B200Array
architecture(::B200Array) = B200()
unsafe_free!(a::B200Array) = (a.ptr != C_NULL && ccall((:ob200_free, lib), Int32, (Ptr{Cvoid},), a.ptr); a.ptr = C_NULL; nothing)

function B200Array{T, N}(::UndefInitializer, dims::NTuple{N, Int}) where {T, N}
    p = Ref{Ptr{Cvoid}}()
    check(ccall((:ob200_malloc, lib), Int32, (Ref{Ptr{Cvoid}}, Csize_t), p, prod(dims) * sizeof(T)))
    a = B200Array{T, N}(p[], C_NULL, dims, nothing)
    finalizer(unsafe_free!, a)
    return a
end
function zeros(FT, ::B200, N::Vararg{Int, D}) where D                      # Grids/zeros.jl:6-7
    a = B200Array{FT, D}(undef, N)
    check(ccall((:ob200_memset, lib), Int32, (Ptr{Cvoid}, Int32, Csize_t), a.ptr, 0, prod(N) * sizeof(FT)))
    return a
end
function arch_array(::B200, h::Array{T, N}) where {T, N}                   # Architectures.jl:102-111
    d = B200Array{T, N}(undef, size(h))
    GC.@preserve h check(ccall((:ob200_upload, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Csize_t), d.ptr, h, sizeof(h)))
    return d
end
arch_array(::B200, a::B200Array) = a
arch_array(::CPU, a::B200Array) = Array(a)
arch_array(::B200, a::Union{AbstractRange, Number, Function, Nothing}) = a
function Array(d::B200Array{T, N}) where {T, N}
    h = Array{T, N}(undef, d.dims)
    if d.field != C_NULL
        GC.@preserve h check(ccall((:ob200_field_get_parent, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), d.field, h))
    else
        GC.@preserve h check(ccall((:ob200_download, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Csize_t), h, d.ptr, sizeof(h)))
    end
    return h
end
function copyto!(d::B200Array{T, N}, h::Array{T, N}) where {T, N}
    size(h) == d.dims || throw(DimensionMismatch("copyto!(::B200Array, ::Array)"))
    if d.field != C_NULL
        GC.@preserve h check(ccall((:ob200_field_set_parent, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), d.field, h))
    else
        GC.@preserve h check(ccall((:ob200_upload, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Csize_t), d.ptr, h, sizeof(h)))
    end
    return d
end

# ---- descriptors (mirror the POD structs of ocean_b200.h; isbits, same field order) ------------------------------
struct GridDesc
    ftype::Int32; N::NTuple{3,Int32}; H::NTuple{3,Int32}; topology::NTuple{3,Int32}
    L::NTuple{3,Float64}; regular::NTuple{3,Int32}; delta::NTuple{3,Float64}
    dC::NTuple{3,Ptr{Float64}}; dC_first::NTuple{3,Int32}; dC_len::NTuple{3,Int32}
    dF::NTuple{3,Ptr{Float64}}; dF_first::NTuple{3,Int32}; dF_len::NTuple{3,Int32}
end
struct BC; kind::Int32; value::Float64; end
const MAX_TRACERS = 8
struct ForcingDesc          # ob200_forcing
    active::Int32; mask_dim::Int32; rate::Float64; mask::Ptr{Float64}
    target_dim::Int32; target_value::Float64; target::Ptr{Float64}
end
struct ModelDesc
    grid::Ptr{Cvoid}; timestepper::Int32; chi::Float64; advection::Int32; weno_zweno::Int32
    weno_coeff::NTuple{6,Ptr{Float64}}                     # [d][loc], d-major
    closure::Int32; nu::Float64; kappa::NTuple{MAX_TRACERS,Float64}
    coriolis_fplane::Int32; f::Float64; buoyancy_tracer::Int32; gravity_tilted::Int32; g_hat::NTuple{3,Float64}
    ntracers::Int32; bcs::NTuple{6 * (3 + MAX_TRACERS), BC}; pressure_solver::Int32
    buoyancy_kind::Int32; temperature_tracer::Int32; salinity_tracer::Int32
    gravitational_acceleration::Float64; thermal_expansion::Float64; haline_contraction::Float64
    smagorinsky_C::Float64; smagorinsky_Cb::Float64; prandtl::NTuple{MAX_TRACERS,Float64}
    amd_Cnu::Float64; amd_Ckappa::NTuple{MAX_TRACERS,Float64}; amd_Cb::Float64; amd_has_Cb::Int32
    closure_vertically_implicit::Int32
    forcing::NTuple{3 + MAX_TRACERS, ForcingDesc}
    background::NTuple{3 + MAX_TRACERS, Ptr{Cvoid}}
end

topo_code(::Type{Periodic}) = Int32(0); topo_code(::Type{Bounded}) = Int32(1); topo_code(::Type{Flat}) = Int32(2)
topo_code(::Type{FullyConnected}) = Int32(3)
loc_code(::Type{Center}) = Int32(0); loc_code(::Type{Face}) = Int32(1); loc_code(::Type{Nothing}) = Int32(0)

const B200Grid = RectilinearGrid{<:Any, <:Any, <:Any, <:Any, <:Any, <:Any, <:Any, <:Any, <:Any, <:Any,
                                 <:Union{B200, AbstractMultiArchitecture}}
const grid_handles = IdDict{Any, Ptr{Cvoid}}()      # grid => ob200_grid* (destroyed by the grid's finalizer hook, INTEGRATION.md)

"Marshal a RectilinearGrid (src/Grids/rectilinear_grid.jl:1-47) into an ob200_grid handle (cached per grid object)."
function grid_handle(grid::RectilinearGrid{FT}) where FT
    haskey(grid_handles, grid) && return grid_handles[grid]
    device(child_arch(architecture(grid)))
    Δc = (grid.Δxᶜᵃᵃ, grid.Δyᵃᶜᵃ, grid.Δzᵃᵃᶜ); Δf = (grid.Δxᶠᵃᵃ, grid.Δyᵃᶠᵃ, grid.Δzᵃᵃᶠ)
    reg = map(x -> x isa Number, Δc)
    vec64(x) = x isa Number ? Float64[] : Float64.(parent(x))          # parents of the OffsetVectors, halos included
    first_index(x) = x isa Number ? Int32(0) : Int32(first(axes(x, 1)))
    keep = (map(vec64, Δc), map(vec64, Δf))
    ptr(v) = isempty(v) ? Ptr{Float64}(C_NULL) : pointer(v)
    desc = GridDesc(FT == Float32 ? 0 : 1, Int32.(size(grid)), Int32.(halo_size(grid)), topo_code.(topology(grid)),
                    Float64.((grid.Lx, grid.Ly, grid.Lz)), Int32.(reg), map(x -> x isa Number ? Float64(x) : 0.0, Δc),
                    map(ptr, keep[1]), map(first_index, Δc), Int32.(map(length, keep[1])),
                    map(ptr, keep[2]), map(first_index, Δf), Int32.(map(length, keep[2])))
    h = Ref{Ptr{Cvoid}}()
    GC.@preserve keep check(ccall((:ob200_grid_create, lib), Int32, (Ref{GridDesc}, Ref{Ptr{Cvoid}}), desc, h))
    grid_handles[grid] = h[]
    return h[]
end
child_arch(a::B200) = a
child_arch(a::AbstractMultiArchitecture) = a.child_architecture

# ---- fields: Fields/field.jl:151-159 -> Grids/new_data.jl:56-61 ---------------------------------------------------
bc_code(::Nothing) = BC(0, 0.0)
bc_code(bc::BoundaryCondition{<:Flux})     = BC(2, constant_value(bc))
bc_code(bc::BoundaryCondition{<:Value})    = BC(3, constant_value(bc))
bc_code(bc::BoundaryCondition{<:Gradient}) = BC(4, constant_value(bc))
bc_code(bc::BoundaryCondition{<:Open})     = BC(5, constant_value(bc))
bc_code(bc::BoundaryCondition)             = BC(1, 0.0)                 # Periodic / communication: decided by the topology
# an array condition crosses as its kind with value 0; its values follow through ob200_field_set_boundary_values
constant_value(bc) = bc.condition === nothing ? 0.0 : bc.condition isa Number ? Float64(bc.condition) :
    bc.condition isa AbstractMatrix ? 0.0 :
    throw(ArgumentError("B200(): only constant and 2-D array boundary conditions are supported (function conditions cannot cross the C ABI)"))
bc_codes(bcs::FieldBoundaryConditions) = map(bc_code, (bcs.west, bcs.east, bcs.south, bcs.north, bcs.bottom, bcs.top))
bc_codes(::Nothing) = ntuple(_ -> BC(0, 0.0), 6)

# ---- array conditions: FluxBoundaryCondition(Q) / ValueBoundaryCondition(Q) / GradientBoundaryCondition(Q), Q a 2-D array
# indexed by the grid's interior indices along the side's tangential dimensions (getbc(bc::BC{<:Any,<:AbstractArray}, i, j,
# grid) = bc.condition[i, j], BoundaryConditions/boundary_condition.jl) --------------------------------------------------------
const SIDES = (:west, :east, :south, :north, :bottom, :top)

"""
The condition of an array boundary condition once it lives in the library (the reference requires it on the device,
boundary_condition.jl:143-149).  `copyto!(q, Q)` and `q .= ...` (a callback varying the forcing in time) call
ob200_field_set_boundary_values, ordered after every step enqueued so far; reads see the host copy of the last values.
"""
mutable struct B200BoundaryArray{T} <: AbstractMatrix{T}
    field :: Ptr{Cvoid}            # ob200_field* of the model field
    side  :: Int32                 # 0..5 = west, east, south, north, bottom, top
    host  :: Matrix{T}             # the values last sent
    owner :: Any                   # keeps the model handle alive
end
size(q::B200BoundaryArray) = size(q.host)
architecture(::B200BoundaryArray) = B200()       # passes the reference's device check of array conditions
Base.getindex(q::B200BoundaryArray, i::Int, j::Int) = q.host[i, j]
Base.setindex!(::B200BoundaryArray, v, i...) = error("set the values of a B200 boundary condition with `copyto!` or `.=`")
function copyto!(q::B200BoundaryArray{T}, h::AbstractMatrix) where T
    size(h) == size(q.host) || throw(DimensionMismatch("boundary values of size $(size(h)), the side needs $(size(q.host))"))
    copyto!(q.host, h)
    GC.@preserve q check(ccall((:ob200_field_set_boundary_values, lib), Int32, (Ptr{Cvoid}, Int32, Ptr{Cvoid}),
                               q.field, q.side, q.host))
    return q
end
copyto!(q::B200BoundaryArray{T}, bc::Base.Broadcast.Broadcasted) where T = copyto!(q, copyto!(similar(q.host), bc))

"The (N_a, N_b) host table of the array condition of `side` of a field at `loc`, checked as the library does, or nothing."
function boundary_table(bc, side, grid, loc)
    bc === nothing && return nothing
    Q = bc.condition
    Q isa AbstractArray || return nothing
    d = (findfirst(==(side), SIDES) - 1) ÷ 2 + 1
    Q isa AbstractMatrix && eltype(Q) <: Real ||
        throw(ArgumentError("B200(): the $side boundary condition must be a 2-D real array, got $(typeof(Q))"))
    any(t -> t === FullyConnected, topology(grid)) &&
        throw(ArgumentError("B200(): array boundary conditions are not supported on slab-decomposed (FullyConnected) grids"))
    topology(grid, d) === Bounded ||
        throw(ArgumentError("B200(): array boundary condition on the $side side of a $(topology(grid, d)) dimension"))
    bc.classification isa Union{Flux, Value, Gradient} ||
        throw(ArgumentError("B200(): array boundary conditions must be Flux, Value or Gradient conditions"))
    loc[d] === Face &&
        throw(ArgumentError("B200(): the $side side of a field on the $("xyz"[d])-faces is the impenetrable wall"))
    shape = Tuple(topology(grid, e) === Flat ? 1 : size(grid, e) for e in 1:3 if e != d)
    size(Q) == shape || throw(ArgumentError("B200(): the $side boundary condition has size $(size(Q)); the grid needs $shape"))
    return Matrix{eltype(grid)}(Array(Q))
end

"Push the array conditions of a model field and return its boundary conditions with those conditions as B200BoundaryArrays."
function attach_boundary_arrays(fbcs::FieldBoundaryConditions, tables, fh::Ptr{Cvoid}, owner)
    isempty(tables) && return fbcs
    conds = map(fieldnames(typeof(fbcs))) do name
        bc = getfield(fbcs, name)
        haskey(tables, name) || return bc
        q = B200BoundaryArray(fh, Int32(findfirst(==(name), SIDES) - 1), similar(tables[name]), owner)
        copyto!(q, tables[name])
        return BoundaryCondition(bc.classification, q)
    end
    return FieldBoundaryConditions(conds...)
end

"Wrap an ob200_field as the OffsetArray `data` of a Field (same axes as Grids/new_data.jl:56-61 gives on CPU)."
function wrap_field(FT, grid, loc, fh::Ptr{Cvoid}, owner)
    sz = Ref{NTuple{3,Int32}}()
    check(ccall((:ob200_field_parent_size, lib), Int32, (Ptr{Cvoid}, Ref{NTuple{3,Int32}}), fh, sz))
    a = B200Array{FT, 3}(C_NULL, fh, Int.(sz[]), owner)
    return offset_data(a, grid, loc)
end
function new_data(FT::DataType, grid::B200Grid, loc, indices=(:, :, :))
    fh = Ref{Ptr{Cvoid}}()
    check(ccall((:ob200_field_create, lib), Int32, (Ptr{Cvoid}, Ref{NTuple{3,Int32}}, Ptr{BC}, Ref{Ptr{Cvoid}}),
                grid_handle(grid), loc_code.(loc), C_NULL, fh))
    data = wrap_field(FT, grid, loc, fh[], grid)
    finalizer(a -> ccall((:ob200_field_destroy, lib), Int32, (Ptr{Cvoid},), a.field), parent(data))
    return data
end
field_handle(f::Field) = parent(f.data).field

# set!(field, f::Function / array / number) (Fields/set!.jl:20-65): as on GPU(), the values are generated on a CPU twin of the
# field and copied; the copy is ob200_field_set_parent (parent layout -> internal layout conversion on the device)
function set!(u::Field{<:Any,<:Any,<:Any,<:Any,<:B200Grid}, v::Union{Function, AbstractArray, Number})
    cpu_grid = Oceananigans.Grids.on_architecture(CPU(), u.grid)
    u_cpu = Field(location(u), cpu_grid; boundary_conditions = u.boundary_conditions)
    set!(u_cpu, v isa B200Array ? Array(v) : v)
    copyto!(parent(u.data), parent(u_cpu.data))
    return u
end

# fill_halo_regions!(fields) BoundaryConditions/fill_halo_regions.jl:34-82.  The boundary conditions live in the library
# field (given at creation for model fields; default for others).
const B200Field = Field{<:Any,<:Any,<:Any,<:Any,<:B200Grid}
fill_halo_regions!(f::B200Field, args...; kw...) = fill_halo_regions!((f,), args...; kw...)
function fill_halo_regions!(fields::Union{Tuple{Vararg{B200Field}}, NamedTuple{<:Any,<:Tuple{Vararg{B200Field}}}}, args...; kw...)
    hs = Ptr{Cvoid}[field_handle(f) for f in fields]
    GC.@preserve hs check(ccall((:ob200_fill_halo_regions, lib), Int32, (Ptr{Ptr{Cvoid}}, Int32), hs, length(hs)))
    return nothing
end

# ---- solvers (Solvers/fft_based_poisson_solver.jl:93-125, fourier_tridiagonal_poisson_solver.jl:74-101,
#      batched_tridiagonal_solver.jl:74-122) ------------------------------------------------------------------------
"The pressure solver of a B200 model: a handle; the plan, the eigenvalues and the storage live in the library."
struct B200PoissonSolver{G}
    grid   :: G
    handle :: Ptr{Cvoid}
    kind   :: Symbol          # :fft or :fourier_tridiagonal
end
function B200PoissonSolver(grid, kind::Symbol=:auto)
    h = Ref{Ptr{Cvoid}}()
    code = kind === :fft ? 1 : kind === :fourier_tridiagonal ? 2 : 0
    check(ccall((:ob200_poisson_create, lib), Int32, (Ptr{Cvoid}, Int32, Ref{Ptr{Cvoid}}), grid_handle(grid), code, h))
    regular = all(x -> x isa Number, (grid.Δxᶜᵃᵃ, grid.Δyᵃᶜᵃ, grid.Δzᵃᵃᶜ))
    return B200PoissonSolver(grid, h[], kind === :auto ? (regular ? :fft : :fourier_tridiagonal) : kind)
end
PressureSolver(::B200, grid::RectilinearGrid) = B200PoissonSolver(grid)                     # NonhydrostaticModels.jl:18-27
FFTBasedPoissonSolver(grid::B200Grid, planner_flag=nothing) = B200PoissonSolver(grid, :fft)
FourierTridiagonalPoissonSolver(grid::B200Grid, planner_flag=nothing) = B200PoissonSolver(grid, :fourier_tridiagonal)

"solve!(ϕ, solver, rhs): rhs is a real (or complex with zero imaginary part) Nx x Ny x Nz array, host or device."
function solve!(ϕ::B200Field, solver::B200PoissonSolver, rhs)
    FT = eltype(solver.grid)
    r = Array{FT, 3}(real.(rhs isa B200Array ? Array(rhs) : rhs))
    GC.@preserve r check(ccall((:ob200_poisson_solve, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
                               solver.handle, field_handle(ϕ), r))
    return ϕ
end
function solve_for_pressure!(pressure::B200Field, solver::B200PoissonSolver, Δt, U★)         # solve_for_pressure.jl:55-89
    check(ccall((:ob200_solve_for_pressure, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Float64, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
                solver.handle, field_handle(pressure), Δt, field_handle(U★.u), field_handle(U★.v), field_handle(U★.w)))
    return nothing
end
"solve!(ϕ, ::BatchedTridiagonalSolver, rhs) for host arrays (the solver's own arrays may be functions of (i,j,k) on CPU only)."
function solve!(ϕ::Array{T,3}, solver::BatchedTridiagonalSolver{<:Any,<:Any,<:Any,<:Any,<:B200Grid}, rhs::Array{T,3}) where T
    Nx, Ny, Nz = size(solver.grid)
    a, c = Float64.(solver.a), Float64.(solver.c)
    b = Float64.(solver.b isa AbstractArray ? solver.b : [solver.b(i, j, k, solver.grid, solver.parameters...) for i=1:Nx, j=1:Ny, k=1:Nz])
    FTc = real(T) == Float32 ? Int32(0) : Int32(1)
    GC.@preserve a b c rhs ϕ check(ccall((:ob200_batched_tridiagonal_solve, lib), Int32,
        (Int32, Int32, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cvoid}, Ptr{Cvoid}),
        FTc, T <: Complex, Nx, Ny, Nz, a, b, c, rhs, ϕ))
    return ϕ
end

# ---- model: nonhydrostatic_model.jl:102-203 --------------------------------------------------------------------------
adv_code(::Nothing) = 0; adv_code(::CenteredSecondOrder) = 1; adv_code(::CenteredFourthOrder) = 2
adv_code(::UpwindBiasedFirstOrder) = 3; adv_code(::UpwindBiasedThirdOrder) = 4; adv_code(::UpwindBiasedFifthOrder) = 5
adv_code(::WENO5) = 6
adv_code(a) = throw(ArgumentError("B200(): unsupported advection scheme $(typeof(a))"))

closure_desc(::Nothing, tracers) = (0, 0.0, ntuple(_ -> 0.0, MAX_TRACERS))
# ScalarDiffusivity with either time discretisation (VerticallyImplicit: ThreeDimensional / Vertical formulation on a Bounded z;
# the library runs the tridiagonal solves itself, so the time stepper's `implicit_solver` stays `nothing`)
vertically_implicit(::ScalarDiffusivity{<:VerticallyImplicitTimeDiscretization}) = Int32(1)
vertically_implicit(::Any) = Int32(0)
function closure_desc(c::ScalarDiffusivity{<:Any, F}, tracers) where F
    (c.ν isa Number && all(κ -> κ isa Number, values(c.κ))) ||
        throw(ArgumentError("B200(): ScalarDiffusivity with constant ν and κ only"))
    code = F <: ThreeDimensionalFormulation ? 1 : F <: HorizontalFormulation ? 2 : 3
    κ = ntuple(t -> t <= length(tracers) ? Float64(c.κ[tracers[t]]) : 0.0, MAX_TRACERS)
    return (code, Float64(c.ν), κ)
end
# SmagorinskyLilly (smagorinsky_lilly.jl:6-72): code 4, C / Cb and the Prandtl numbers travel in their own descriptor fields
closure_desc(c::SmagorinskyLilly{<:ExplicitTimeDiscretization}, tracers) = (4, 0.0, ntuple(_ -> 0.0, MAX_TRACERS))
smagorinsky_desc(c::SmagorinskyLilly, tracers) =
    (Float64(c.C), Float64(c.Cb), ntuple(t -> t <= length(tracers) ? Float64(c.Pr isa Number ? c.Pr : c.Pr[tracers[t]]) : 1.0, MAX_TRACERS))
smagorinsky_desc(c, tracers) = (0.0, 0.0, ntuple(_ -> 1.0, MAX_TRACERS))
# AnisotropicMinimumDissipation (anisotropic_minimum_dissipation.jl:96-105): code 5, constant Poincaré constants only
closure_desc(c::AnisotropicMinimumDissipation{<:ExplicitTimeDiscretization}, tracers) = (5, 0.0, ntuple(_ -> 0.0, MAX_TRACERS))
function amd_desc(c::AnisotropicMinimumDissipation, tracers)
    (c.Cν isa Number && all(x -> x isa Number, values(c.Cκ))) ||
        throw(ArgumentError("B200(): AnisotropicMinimumDissipation with constant Cν, Cκ only"))
    Cκ = ntuple(t -> t <= length(tracers) ? Float64(c.Cκ[tracers[t]]) : 0.0, MAX_TRACERS)
    return (Float64(c.Cν), Cκ, c.Cb === nothing ? 0.0 : Float64(c.Cb), Int32(c.Cb !== nothing))
end
amd_desc(c, tracers) = (0.0, ntuple(_ -> 0.0, MAX_TRACERS), 0.0, Int32(0))
closure_desc(c, tracers) = throw(ArgumentError("B200(): unsupported closure $(typeof(c)) (tuples of closures, function-valued coefficients " *
                                               "and vertically implicit diffusion are outside the B200 path)"))

"The ENO coefficient tables of WENO5(grid=grid) for stretched dimensions (weno_fifth_order.jl:562-584): [dim][Face, Center]."
function weno_tables(a::WENO5)
    tabs = (a.coeff_xᶠᵃᵃ, a.coeff_xᶜᵃᵃ, a.coeff_yᵃᶠᵃ, a.coeff_yᵃᶜᵃ, a.coeff_zᵃᵃᶠ, a.coeff_zᵃᵃᶜ)
    # each table: 4 stencil shifts (r = -1, 0, 1, 2) of OffsetVector{NTuple{3}} -> flat Float64 [4][N+2][3]
    flat(t) = t === nothing ? Float64[] : Float64[t[r][i][q] for q in 1:3, i in eachindex(t[1]), r in 1:4][:]
    return map(flat, tabs)
end
weno_tables(::Any) = ntuple(_ -> Float64[], 6)

# ---- forcing: Relaxation(; rate, mask, target) (Forcings/relaxation.jl) tabulated at the forced field's nodes ----------------
# the types of the defaults mask = onefunction, target = zerofunction, taken from the constructor itself
const OneFunction = typeof(Relaxation(rate = 1).mask)
const ZeroFunction = typeof(Relaxation(rate = 1).target)
const SupportedRelaxation = Relaxation{<:Number, <:Union{OneFunction, GaussianMask}, <:Union{Number, ZeroFunction, LinearTarget}}
dim_code(::GaussianMask{D}) where D = D === :x ? 0 : D === :y ? 1 : 2
dim_code(::LinearTarget{D}) where D = D === :x ? 0 : D === :y ? 1 : 2
function forcing_nodes(grid, loc, d, what)
    topology(grid, d + 1) === Flat && throw(ArgumentError("B200(): Relaxation $what along the Flat dimension $("xyz"[d + 1])"))
    ξ = (xnodes, ynodes, znodes)[d + 1](loc[d + 1](), grid)
    return ξ
end
"(active, mask_dim, rate, mask table, target_dim, target value, target table) of one Relaxation at location `loc`"
function relaxation_tables(r::SupportedRelaxation, grid, loc)
    node(d, ξ) = ntuple(q -> q == d + 1 ? ξ : zero(ξ), 3)
    md, M = -1, Float64[]
    if r.mask isa GaussianMask
        md = dim_code(r.mask)
        M = Float64[r.rate * r.mask(node(md, ξ)...) for ξ in forcing_nodes(grid, loc, md, "mask")]     # rate * mask first
    end
    td, T, tv = -1, Float64[], r.target isa Number ? Float64(r.target) : 0.0
    if r.target isa LinearTarget
        td = dim_code(r.target)
        T = Float64[r.target(node(td, ξ)..., 0) for ξ in forcing_nodes(grid, loc, td, "target")]
    end
    return md, Float64(r.rate), M, td, tv, T
end
relaxation_tables(f, grid, loc) =
    throw(ArgumentError("B200(): only Relaxation(; rate::Number, mask = onefunction | GaussianMask, target = Number | " *
                        "zerofunction | LinearTarget) forcings cross the C ABI; got $(typeof(f))"))

function forcing_desc(forcing, grid, names)
    for n in keys(forcing)
        n in names || throw(ArgumentError("forcing name $n is not one of the model's fields $names"))   # model_forcing.jl
    end
    locs = (u = (Face, Center, Center), v = (Center, Face, Center), w = (Center, Center, Face))
    keep = Vector{Float64}[]
    none = ForcingDesc(0, -1, 0.0, C_NULL, -1, 0.0, C_NULL)
    descs = ntuple(3 + MAX_TRACERS) do q
        q <= length(names) && haskey(forcing, names[q]) || return none
        n = names[q]
        md, rate, M, td, tv, T = relaxation_tables(forcing[n], grid, haskey(locs, n) ? locs[n] : (Center, Center, Center))
        push!(keep, M, T)
        ForcingDesc(1, md, rate, isempty(M) ? C_NULL : pointer(M), td, tv, isempty(T) ? C_NULL : pointer(T))
    end
    return descs, keep
end

# ---- background_fields (Models/NonhydrostaticModels/background_fields.jl) tabulated over each field's parent ----------------
# The reference's own regularize_background_field builds the FunctionField (a function, or a BackgroundField with parameters) on
# the CPU twin of the grid; its value at every parent index, halos included, crosses the ABI as a parent array of the grid's float
# type.  Sampled once, at the clock time of construction: a time-dependent background is advanced by the caller through the model
# field "bg_<name>", wrapped as `model.auxiliary_fields.b200_background_fields.<name>` (set! on it writes the parent).
const bg_regularize = Oceananigans.Models.NonhydrostaticModels.regularize_background_field
function background_table(bf, grid, loc, clock)
    cpu_grid = Oceananigans.Grids.on_architecture(CPU(), grid)
    f = bf isa Oceananigans.Fields.AbstractField ? bf :
        (bf isa Function || bf isa Oceananigans.Models.NonhydrostaticModels.BackgroundField) ?
        bg_regularize(loc..., bf, cpu_grid, clock) :
        throw(ArgumentError("B200(): a background field must be a function, a BackgroundField or a field; got $(typeof(bf))"))
    FT = eltype(grid)
    ranges = ntuple(3) do d
        N, H = size(grid, d), halo_size(grid)[d]
        topology(grid, d) === Flat ? (1:1) : ((1 - H):(N + H + (loc[d] === Face && topology(grid, d) === Bounded ? 1 : 0)))
    end
    return FT[f[i, j, k] for i in ranges[1], j in ranges[2], k in ranges[3]]
end
function background_desc(background_fields, grid, names, clock)
    for n in keys(background_fields)
        n in names || throw(ArgumentError("background field name $n is not one of the model's fields $names"))
    end
    locs = (u = (Face, Center, Center), v = (Center, Face, Center), w = (Center, Center, Face))
    tabs = Dict(n => background_table(background_fields[n], grid, haskey(locs, n) ? locs[n] : (Center, Center, Center), clock)
                for n in keys(background_fields))
    ptrs = ntuple(3 + MAX_TRACERS) do q
        q <= length(names) && haskey(tabs, names[q]) ? Ptr{Cvoid}(pointer(tabs[names[q]])) : Ptr{Cvoid}(C_NULL)
    end
    return ptrs, collect(values(tabs))
end

"Translate the model configuration into ob200_model_desc; everything outside the supported set is an ArgumentError."
function model_desc(grid, gh; advection, buoyancy, coriolis, closure, tracers, timestepper, boundary_conditions, χ = 0.1,
                    stokes_drift = nothing, forcing = NamedTuple(), background_fields = NamedTuple(), particles = nothing,
                    immersed_boundary = nothing, clock = Clock{eltype(grid)}(0, 0, 1))
    isnothing(stokes_drift) && isnothing(particles) && isnothing(immersed_boundary) ||
        throw(ArgumentError("B200(): stokes_drift, particles and immersed boundaries are not supported"))
    length(tracers) <= MAX_TRACERS || throw(ArgumentError("B200(): at most $MAX_TRACERS tracers"))
    ts = timestepper === :RungeKutta3 ? 1 : timestepper === :QuasiAdamsBashforth2 ? 0 :
         throw(ArgumentError("B200(): timestepper must be :RungeKutta3 or :QuasiAdamsBashforth2"))
    clo, ν, κ = closure_desc(closure, tracers)
    fplane, f = coriolis === nothing ? (0, 0.0) : coriolis isa FPlane ? (1, Float64(coriolis.f)) :
                throw(ArgumentError("B200(): coriolis must be nothing or FPlane"))
    btr, tilted, ĝ = -1, 0, (0.0, 0.0, 1.0)
    bkind, iT, iS, grav, α, β = 0, -1, -1, 0.0, 0.0, 0.0
    if buoyancy !== nothing
        bm = buoyancy.model
        if bm isa BuoyancyTracer
            btr = findfirst(==(:b), tracers) - 1
        elseif bm isa SeawaterBuoyancy{<:Any, <:LinearEquationOfState}      # linear_equation_of_state.jl:69-77
            bkind = 1
            req = required_tracers(bm)
            iT = :T in req ? findfirst(==(:T), tracers) - 1 : -1
            iS = :S in req ? findfirst(==(:S), tracers) - 1 : -1
            grav = Float64(bm.gravitational_acceleration)
            α, β = Float64(bm.equation_of_state.thermal_expansion), Float64(bm.equation_of_state.haline_contraction)
        else
            throw(ArgumentError("B200(): buoyancy must be nothing, BuoyancyTracer() or SeawaterBuoyancy with LinearEquationOfState"))
        end
        if !(buoyancy.gravity_unit_vector isa ZDirection)
            tilted = 1; ĝ = Float64.(Tuple(buoyancy.gravity_unit_vector))
        end
    end
    tabs = weno_tables(advection)
    names = (:u, :v, :w, tracers...)
    bcs = ntuple(6 * (3 + MAX_TRACERS)) do q
        fidx, side = divrem(q - 1, 6)
        fidx < length(names) ? bc_codes(boundary_conditions[names[fidx + 1]])[side + 1] : BC(0, 0.0)
    end
    frc, frc_tabs = forcing_desc(forcing, grid, names)
    bg, bg_tabs = background_desc(background_fields, grid, names, clock)
    ptr(v) = isempty(v) ? Ptr{Float64}(C_NULL) : pointer(v)
    desc = ModelDesc(gh, ts, χ, adv_code(advection), advection isa WENO5 ? Int32(advection.zweno) : Int32(1),
                     map(ptr, tabs), clo, ν, κ, fplane, f, btr, tilted, ĝ, length(tracers), bcs, 0,
                     bkind, iT, iS, grav, α, β, smagorinsky_desc(closure, tracers)..., amd_desc(closure, tracers)...,
                     vertically_implicit(closure), frc, bg)
    # the tables must be GC.@preserve'd across ob200_model_create (host pointers are borrowed)
    return desc, (tabs, frc_tabs, bg_tabs)
end

model_field(mh, name) = (h = Ref{Ptr{Cvoid}}(); check(ccall((:ob200_model_field, lib), Int32,
                         (Ptr{Cvoid}, Cstring, Ref{Ptr{Cvoid}}), mh, name, h)); h[])

mutable struct ModelHandle
    ptr :: Ptr{Cvoid}
end

"""
    b200_nonhydrostatic_model(; grid, kw...)

Called by the first line of the reference constructor when `architecture(grid) isa B200` (INTEGRATION.md, hook 2).
Creates the library model, wraps ITS fields (state, tendencies, pressures) as Oceananigans `Field`s with the regularised
boundary conditions, and hands them to the reference's own constructor through its `velocities`, `tracers`, `pressures`,
`timestepper` and `pressure_solver` keywords, so that everything downstream (Simulation, output writers, diagnostics,
`set!`, `model.velocities.u` ...) sees an ordinary NonhydrostaticModel.
"""
function b200_nonhydrostatic_model(; grid, clock = Clock{eltype(grid)}(0, 0, 1), advection = CenteredSecondOrder(),
                                   buoyancy = nothing, coriolis = nothing, closure = nothing,
                                   boundary_conditions::NamedTuple = NamedTuple(), tracers = (),
                                   timestepper = :QuasiAdamsBashforth2, auxiliary_fields = NamedTuple(), kw...)
    FT = eltype(grid)
    tracers = tupleit(tracers)
    # halo inflation exactly as nonhydrostatic_model.jl:140-148 (the library refuses too small a halo)
    Hreq = Oceananigans.Models.NonhydrostaticModels.inflate_halo_size(halo_size(grid)..., topology(grid), advection, closure)
    any(halo_size(grid) .< Hreq) && (grid = with_halo(Hreq, grid))
    names = (:u, :v, :w, tracers...)
    default_bcs = NamedTuple{names}(FieldBoundaryConditions() for _ in names)
    bcs = regularize_field_boundary_conditions(merge(default_bcs, boundary_conditions), grid, names)
    buoyancy = Oceananigans.BuoyancyModels.regularize_buoyancy(buoyancy)
    locs = (u = (Face, Center, Center), v = (Center, Face, Center), w = (Center, Center, Face))
    loc_of(n) = haskey(locs, n) ? locs[n] : (Center, Center, Center)
    # array boundary conditions: checked before any library call, pushed once the model exists
    tables = Dict(n => Dict(s => t for s in SIDES for t in (boundary_table(getfield(bcs[n], s), s, grid, loc_of(n)),)
                            if t !== nothing) for n in names)
    gh = grid_handle(grid)
    desc, keep = model_desc(grid, gh; advection, buoyancy, coriolis, closure, tracers, timestepper,
                            boundary_conditions = bcs, clock, kw...)
    mh = Ref{Ptr{Cvoid}}()
    GC.@preserve keep check(ccall((:ob200_model_create, lib), Int32, (Ref{ModelDesc}, Ref{Ptr{Cvoid}}), desc, mh))
    handle = ModelHandle(mh[])
    finalizer(h -> ccall((:ob200_model_destroy, lib), Int32, (Ptr{Cvoid},), h.ptr), handle)

    libname(n) = n in (:u, :v, :w) ? String(n) : "c$(findfirst(==(n), tracers) - 1)"
    bcs = NamedTuple{names}(attach_boundary_arrays(bcs[n], tables[n], model_field(mh[], libname(n)), handle) for n in names)
    wrap(n, prefix = "", fbcs = bcs[n]) = Field(loc_of(n), grid; boundary_conditions = fbcs,
                                                data = wrap_field(FT, grid, loc_of(n), model_field(mh[], prefix * libname(n)), handle))
    velocities = NamedTuple{(:u, :v, :w)}(wrap(n) for n in (:u, :v, :w))
    tracer_fields = NamedTuple{tracers}(wrap(n) for n in tracers)
    ccc = (Center, Center, Center)
    pfield(name) = Field(ccc, grid; data = wrap_field(FT, grid, ccc, model_field(mh[], name), handle))
    pressures = (pNHS = pfield("pNHS"), pHY′ = topology(grid, 3) === Flat ? nothing : pfield("pHY"))
    G(prefix) = NamedTuple{names}(wrap(n, prefix, FieldBoundaryConditions(grid, loc_of(n))) for n in names)
    ts = timestepper === :RungeKutta3 ? RungeKutta3TimeStepper(grid, tracers; Gⁿ = G("Gn_"), G⁻ = G("Gm_")) :
                                        QuasiAdamsBashforth2TimeStepper(grid, tracers; Gⁿ = G("Gn_"), G⁻ = G("Gm_"))
    # diffusivity_fields.νₑ of SmagorinskyLilly is the library's "nu_e" field (κₑ stays the reference's lazy νₑ / Pr operation)
    diffusivity_fields = closure isa AnisotropicMinimumDissipation ?
        (; νₑ = pfield("nu_e"), κₑ = NamedTuple{tracers}(Tuple(pfield("kappa_e$(t - 1)") for t in 1:length(tracers)))) :
        closure isa SmagorinskyLilly ?
        (; νₑ = pfield("nu_e"), κₑ = NamedTuple{tracers}(Tuple(pfield("nu_e") / (closure.Pr isa Number ? closure.Pr : closure.Pr[n]) for n in tracers))) : nothing
    # the library's background fields "bg_<name>": writing their parent (set!, copyto!) replaces the values from the next step on
    bgnames = Tuple(n for n in names if haskey(get(kw, :background_fields, NamedTuple()), n))
    background_fields = NamedTuple{bgnames}(wrap(n, "bg_", FieldBoundaryConditions(grid, loc_of(n))) for n in bgnames)
    solver = B200PoissonSolver(grid)
    return Oceananigans.Models.NonhydrostaticModels.reference_nonhydrostatic_model(;      # the unchanged constructor body (hook 2)
        grid, clock, advection, buoyancy, coriolis, closure, boundary_conditions = bcs, tracers = tracer_fields,
        timestepper = ts, velocities, pressures, diffusivity_fields, pressure_solver = solver,
        auxiliary_fields = merge(auxiliary_fields, (; b200_handle = handle, b200_background_fields = background_fields)))
end

const B200Model = NonhydrostaticModel{<:Any, <:Any, <:B200}
handle(model::B200Model) = model.auxiliary_fields.b200_handle.ptr

# TimeSteppers/runge_kutta_3.jl:81-152, quasi_adams_bashforth_2.jl:70-104: one library call enqueues the whole step (no host
# synchronisation); the clock is mirrored back so that Simulation callbacks / stop criteria see it
function time_step!(model::B200Model, Δt; euler=false)
    Δt == 0 && @warn "Δt == 0 may cause model blowup!"
    check(ccall((:ob200_model_time_step, lib), Int32, (Ptr{Cvoid}, Float64, Int32), handle(model), Δt, euler))
    t, it = Ref{Float64}(), Ref{Int64}()
    ccall((:ob200_model_clock, lib), Int32, (Ptr{Cvoid}, Ref{Float64}, Ref{Int64}), handle(model), t, it)
    model.clock.time = t[]; model.clock.iteration = it[]
    return nothing
end
update_state!(model::B200Model, callbacks=[]) =
    check(ccall((:ob200_model_update_state, lib), Int32, (Ptr{Cvoid},), handle(model)))
calculate_tendencies!(model::B200Model, callbacks=[]) =
    check(ccall((:ob200_model_calculate_tendencies, lib), Int32, (Ptr{Cvoid},), handle(model)))
# calculate_pressure_correction! + pressure_correct_velocities! are one library call; the second is a no-op
calculate_pressure_correction!(model::B200Model, Δt) =
    check(ccall((:ob200_model_pressure_project, lib), Int32, (Ptr{Cvoid}, Float64), handle(model), Δt))
pressure_correct_velocities!(::B200Model, Δt) = nothing
store_tendencies!(::B200Model) = nothing            # pointer swap inside the library

"max |div U| and kinetic energy on the device (used by NaNChecker / TimeStepWizard-style callbacks without downloading fields)"
function diagnostics(model::B200Model)
    d, ke = Ref{Float64}(), Ref{Float64}()
    check(ccall((:ob200_model_diagnostics, lib), Int32, (Ptr{Cvoid}, Ref{Float64}, Ref{Float64}), handle(model), d, ke))
    return (max_abs_div = d[], kinetic_energy = ke[])
end
"sum, sum of squares, max |.| and NaN flag of a field's interior (Simulations/nan_checker.jl:33-52 without a download)"
function reduce_field(f::B200Field)
    s, s2, m, nan = Ref{Float64}(), Ref{Float64}(), Ref{Float64}(), Ref{Int32}()
    check(ccall((:ob200_field_reduce, lib), Int32, (Ptr{Cvoid}, Ref{Float64}, Ref{Float64}, Ref{Float64}, Ref{Int32}),
                field_handle(f), s, s2, m, nan))
    return (sum = s[], sumsq = s2[], maxabs = m[], has_nan = nan[] != 0)
end

# ---- output path: OutputWriters/fetch_output.jl:24-36 with a FieldSlicer, horizontal averages, checkpoints -----------------------
# the slice / mean is formed on the device; only it travels (download stream; ob200_sync before the host array is read)
function fetch_slice(f::B200Field, lo::NTuple{3, Int}, hi::NTuple{3, Int})
    out = Array{eltype(f.grid)}(undef, (hi .- lo .+ 1)...)
    check(ccall((:ob200_field_slice_async, lib), Int32, (Ptr{Cvoid}, Ref{NTuple{3, Int32}}, Ref{NTuple{3, Int32}}, Ptr{Cvoid}),
                field_handle(f), Int32.(lo), Int32.(hi), out))
    check(ccall((:ob200_sync, lib), Int32, ()))
    return out
end
function Oceananigans.OutputWriters.fetch_output(f::B200Field, model, slicer)
    n, H = size(f), Oceananigans.Grids.halo_size(f.grid)
    rng(r, d) = r isa Colon ? (slicer.with_halos ? (1 - H[d], n[d] + H[d]) : (1, n[d])) : r isa Int ? (r, r) : (first(r), last(r))
    b = (rng(slicer.i, 1), rng(slicer.j, 2), rng(slicer.k, 3))
    return fetch_slice(f, first.(b), last.(b))
end
function Statistics.mean(f::B200Field; dims)
    flags = ntuple(d -> Int32(d in dims), 3)
    out = Array{eltype(f.grid)}(undef, ntuple(d -> flags[d] == 1 ? 1 : size(f, d), 3)...)
    check(ccall((:ob200_field_average_async, lib), Int32, (Ptr{Cvoid}, Ref{NTuple{3, Int32}}, Ptr{Cvoid}), field_handle(f), flags, out))
    check(ccall((:ob200_sync, lib), Int32, ()))
    return out
end
# Checkpointer pickup (checkpointer.jl:201-262): after set!-ing the parents of the prognostic fields, G^n and G^- from the file
function restore_clock!(model::B200Model, time, iteration, previous_Δt)
    check(ccall((:ob200_model_set_clock, lib), Int32, (Ptr{Cvoid}, Float64, Int64, Float64), handle(model), time, iteration, previous_Δt))
    model.clock.time = time; model.clock.iteration = iteration
    return nothing
end
function previous_time_step(model::B200Model)
    dt = Ref{Float64}()
    check(ccall((:ob200_model_previous_time_step, lib), Int32, (Ptr{Cvoid}, Ref{Float64}), handle(model), dt))
    return dt[]
end

# cell_advection_timescale(model) (Utils/cell_advection_timescale.jl:4-21) without downloading the velocities: the three
# maximum(abs, parent(.)) reductions run on the device, the division by the minimum spacings stays host logic
import Oceananigans.Utils: cell_advection_timescale
function cell_advection_timescale(model::B200Model)
    m = Ref{NTuple{3, Float64}}()
    check(ccall((:ob200_model_max_abs_velocities, lib), Int32, (Ptr{Cvoid}, Ref{NTuple{3, Float64}}), handle(model), m))
    umax, vmax, wmax = m[]
    g = model.grid
    return min(Oceananigans.Grids.min_Δx(g) / umax, Oceananigans.Grids.min_Δy(g) / vmax, Oceananigans.Grids.min_Δz(g) / wmax)
end
Oceananigans.Simulations.hasnan(model::B200Model) = reduce_field(model.velocities.u).has_nan      # nan_checker.jl:33-36

# ---- several GPUs: MultiArch(B200(); ranks=(1, R, 1)) (Distributed/multi_architectures.jl:64-113) --------------------------
"Called once per process after MPI.Init, before any grid on a MultiArch{B200} is created: distributes the NCCL id with MPI."
function init_multi_arch!(arch::AbstractMultiArchitecture, MPI)
    arch.ranks[1] == 1 && arch.ranks[3] == 1 || throw(ArgumentError("B200(): slab decomposition in y only, ranks = (1, R, 1)"))
    device(arch.child_architecture)
    id = zeros(UInt8, 128)
    arch.local_rank == 0 && check(ccall((:ob200_comm_unique_id, lib), Int32, (Ptr{UInt8},), id))
    MPI.Bcast!(id, 0, arch.communicator)
    check(ccall((:ob200_comm_init, lib), Int32, (Int32, Int32, Ptr{UInt8}), arch.ranks[2], arch.local_rank, id))
    return nothing
end

export B200
end # module
