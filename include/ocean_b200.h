/*
 * ocean_b200.h -- C ABI of libocean_b200.so: the B200-native NonhydrostaticModel time step
 * behind Oceananigans' architecture dispatch (a new `B200()` next to `CPU()`/`GPU()`,
 * reference src/Architectures.jl:68-143).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, POD descriptors copied on entry.
 *   - every function returns int32 status: 0 = OK, nonzero = error; the message is
 *     retrieved with ob200_last_error() (thread-local).  No exceptions cross the boundary.
 *   - host pointers are borrowed for the duration of the call only.
 *   - device memory is owned by the handle that allocated it and released by *_destroy.
 *   - all work is enqueued on one CUDA stream per process (ob200_set_stream); entry points
 *     that return data to the host synchronise that stream, the others do not.
 *   - arrays are column-major, x fastest.  "parent" arrays have the reference's layout:
 *     (Nx+2Hx) x (Ny+2Hy) x (Nz+2Hz), +1 along a Bounded dimension for Face-located fields,
 *     extent N and halo 0 along Flat dimensions (reference src/Grids/new_data.jl:16-22,56-61).
 *     Internally fields live in a padded, sector-aligned layout; upload/download convert.
 *   - there is NO CPU fallback: every entry point fails if no CUDA device is usable.
 *
 * Each entry point cites the reference interface (path relative to /root/reference/src) it
 * replaces.  INTEGRATION.md shows the Julia `ccall` shim that binds them.
 */
#ifndef OCEAN_B200_H
#define OCEAN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OB200_VERSION 100

/* ---- enums ---------------------------------------------------------------------------- */
enum { OB200_F32 = 0, OB200_F64 = 1 };                       /* eltype(grid)                   */
enum { OB200_PERIODIC = 0, OB200_BOUNDED = 1, OB200_FLAT = 2,
       OB200_FULLY_CONNECTED = 3 };   /* Grids topology; FullyConnected = split over ranks (Distributed) */
enum { OB200_CENTER = 0, OB200_FACE = 1 };                   /* Center / Face                  */
enum { OB200_BC_NONE = 0, OB200_BC_PERIODIC = 1, OB200_BC_FLUX = 2, OB200_BC_VALUE = 3,
       OB200_BC_GRADIENT = 4, OB200_BC_OPEN = 5 };           /* BoundaryConditions classes     */
enum { OB200_ADV_NONE = 0, OB200_ADV_CENTERED2 = 1, OB200_ADV_CENTERED4 = 2, OB200_ADV_UPWIND1 = 3,
       OB200_ADV_UPWIND3 = 4, OB200_ADV_UPWIND5 = 5, OB200_ADV_WENO5 = 6 };   /* Advection      */
enum { OB200_CLOSURE_NONE = 0, OB200_CLOSURE_3D = 1, OB200_CLOSURE_HORIZONTAL = 2,
       OB200_CLOSURE_VERTICAL = 3,                           /* ScalarDiffusivity formulations */
       OB200_CLOSURE_SMAGORINSKY_LILLY = 4,                  /* SmagorinskyLilly LES closure   */
       OB200_CLOSURE_AMD = 5 };                              /* AnisotropicMinimumDissipation  */
enum { OB200_TS_AB2 = 0, OB200_TS_RK3 = 1 };                 /* :QuasiAdamsBashforth2 / :RungeKutta3 */
enum { OB200_SIDE_WEST = 0, OB200_SIDE_EAST = 1, OB200_SIDE_SOUTH = 2, OB200_SIDE_NORTH = 3,
       OB200_SIDE_BOTTOM = 4, OB200_SIDE_TOP = 5 };
enum { OB200_SOLVER_AUTO = 0, OB200_SOLVER_FFT = 1, OB200_SOLVER_FOURIER_TRIDIAGONAL = 2 };

typedef struct ob200_grid ob200_grid;
typedef struct ob200_field ob200_field;
typedef struct ob200_model ob200_model;
typedef struct ob200_poisson ob200_poisson;

/* ---- descriptors ---------------------------------------------------------------------- */

/* RectilinearGrid (Grids/rectilinear_grid.jl:1-47).  For a regular dimension `delta` is the
 * spacing already rounded to the grid's float type by the host (grid_generation.jl:83-107).
 * For a stretched dimension the host passes the reference's own metric vectors (parents of
 * the OffsetArrays grid.Δzᵃᵃᶜ / grid.Δzᵃᵃᶠ, halos included) with the Julia index of their
 * first element (grid_generation.jl:28-80).  Values are passed as double whatever `ftype`. */
typedef struct {
    int32_t ftype;
    int32_t N[3];
    int32_t H[3];
    int32_t topology[3];
    double  L[3];
    int32_t regular[3];
    double  delta[3];
    const double* dC[3];  int32_t dC_first[3]; int32_t dC_len[3];   /* Δ at centers  */
    const double* dF[3];  int32_t dF_first[3]; int32_t dF_len[3];   /* Δ at faces    */
} ob200_grid_desc;

/* One boundary condition (BoundaryConditions/boundary_condition.jl): class + constant value.
 * Function-valued conditions cannot cross a C ABI and are rejected by the shim. */
typedef struct { int32_t kind; double value; } ob200_bc;

#define OB200_MAX_TRACERS 8

/* Relaxation(; rate, mask, target) (Forcings/relaxation.jl) of one prognostic field, tabulated by the host at the field's
 * own nodes: G += M[ξ_mask] * (T[ξ_target] - ψ), M = rate * mask, added last in the tendency sum as the reference's
 * `forcings.ψ(i, j, k, grid, clock, model_fields)`.  A table along dimension d holds the values at the field's interior
 * nodes along d, Julia index 1..n (n = N[d], + 1 for a Face location on a Bounded dimension); the library rounds them to
 * the grid's float type.  A zero-initialised descriptor is "no forcing".  Function-valued forcings are rejected by the shim. */
typedef struct {
    int32_t active;                /* 0: no forcing                                                                    */
    int32_t mask_dim;              /* -1: mask = onefunction (M = rate everywhere); 0/1/2: GaussianMask{:x/:y/:z}        */
    double  rate;                  /* M where mask_dim = -1                                                            */
    const double* mask;            /* rate * mask at the field's interior nodes along mask_dim                         */
    int32_t target_dim;            /* -1: constant target (Number, zerofunction -> 0); 0/1/2: LinearTarget{:x/:y/:z}   */
    double  target_value;          /* T where target_dim = -1                                                          */
    const double* target;          /* target at the field's interior nodes along target_dim                            */
} ob200_forcing;

/* NonhydrostaticModel(; grid, advection, closure, coriolis, buoyancy, tracers, timestepper,
 * boundary_conditions) (Models/NonhydrostaticModels/nonhydrostatic_model.jl:102-203). */
typedef struct {
    const ob200_grid* grid;
    int32_t timestepper;            /* OB200_TS_*                                              */
    double  chi;                    /* AB2 χ (quasi_adams_bashforth_2.jl:6-40), default 0.1    */
    int32_t advection;              /* OB200_ADV_*                                             */
    int32_t weno_zweno;             /* WENO5(zweno=true) default (weno_fifth_order.jl:167)     */
    /* WENO5(grid=grid) ENO coefficient tables for stretched dimensions, else NULL:
     * weno_coeff[d][loc] -> 4 tables (r=-1,0,1,2) x (N[d]+2) entries (index 0..N+1) x 3 doubles
     * (weno_fifth_order.jl:562-584), loc 0 = Face table (coeff_xᶠᵃᵃ), 1 = Center table. */
    const double* weno_coeff[3][2];
    int32_t closure;                /* OB200_CLOSURE_*                                         */
    double  nu;                     /* ScalarDiffusivity ν                                     */
    double  kappa[OB200_MAX_TRACERS];
    int32_t coriolis_fplane;        /* 0 = nothing, 1 = FPlane                                 */
    double  f;
    int32_t buoyancy_tracer;        /* -1 = buoyancy nothing, else index of tracer :b          */
    int32_t gravity_tilted;         /* 0 = ZDirection, 1 = gravity_unit_vector given           */
    double  g_hat[3];
    int32_t ntracers;
    ob200_bc bcs[3 + OB200_MAX_TRACERS][6];   /* per prognostic field (u,v,w,tracers...), per side */
    int32_t pressure_solver;        /* OB200_SOLVER_AUTO picks as NonhydrostaticModels.jl:18-27 */
    /* SeawaterBuoyancy with LinearEquationOfState (BuoyancyModels/seawater_buoyancy.jl:10-73,
     * linear_equation_of_state.jl:69-77: b = g (α T - β S), g α T, or -g β S): buoyancy_kind 0 = `buoyancy_tracer`
     * above (BuoyancyTracer or nothing), 1 = seawater; temperature_tracer / salinity_tracer = tracer index,
     * -1 for a constant (inactive) one.  Nonlinear equations of state are rejected by the shim. */
    int32_t buoyancy_kind;
    int32_t temperature_tracer, salinity_tracer;
    double  gravitational_acceleration, thermal_expansion, haline_contraction;
    /* SmagorinskyLilly(C, Cb, Pr) (TurbulenceClosures/turbulence_closure_implementations/smagorinsky_lilly.jl:6-72):
     * eddy viscosity νₑ = (C Δ)² sqrt(2 Σ²) sqrt(1 - min(1, Cb N² / Σ²)) recomputed in update_state!, κₑ = νₑ / Pr per
     * tracer.  The model field "nu_e" is diffusivity_fields.νₑ. */
    double  smagorinsky_C, smagorinsky_Cb;
    double  prandtl[OB200_MAX_TRACERS];
    /* AnisotropicMinimumDissipation(Cν, Cκ, Cb) (turbulence_closure_implementations/anisotropic_minimum_dissipation.jl:96-105,
     * 180-220): constant Poincaré constants; amd_has_Cb = 0 is `Cb = nothing` (no buoyancy modification).  The model fields
     * "nu_e" and "kappa_e<k>" are diffusivity_fields.νₑ and diffusivity_fields.κₑ[k]. */
    double  amd_Cnu, amd_Ckappa[OB200_MAX_TRACERS], amd_Cb;
    int32_t amd_has_Cb;
    /* ScalarDiffusivity(VerticallyImplicitTimeDiscretization(), ...) (TurbulenceClosures/vertically_implicit_diffusion_solver.jl,
     * abstract_scalar_diffusivity_closure.jl:214-255): 1 = the z-derivative parts of the vertical fluxes are integrated
     * implicitly by a tridiagonal solve after every substep (ThreeDimensional / Vertical formulation, Bounded z only) */
    int32_t closure_vertically_implicit;
    /* forcing = (u = Relaxation(...), ...) (nonhydrostatic_model.jl:102-203, Forcings/model_forcing.jl): per prognostic
     * field u, v, w, tracers...; appended last so that every earlier member keeps its offset */
    ob200_forcing forcing[3 + OB200_MAX_TRACERS];
    /* background_fields = (u = ..., b = ...) (Models/NonhydrostaticModels/background_fields.jl): per prognostic field u, v, w,
     * tracers..., a host parent array in the reference layout (grid float type, halos included, at the field's own location)
     * holding the background at every node, or NULL for none.  The library copies it into a model-owned field ("bg_u",
     * "bg_v", "bg_w", "bg_c<k>" of ob200_model_field); ob200_field_set_parent on that field replaces the values from the next
     * step on.  Its halos are never filled.  Each tendency gains - div(U_bg, ψ) - div(U, ψ_bg) with the model's advection
     * scheme, right after the advection of ψ by U; backgrounds enter no other term.  Appended last like `forcing`. */
    const void* background[3 + OB200_MAX_TRACERS];
} ob200_model_desc;

/* ---- library / device ----------------------------------------------------------------- */
int32_t ob200_version(void);
/* Architectures.jl device(arch): select the CUDA device for this process. */
int32_t ob200_init(int32_t device);
/* All subsequent work is enqueued on `cuda_stream` (a cudaStream_t; NULL = legacy default). */
int32_t ob200_set_stream(void* cuda_stream);
int32_t ob200_sync(void);
size_t  ob200_last_error(char* buf, size_t len);
/* number of kernels launched by the library so far in this process (bench evidence) */
int64_t ob200_launch_count(void);

/* ---- raw memory: Architectures.jl array_type / arch_array / zeros / unsafe_free! -------- */
int32_t ob200_malloc(void** dev_ptr, size_t bytes);
int32_t ob200_free(void* dev_ptr);
int32_t ob200_memset(void* dev_ptr, int32_t value, size_t bytes);
int32_t ob200_upload(void* dst_dev, const void* src_host, size_t bytes);     /* arch_array(arch, a) */
int32_t ob200_download(void* dst_host, const void* src_dev, size_t bytes);   /* Array(a)            */

/* ---- grid ----------------------------------------------------------------------------- */
int32_t ob200_grid_create(const ob200_grid_desc* desc, ob200_grid** out);
int32_t ob200_grid_destroy(ob200_grid* g);

/* ---- fields: Fields/field.jl:16-31,165-194 --------------------------------------------- */
int32_t ob200_field_create(const ob200_grid* g, const int32_t loc[3], const ob200_bc bcs[6],
                           ob200_field** out);
int32_t ob200_field_destroy(ob200_field* f);
/* size(parent(field)) in the reference layout */
int32_t ob200_field_parent_size(const ob200_field* f, int32_t out[3]);
/* parent(field) .= host array  /  Array(parent(field)); element type = grid ftype */
int32_t ob200_field_set_parent(ob200_field* f, const void* host_parent);
int32_t ob200_field_get_parent(const ob200_field* f, void* host_parent);
/* same, without a final synchronisation: the DMA runs on the library's upload / download copy streams (one per
 * direction), ordered against the compute stream by events, so that the transfers of successive steps overlap the
 * kernels.  The host buffer (pinned for a truly asynchronous copy) must stay valid until ob200_sync() or, for
 * downloads, until ob200_sync_downloads() has passed the batch it belongs to. */
int32_t ob200_field_set_parent_async(ob200_field* f, const void* host_parent);
int32_t ob200_field_get_parent_async(const ob200_field* f, void* host_parent);
/* marks the downloads enqueued so far as one batch / blocks until all batches except the `keep_in_flight` most
 * recent ones have been delivered to host memory (OutputWriters/fetch_output.jl:24-36 is the synchronous analogue) */
int32_t ob200_mark_download_batch(void);
int32_t ob200_sync_downloads(int32_t keep_in_flight);
/* output path (OutputWriters/fetch_output.jl:24-36 with a FieldSlicer, OutputWriters/field_slicer.jl; AveragedField /
 * mean(field, dims = ...)): the index box lo[d]..hi[d] (Julia indices, 1-based, halo indices allowed) is gathered ON THE DEVICE
 * into a dense column-major array of hi - lo + 1, resp. the interior is averaged over the dimensions with dims[d] != 0
 * (result: column-major, averaged dimensions of extent 1; Float64 accumulation in a fixed order); only the result travels to
 * the host, on the download stream: host memory (pinned for a truly asynchronous copy) is valid after ob200_sync() or
 * ob200_sync_downloads() like ob200_field_get_parent_async */
int32_t ob200_field_slice_async(const ob200_field* f, const int32_t lo[3], const int32_t hi[3], void* host_dst);
int32_t ob200_field_average_async(const ob200_field* f, const int32_t dims[3], void* host_dst);
/* internal device storage: base pointer, index of Julia (1,1,1), strides in elements */
int32_t ob200_field_device_view(const ob200_field* f, void** base, int64_t offset111[1],
                                int64_t strides[3]);
/* fill_halo_regions!(fields) BoundaryConditions/fill_halo_regions.jl:34-82 */
int32_t ob200_fill_halo_regions(ob200_field* const* fields, int32_t n);
/* FluxBoundaryCondition(Q) / ValueBoundaryCondition(Q) / GradientBoundaryCondition(Q) with a 2-D array Q (getbc(bc, i, j, grid)
 * = bc.condition[i, j], BoundaryConditions/boundary_condition.jl): the condition of `side` becomes the array `values` (grid float
 * type, column-major, (N_a, N_b) of the grid's two tangential dimensions in x, y, z order, Flat = 1: Q[j, k] on x sides, Q[i, k]
 * on y sides, Q[i, j] on z sides), or the constant `value` again when values == NULL; kind must be Flux, Value or Gradient.
 * The field owns the device copy.  The copy is enqueued on the library stream, after every step enqueued so far, so calling
 * this between steps (model fields through ob200_model_field) varies the condition in time from the next step on.  Fails for a
 * Periodic, Flat or FullyConnected side, kind Open / None, the side normal to a Face location (u on x sides, v on y, w on z:
 * the impenetrable wall) and any grid with a FullyConnected (slab-decomposed) dimension.  Array Flux conditions of a model's
 * prognostic fields are added by one boundary-plane pass per Bounded dimension after the tendency kernels. */
int32_t ob200_field_set_boundary_values(ob200_field* f, int32_t side, const void* values);
/* device reductions over the interior (Simulations NaNChecker / wizard / diagnostics) */
int32_t ob200_field_reduce(const ob200_field* f, double* sum, double* sumsq, double* maxabs,
                           int32_t* has_nan);

/* ---- Poisson solvers: Solvers/fft_based_poisson_solver.jl, fourier_tridiagonal_poisson_solver.jl */
int32_t ob200_poisson_create(const ob200_grid* g, int32_t kind, ob200_poisson** out);
int32_t ob200_poisson_destroy(ob200_poisson* s);
/* solve!(ϕ, solver, rhs): rhs is a real host array Nx*Ny*Nz of the grid's float type
 * (the real part of solver.storage; for the Fourier-tridiagonal solver it is the source term
 * BEFORE multiplication by Δzᶜ, i.e. the argument of set_source_term!). */
int32_t ob200_poisson_solve(ob200_poisson* s, ob200_field* phi, const void* rhs_host);
/* solve_for_pressure!(pressure, solver, Δt, U★) Models/NonhydrostaticModels/solve_for_pressure.jl:55-89 */
int32_t ob200_solve_for_pressure(ob200_poisson* s, ob200_field* pressure, double dt,
                                 const ob200_field* u, const ob200_field* v, const ob200_field* w);
/* solve!(ϕ, ::BatchedTridiagonalSolver, rhs) Solvers/batched_tridiagonal_solver.jl:74-122:
 * a, c: Nz-1 doubles; b: Nx*Ny*Nz doubles; rhs/phi: Nx*Ny*Nz (complex if is_complex) host arrays
 * of the float type `ftype`. */
int32_t ob200_batched_tridiagonal_solve(int32_t ftype, int32_t is_complex, int32_t Nx, int32_t Ny,
                                        int32_t Nz, const double* a, const double* b,
                                        const double* c, const void* rhs_host, void* phi_host);

/* ---- model ---------------------------------------------------------------------------- */
int32_t ob200_model_create(const ob200_model_desc* desc, ob200_model** out);
int32_t ob200_model_destroy(ob200_model* m);
/* model.velocities.u / model.tracers.b / model.pressures.pNHS / timestepper.Gⁿ.u ...
 * names: "u","v","w","c<k>" (k-th tracer, 0-based),"pNHS","pHY","Gn_u",...,"Gm_c0","nu_e" (SmagorinskyLilly, AMD),"kappa_e<k>" (AMD),
 * "bg_u",...,"bg_c<k>" (the background of that field; an error for a field without one).
 * The returned handle is borrowed (owned by the model). */
int32_t ob200_model_field(ob200_model* m, const char* name, ob200_field** out);
/* update_state!(model) update_nonhydrostatic_model_state.jl:14-37 */
int32_t ob200_model_update_state(ob200_model* m);
/* calculate_tendencies!(model) calculate_nonhydrostatic_tendencies.jl:12-36 (Gⁿ only) */
int32_t ob200_model_calculate_tendencies(ob200_model* m);
/* calculate_pressure_correction! + pressure_correct_velocities! pressure_correction.jl:10-56;
 * with update_state!, this is the projection `set!(model; ...)` applies (set_nonhydrostatic_model.jl:51-56) */
int32_t ob200_model_pressure_project(ob200_model* m, double dt);
/* time_step!(model, Δt) TimeSteppers/runge_kutta_3.jl:81-152, quasi_adams_bashforth_2.jl:70-104.
 * `euler` forces a forward-Euler step (AB2 only).  Enqueues the whole step; does not sync. */
int32_t ob200_model_time_step(ob200_model* m, double dt, int32_t euler);
/* model.clock (TimeSteppers/clock.jl) */
int32_t ob200_model_clock(const ob200_model* m, double* time, int64_t* iteration);
int32_t ob200_model_set_clock(ob200_model* m, double time, int64_t iteration, double previous_dt);
/* the Δt of the last step (QuasiAdamsBashforth2 compares it with the next one, quasi_adams_bashforth_2.jl:76-81): saved by
 * the Checkpointer so that a restored run continues bit for bit (OutputWriters/checkpointer.jl:64-95,201-262) */
int32_t ob200_model_previous_time_step(const ob200_model* m, double* dt);
/* maximum(abs, parent(u / v / w)) in one call: the device part of cell_advection_timescale
 * (Utils/cell_advection_timescale.jl:4-21, used by TimeStepWizard Simulations/time_step_wizard.jl:78-95 and the CFL
 * diagnostics); NaN if a velocity holds a NaN (NaNChecker, Simulations/nan_checker.jl:33-52) */
int32_t ob200_model_max_abs_velocities(ob200_model* m, double out[3]);
/* max |div U| and kinetic energy 0.5*sum(u^2+v^2+w^2) over the interior (diagnostics) */
int32_t ob200_model_diagnostics(ob200_model* m, double* max_abs_div, double* kinetic_energy);

/* ---- several GPUs: MultiArch(ranks=(1,R,1)) slab decomposition in y (src/Distributed) -------------
 * One process per GPU.  Rank 0 creates the NCCL id, the host distributes it (MPI.bcast in the Julia shim,
 * torch.distributed / a file here), every rank calls ob200_comm_init BEFORE creating grids whose y topology
 * is OB200_FULLY_CONNECTED.  Such a grid describes the LOCAL slab (N[1] = Ny/R, L[1] = Ly/R); halos in y are
 * exchanged with the neighbouring ranks (halo_communication.jl:62-183) and the Poisson solver transposes
 * between y-slabs and kx-slabs with all-to-all exchanges (distributed_fft_based_poisson_solver.jl:146-196). */
int32_t ob200_comm_unique_id(char out[128]);
int32_t ob200_comm_init(int32_t nranks, int32_t rank, const char id[128]);
int32_t ob200_comm_destroy(void);
int32_t ob200_comm_allreduce(double* values, int32_t n, int32_t op);

/* ---- measurement knobs (no reference counterpart; used by bench.py and the tests) ---------- */
/* number of cached TMA tensor-map encodings (entries are evicted when the buffers they describe are freed) */
int64_t ob200_debug_cached_tensor_maps(void);
/* force the general kernels (on = 0) instead of the specialised headline kernels */
int32_t ob200_model_use_fast_kernels(ob200_model* m, int32_t on);
/* per-phase CUDA-event timing on the library stream: phases "tendency" (one event pair per
 * tendency-kernel launch), "poisson", "halo", "pressure_correct", "hydrostatic", "boundary_flux" (the array Flux pass, one pair per
 * launch, also inside "tendency") */
int32_t ob200_profile_enable(int32_t on);
int32_t ob200_profile_reset(void);
int32_t ob200_profile_query(const char* phase, double* total_ms, int64_t* count);

#ifdef __cplusplus
}
#endif
#endif /* OCEAN_B200_H */
