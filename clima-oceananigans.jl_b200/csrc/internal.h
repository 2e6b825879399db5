// internal.h -- host-side launcher declarations shared by the translation units.
#pragma once
#include "common.cuh"
#include <functional>
#include "physics.cuh"

namespace ob {

constexpr int MAXF = 12;   // max fields in one batched halo launch

// ---- kernels.cu ---------------------------------------------------------------------------
template <class FT>
struct HaloBatch {
    int n;
    FT* p0[MAXF];          // Julia-(0,0,0) pointers
    int loc[MAXF][3];
    int bc_kind[MAXF][6];
    FT bc_val[MAXF][6];
    const FT* bc_tab[MAXF][6];   // array condition of a Bounded side (ob200_field_set_boundary_values), null = bc_val
};
template <class FT> void launch_fill_halos(const GridD<FT>& g, const HaloBatch<FT>& hb);
// the slab-decomposed fill in two phases (kernels.cu): 0 = Periodic halos of the owned rows, 1 = neighbour exchange + Periodic
// halos of the received rows; for the overlap of phase 1 with the interior tiles of the next tendency launch
template <class FT> bool halo_overlap_supported(const GridD<FT>& g);
template <class FT> void launch_fill_halos_phase(const GridD<FT>& g, const HaloBatch<FT>& hb, int phase);
// slab-decomposed dimension d: exchange `np` boundary planes (interior extent of the other dimensions) with the ring
// neighbours through peer memory; need_lo / need_hi select which of this rank's halos are filled
template <class FT>
void launch_exchange_planes(const GridD<FT>& g, const HaloBatch<FT>& hb, int d, int np, bool need_lo, bool need_hi);
template <class FT> int single_comm_dim(const GridD<FT>& g);

// substep modes for the fused tendency kernels
enum { SUB_NONE = 0, SUB_RK3_FIRST = 1, SUB_RK3 = 2, SUB_AB2 = 3 };
template <class FT>
struct Substep {
    int mode;
    FT dt, c1, c2;         // RK3_FIRST: unew = u + c1*G (c1 = dt*γ) ; RK3: u + dt*(c1*G + c2*Gm)
                           // AB2: u + dt*(c1*G - c2*Gm)
};
template <class FT>
struct FluxBC {            // constant Flux boundary conditions of the field being stepped
    int kind[6];
    FT val[6];
};
// array Flux boundary conditions (FluxBoundaryCondition(Q), Q a 2-D array) of the Bounded dimension d, for all fields that
// have one, after the tendency kernels: G^n += Q A / V at the boundary cells (apply_flux_bcs.jl:35-160) and, with a substep,
// the new state of those cells recomputed from the old state, the final G^n and G^-
template <class FT>
struct BoundaryFluxes {
    int n;
    int comp[MAXF];                  // 0, 1, 2 = u, v, w; 3 = a tracer
    const FT* Q[MAXF][2];            // low / high side table, (N_a, N_b) column-major, null = no array there
    FT* Gn[MAXF];
    const FT* Gm[MAXF];
    const FT* psi[MAXF];             // old state
    FT* psi_new[MAXF];               // new state (unused with SUB_NONE)
    Substep<FT> ss;
};
template <class FT> void launch_boundary_fluxes(const GridD<FT>& g, int d, const BoundaryFluxes<FT>& a);
// general tendency (+ optional fused substep) for prognostic field `comp`
template <class FT>
void launch_tendency_general(const Phys<FT>& P, int comp, const FT* const U[3], const FT* psi,
                             const FT* pHY, const Buoy<FT>& b, const FluxBC<FT>& fbc, FT* Gn,
                             const FT* Gm, FT* psi_new, const Substep<FT>& ss, bool closure_only = false,
                             int background_only = 0);
// true if launch_tendency_general(..., closure_only = true) is available for this model (3-D grid)
template <class FT> bool closure_only_supported(const Phys<FT>& P);
// background_only = 1 / 2: G^n = / += - div(U_bg, ψ) - div(U, ψ_bg) alone (zero for a field without background terms), for the
// fused kernel's accumulate form; true if available for this model (3-D grid, an advection scheme)
template <class FT> bool background_only_supported(const Phys<FT>& P);
// fast path (all non-Flat dimensions periodic, regular, WENO5 uniform, no closure, optional FPlane, field not forced and
// without background terms):
// the TMA-staged kernel on 3-D grids, the direct-load kernel on 2-D grids; returns false if the configuration is not
// covered
template <class FT>
bool launch_tendency_fast(const Phys<FT>& P, int comp, const FT* const U[3], const FT* psi,
                          const FT* pHY, FT* Gn, const FT* Gm, FT* psi_new, const Substep<FT>& ss);

// tendency_fused.cu: all prognostic fields of the specialised configuration in ONE launch.  Returns how many leading
// fields (u, v, w, first tracer) it handled: 0 if the configuration is not covered, otherwise 3 + min(ntracers, 1);
// the caller steps the remaining tracers with the per-field kernels.
constexpr int FUSED_MAXF = 5;
template <class FT>
struct FusedFields {
    int nf;
    const FT* state[FUSED_MAXF];     // Julia-(0,0,0) pointers: u, v, w, tracers
    const FT* Gm[FUSED_MAXF];
    FT* Gn[FUSED_MAXF];
    FT* nw[FUSED_MAXF];              // out-of-place new state (null: tendencies only)
    const FT* pHY;
    Substep<FT> ss;
    FluxBC<FT> fbc[FUSED_MAXF];      // constant Flux boundary conditions (Bounded z variant)
    bool accumulate = false;         // G^n already holds the closure's part (launch_tendency_general closure_only): add to it
    bool gn_terms = false;           // G^n already holds precomputed terms (background pass, relaxation pass): add to it
};
// part: 0 = every tile; 1 = the tile rows whose stencils stay inside the rows this rank owns along a slab-decomposed y (they
// need no neighbour data); 2 = the remaining (boundary) tile rows.  Returns the number of fields handled, 0 = not applicable.
namespace fz {
template <class FT> int launch(const Phys<FT>& P, const FusedFields<FT>& a, int part = 0);
// 0: not applicable; 1: handles the model's closure itself (or there is none); 2: applicable if the closure's flux divergence
// is precomputed into G^n (FusedFields::accumulate)
template <class FT> int supported(const Phys<FT>& P, int nf);
}

// SmagorinskyLilly eddy viscosity over the interior (the caller fills its halos)
template <class FT>
void launch_smagorinsky(const Phys<FT>& P, const Buoy<FT>& B, const FT* u, const FT* v, const FT* w, FT* nue);

// vertically implicit diffusion step of one field, in place (scratch: a field-sized buffer for the Thomas coefficients)
template <class FT>
void launch_implicit_vertical_diffusion(const GridD<FT>& g, FT* field_p0, FT* scratch_p0, FT kappa, FT dt, bool z_face);
// AnisotropicMinimumDissipation: eddy viscosity and the tracers' eddy diffusivities over the interior
template <class FT>
void launch_amd(const Phys<FT>& P, const Buoy<FT>& B, const FT* u, const FT* v, const FT* w, FT* nue, int ntr,
                const FT* const* c, FT* const* ke);

template <class FT, class CT>
void launch_pressure_rhs(const GridD<FT>& g, const FT* u, const FT* v, const FT* w, FT dt,
                         bool times_dz, CT* rhs);
// periodic_wrap (only if periodic_wrap_supported(g): all non-Flat dimensions Periodic and regular): operands are
// read with periodic wrap-around instead of from halos, so the fills that precede these kernels in the reference
// can be merged into one fill at the end of the stage
template <class FT> bool periodic_wrap_supported(const GridD<FT>& g);
template <class FT>
void launch_pressure_correct(const GridD<FT>& g, FT* u, FT* v, FT* w, const FT* p, FT dt, bool periodic_wrap);
template <class FT>
void launch_hydrostatic_pressure(const GridD<FT>& g, const Buoy<FT>& b, FT gz, FT* pHY, bool periodic_wrap);
template <class FT>
void launch_to_internal(const GridD<FT>& g, const int psize[3], const int loc[3], const FT* parent, FT* base);
template <class FT>
void launch_from_internal(const GridD<FT>& g, const int psize[3], const int loc[3], const FT* base, FT* parent);
// reductions over Julia box [1..n0]x[1..n1]x[1..n2]; out (device, 4 doubles): sum, sumsq, maxabs, nan
template <class FT>
void launch_reduce(const GridD<FT>& g, const FT* p0, const int n[3], double* out4);
// same over the Julia box [lo, lo + n) (e.g. the whole parent array, halos included)
template <class FT>
void launch_reduce_box(const GridD<FT>& g, const FT* p0, const int lo[3], const int n[3], double* out4);
// output path: dense copy of an index box (Julia indices lo .. lo + n - 1, halos allowed) / mean over the flagged dimensions
// of the interior box n; p0 = the field's Julia-(0,0,0) pointer
template <class FT> void launch_slice(const GridD<FT>& g, const FT* p0, const int lo[3], const int n[3], FT* out);
template <class FT> void launch_average(const GridD<FT>& g, const FT* p0, const int n[3], const int dims[3], FT* out);
template <class FT>
void launch_max_divergence(const GridD<FT>& g, const FT* u, const FT* v, const FT* w, double* out4);

// ---- fft.cu ---------------------------------------------------------------------------------
template <class FT>
struct PoissonPlan;      // opaque
template <class FT> PoissonPlan<FT>* poisson_plan_create(const GridD<FT>& g, int kind,
                                                         const double* dzF_host, const double* dzC_host);
template <class FT> void poisson_plan_destroy(PoissonPlan<FT>* p);
template <class FT> void* poisson_storage(PoissonPlan<FT>* p);          // complex Nx*Ny*Nz (device)
template <class FT> int poisson_kind(PoissonPlan<FT>* p);
// solve with the rhs already in storage; writes the real solution into phi (internal layout)
template <class FT> void poisson_solve(PoissonPlan<FT>* p, const GridD<FT>& g, FT* phi_p0);
// ---- fft_fast.cu: half-spectrum / register-radix fast path (Periodic power-of-two dims) ---------
namespace ff {
template <class FT> struct FastPoisson;
template <class FT> bool fast_poisson_supported(const GridD<FT>& g);
// Fourier-tridiagonal variant (Bounded z solved by a Thomas sweep on the half spectrum)
template <class FT> bool fast_ft_supported(const GridD<FT>& g);
template <class FT> void fast_poisson_set_tridiagonal(FastPoisson<FT>* p, const double* dzF_dev, const double* dzC_dev);
template <class FT> FastPoisson<FT>* fast_poisson_create(const GridD<FT>& g);
template <class FT> void fast_poisson_destroy(FastPoisson<FT>* p);
// z Bounded on a regular grid inside the FFT-based solver: the z pass (DCT, eigenvalue divide, inverse DCT on the half
// spectrum) is the caller's hook (fft.cu); info = the half spectrum [Nz][Ny][NXP] and the eigenvalue tables in its order
struct FastSpecInfo { void* spec; int NXH, NXP, Ny, Nz; const double* lamx; const double* lamy; };
template <class FT> FastSpecInfo fast_poisson_spec_info(FastPoisson<FT>* p);
template <class FT> void fast_poisson_set_zhook(FastPoisson<FT>* p, std::function<void()> hook);
template <class FT> bool fast_bounded_y_supported(const GridD<FT>& g);
template <class FT> void fast_poisson_set_yhook(FastPoisson<FT>* p, std::function<void(int)> hook, const double* lamy_dev);
// source term = div(u,v,w)/dt computed on the fly, or a real Nx*Ny*Nz device array `real_in`
template <class FT>
void fast_poisson_solve(FastPoisson<FT>* p, const GridD<FT>& g, const FT* u, const FT* v, const FT* w, FT dt,
                        const FT* real_in, FT* phi_p0);
}  // namespace ff
// true if the plan owns a fast path; then the two entry points below may be used
template <class FT> bool poisson_has_fast(PoissonPlan<FT>* p);
template <class FT>
void poisson_solve_velocities(PoissonPlan<FT>* p, const GridD<FT>& g, const FT* u, const FT* v, const FT* w,
                              FT dt, FT* phi_p0);
template <class FT>
void poisson_solve_real(PoissonPlan<FT>* p, const GridD<FT>& g, const FT* rhs_real_dev, FT* phi_p0);
template <class FT>
void batched_tridiagonal(int Nx, int Ny, int Nz, bool is_complex, const double* a_dev,
                         const double* b_dev, const double* c_dev, const void* rhs_dev,
                         void* phi_dev, FT* scratch_dev);

}  // namespace ob
