// physics.cuh -- pointwise operators, advection schemes, closure and tendency functions.
//
// This is the GENERAL path: every topology (Periodic/Bounded/Flat per dimension), every
// in-scope scheme and closure, regular and stretched spacings.  It follows the reference's
// operation order term by term (files cited at each function; paths relative to
// /root/reference/src).  The specialised fast kernels in tendency_fast.cuh compute the
// same quantities for the headline configuration with shared sub-expressions.
#pragma once
#include "common.cuh"
#include "weno_fast.cuh"

namespace ob {

#define OBD __device__ __forceinline__

enum { ADV_NONE = 0, ADV_C2 = 1, ADV_C4 = 2, ADV_U1 = 3, ADV_U3 = 4, ADV_U5 = 5, ADV_WENO5 = 6 };
enum { CLO_NONE = 0, CLO_3D = 1, CLO_H = 2, CLO_V = 3, CLO_SMAG = 4, CLO_AMD = 5 };
enum { SIDE_LEFT = 0, SIDE_RIGHT = 1 };

// buoyancy_perturbation(i, j, k, grid, b, C): BuoyancyTracer (buoyancy_tracer.jl:12) or SeawaterBuoyancy with the linear
// equation of state (linear_equation_of_state.jl:69-77; the reference's evaluation order is kept)
enum { BUOY_NONE = 0, BUOY_TRACER = 1, BUOY_TS = 2, BUOY_T = 3, BUOY_S = 4 };
template <class FT>
struct Buoy {
    int mode;
    const FT* T;            // the buoyancy tracer (BUOY_TRACER) or temperature
    const FT* S;            // salinity
    FT g, alpha, beta;      // g, thermal expansion, haline contraction
    FT ga, ngb;             // g * alpha, (-g) * beta
};
template <class FT>
OBD FT buoyancy_at(const Buoy<FT>& B, long long p) {
    switch (B.mode) {
        case BUOY_TRACER: return B.T[p];
        case BUOY_TS: return B.g * (B.alpha * B.T[p] - B.beta * B.S[p]);
        case BUOY_T: return B.ga * B.T[p];
        case BUOY_S: return B.ngb * B.S[p];
        default: return FT(0);
    }
}

// Relaxation(; rate, mask, target) of one prognostic field (Forcings/relaxation.jl): rate * mask and target tabulated by the
// host at the field's own nodes along one dimension each (capi.cu build_phys); md / td = -1: the constant mc / tc
template <class FT>
struct Relax {
    int on;
    int md, td;                      // dimension of the mask / target table, -1 = constant
    const FT* M;                     // rate * mask, Julia index 1..n along md
    const FT* T;                     // target, Julia index 1..n along td
    FT mc, tc;
};
// the forcing term rate * mask * (target - ψ) at Julia indices (i, j, k), ψ = the forced field there
template <class FT>
OBD FT relaxation(const Relax<FT>& r, int i, int j, int k, FT psi) {
    const FT M = r.md < 0 ? r.mc : __ldg(r.M + (r.md == 0 ? i : (r.md == 1 ? j : k)));
    const FT T = r.td < 0 ? r.tc : __ldg(r.T + (r.td == 0 ? i : (r.td == 1 ? j : k)));
    return M * (T - psi);
}

template <class FT>
struct Phys {
    GridD<FT> g;
    int scheme, zweno, buffer;       // buffer = Nᴮ of the scheme (Advection.jl:36-40)
    const FT* wc[3][2];              // stretched WENO tables [dim][0 = Face, 1 = Center] or null
    const FT* wzp[2];                // the z tables packed per (index, side) for tendency_fused.cu (capi.cu build_phys)
    int closure;
    int vitd;                        // VerticallyImplicitTimeDiscretization (ScalarDiffusivity, Bounded z): see viscous_Aflux
    FT nu, kappa[8];                 // ScalarDiffusivity constants; SmagorinskyLilly: kappa[t] = Prandtl number of tracer t
    const FT* nue;                   // SmagorinskyLilly / AMD: eddy viscosity at cell centres (Julia-(0,0,0) pointer), halos filled
    FT smagC, smagCb;
    const FT* kappae[8];             // AnisotropicMinimumDissipation: eddy diffusivity of tracer t at cell centres
    FT amdCnu, amdCk[8], amdCb;      // Poincaré constants; amdHasCb = 0: buoyancy modification off (Cb = nothing)
    int amdHasCb;
    int fplane;
    FT f;
    int btr, tilted;                 // buoyancy tracer index (-1 none); tilted gravity flag
    FT ghat[3];
    int ntr;
    Relax<FT> frc[3 + 8];            // forcing of u, v, w, tracers (on = 0: none)
    // background_fields (background_fields.jl): bg[q] = the background of prognostic field q (Julia-(0,0,0) pointer, halos
    // as given by the host, never filled) or null; bgU = the background velocities, all null without any, a missing one
    // pointing to a zeroed field (a ZeroField's fluxes are exactly zero)
    const FT* bg[3 + 8];
    const FT* bgU[3];
};

// whether field `comp` has a non-zero background term - div(U_bg, ψ) - div(U, ψ_bg)
template <class FT>
__host__ __device__ inline bool has_background(const Phys<FT>& P, int comp) {
    return P.scheme != ADV_NONE && (P.bgU[0] || P.bg[comp]);
}

struct Pt {
    long long p;   // linear offset from the Julia-(0,0,0) pointer
    int i[3];      // Julia indices
};

template <class FT>
OBD Pt sh(const GridD<FT>& g, Pt q, int d, int n) {
    q.p += n * g.st[d];
    q.i[d] += n;
    return q;
}

#ifdef OB200_STRICT
template <class FT> OBD FT div6(FT x) { return x / FT(6); }
template <class FT> OBD FT div60(FT x) { return x / FT(60); }
#else
template <class FT> OBD FT div6(FT x) { return x * FT(1.0 / 6.0); }
template <class FT> OBD FT div60(FT x) { return x * FT(1.0 / 60.0); }
#endif

// ---- Operators/difference_operators.jl:7-49, interpolation_operators.jl:20-114 ------------
template <class FT> OBD FT dC(const GridD<FT>& g, const FT* f, Pt q, int d) {   // δxᶜᵃᵃ
    return g.topo[d] == OB_FLAT ? FT(0) : f[q.p + g.st[d]] - f[q.p];
}
template <class FT> OBD FT dFc(const GridD<FT>& g, const FT* f, Pt q, int d) {  // δxᶠᵃᵃ
    return g.topo[d] == OB_FLAT ? FT(0) : f[q.p] - f[q.p - g.st[d]];
}
template <class FT> OBD FT IC(const GridD<FT>& g, const FT* f, Pt q, int d) {   // ℑxᶜᵃᵃ
    return g.topo[d] == OB_FLAT ? f[q.p] : FT(0.5) * (f[q.p] + f[q.p + g.st[d]]);
}
template <class FT> OBD FT IF(const GridD<FT>& g, const FT* f, Pt q, int d) {   // ℑxᶠᵃᵃ
    return g.topo[d] == OB_FLAT ? f[q.p] : FT(0.5) * (f[q.p - g.st[d]] + f[q.p]);
}
template <class FT> OBD FT I2(const GridD<FT>& g, const FT* f, Pt q, int d, int loc) {
    return loc == OB_C ? IC(g, f, q, d) : IF(g, f, q, d);
}
// ∂ at result location loc along d: δ / Δ (derivative_operators.jl:6-29)
template <class FT> OBD FT deriv(const GridD<FT>& g, const FT* f, Pt q, int d, int loc) {
    FT del = loc == OB_C ? dC(g, f, q, d) : dFc(g, f, q, d);
#ifndef OB200_STRICT
    if (g.regular[d]) return del * g.invd[d];       // one rounding instead of a Float64 division (~20 instructions)
    if (d == 2 && g.izC) return del * (loc == OB_F ? g.izF[q.i[2]] : g.izC[q.i[2]]);      // stretched z: tabulated reciprocals
#endif
    return del / spacing(g, d, loc, q.i[d]);
}

// ---- metrics (spacings_and_areas_and_volumes.jl:173-236) ---------------------------------
template <class FT> OBD FT areaA(const GridD<FT>& g, int d, Pt q, int lx, int ly, int lz) {
    if (d == 0) return spacing(g, 1, ly, q.i[1]) * spacing(g, 2, lz, q.i[2]);
    if (d == 1) return spacing(g, 0, lx, q.i[0]) * spacing(g, 2, lz, q.i[2]);
    return spacing(g, 0, lx, q.i[0]) * spacing(g, 1, ly, q.i[1]);
}
template <class FT> OBD FT volume(const GridD<FT>& g, Pt q, int lx, int ly, int lz) {
    return (spacing(g, 0, lx, q.i[0]) * spacing(g, 1, ly, q.i[1])) * spacing(g, 2, lz, q.i[2]);
}

// ---- centered_fourth_order.jl:17-33 ------------------------------------------------------
template <class FT> OBD FT I3(const GridD<FT>& g, const FT* c, Pt q, int d) {
    // ℑ³: c[i] - δ(δ c)(i) / 6 ; identical operation order for the ᶜ and ᶠ variants
    if (g.topo[d] == OB_FLAT) return c[q.p];
    long long s = g.st[d];
    FT c0 = c[q.p];
    return c0 - div6((c[q.p + s] - c0) - (c0 - c[q.p - s]));
}
template <class FT> OBD FT sym4(const GridD<FT>& g, const FT* c, Pt q, int d, int loc) {
    if (g.topo[d] == OB_FLAT) return c[q.p];
    if (loc == OB_C) return FT(0.5) * (I3(g, c, q, d) + I3(g, c, sh(g, q, d, 1), d));
    return FT(0.5) * (I3(g, c, sh(g, q, d, -1), d) + I3(g, c, q, d));
}

// ---- WENO5: weno_fifth_order.jl:266-272,299-317,380-403,489-532 ----------------------------
// v = psi at offsets (-3..+1) for LEFT, (-2..+2) for RIGHT relative to the face index.
// cf = 9 coefficients (p0: 3, p1: 3, p2: 3) for the three sub-stencils psi0, psi1, psi2.
template <class FT>
OBD FT weno5_core(int side, int zweno, FT a, FT b, FT c, FT d, FT e, const FT* cf) {
    // LEFT : psi2=(a,b,c) psi1=(b,c,d) psi0=(c,d,e);  RIGHT: same with the right-shifted window
    const FT c1312 = FT(13.0 / 12.0), c14 = FT(0.25);
    FT t2 = (a - 2 * b) + c, t1 = (b - 2 * c) + d, t0 = (c - 2 * d) + e;
    FT s0, s1, s2;
    FT C0, C1, C2;
    s1 = b - d;
    if (side == SIDE_LEFT) {            // :311-313
        s0 = (3 * c - 4 * d) + e;       // psi0: 3ψ1 - 4ψ2 + ψ3
        s2 = (a - 4 * b) + 3 * c;       // psi2: ψ1 - 4ψ2 + 3ψ3
        C0 = FT(3.0 / 10.0); C1 = FT(3.0 / 5.0); C2 = FT(1.0 / 10.0);
    } else {                            // :315-317 (not the mirror image; see SURVEY §7)
        s0 = (c - 4 * d) + 3 * e;       // psi0: ψ1 - 4ψ2 + 3ψ3
        s2 = (3 * a - 4 * b) + c;       // psi2: 3ψ1 - 4ψ2 + ψ3
        C0 = FT(1.0 / 10.0); C1 = FT(3.0 / 5.0); C2 = FT(3.0 / 10.0);
    }
    FT p0 = (cf[0] * c + cf[1] * d) + cf[2] * e;
    FT p1 = (cf[3] * b + cf[4] * c) + cf[5] * d;
    FT p2 = (cf[6] * a + cf[7] * b) + cf[8] * c;
#ifndef OB200_STRICT
    if constexpr (sizeof(FT) == 8) {
        // Same rational function with ONE reciprocal instead of six divisions (see weno_fast.cuh):
        // sum_k w_k p_k = (sum_k g_k p_k) / (sum_k g_k), g_k = C_k (E_k + tau^2) prod_{j != k} E_j, E_k = (beta_k + eps)^2,
        // evaluated with 4 beta and 4 eps (everything is homogeneous in beta); differences ~1e-16 relative.
        const FT k133 = FT(13.0 / 3.0), eps4 = FT(4.0e-6);
        FT B0 = fma(s0, s0, k133 * (t0 * t0)), B1 = fma(s1, s1, k133 * (t1 * t1)), B2 = fma(s2, s2, k133 * (t2 * t2));
        FT D0 = B0 + eps4, D1 = B1 + eps4, D2 = B2 + eps4;
        FT E0 = D0 * D0, E1 = D1 * D1, E2 = D2 * D2;
        FT P12 = E1 * E2, P02 = E0 * E2, P01 = E0 * E1;
        FT g0, g1, g2;
        if (zweno) {
            FT tau = B2 - B0, tt = tau * tau, PI = E0 * P12;
            g0 = C0 * fma(tt, P12, PI); g1 = C1 * fma(tt, P02, PI); g2 = C2 * fma(tt, P01, PI);
        } else {
            g0 = C0 * P12; g1 = C1 * P02; g2 = C2 * P01;
        }
        FT den = (g0 + g1) + g2;
        FT num = fma(g0, p0, fma(g1, p1, g2 * p2));
        double r0;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"((double)den));
        double er = fma(-(double)den, r0, 1.0), q0 = (double)num * r0;
        return (FT)fma(q0, fma(er, er, er), q0);
    }
#endif
    FT b0 = c1312 * (t0 * t0) + c14 * (s0 * s0);
    FT b1 = c1312 * (t1 * t1) + c14 * (s1 * s1);
    FT b2 = c1312 * (t2 * t2) + c14 * (s2 * s2);
    const FT eps = FT(1e-6);
    FT a0, a1, a2;
    if (zweno) {                        // :386-390
        FT tau = fabs(b2 - b0);
        FT q0 = tau / (b0 + eps), q1 = tau / (b1 + eps), q2 = tau / (b2 + eps);
        a0 = C0 * (1 + q0 * q0);
        a1 = C1 * (1 + q1 * q1);
        a2 = C2 * (1 + q2 * q2);
    } else {                            // :392-394
        FT d0 = b0 + eps, d1 = b1 + eps, d2 = b2 + eps;
        a0 = C0 / (d0 * d0);
        a1 = C1 / (d1 * d1);
        a2 = C2 / (d2 * d2);
    }
    FT sa = (a0 + a1) + a2;
    FT w0 = a0 / sa, w1 = a1 / sa, w2 = a2 / sa;
    return (w0 * p0 + w1 * p1) + w2 * p2;
}

template <class FT>
OBD void weno_uniform_coeffs(int side, FT* cf) {
    // coeff_left_p0..p2 :518-520 ; right = reversed (:522-524)
    if (side == SIDE_LEFT) {
        cf[0] = FT(1.0 / 3.0);  cf[1] = FT(5.0 / 6.0);  cf[2] = -FT(1.0 / 6.0);
        cf[3] = -FT(1.0 / 6.0); cf[4] = FT(5.0 / 6.0);  cf[5] = FT(1.0 / 3.0);
        cf[6] = FT(1.0 / 3.0);  cf[7] = -FT(7.0 / 6.0); cf[8] = FT(11.0 / 6.0);
    } else {
        cf[0] = FT(11.0 / 6.0); cf[1] = -FT(7.0 / 6.0); cf[2] = FT(1.0 / 3.0);
        cf[3] = FT(1.0 / 3.0);  cf[4] = FT(5.0 / 6.0);  cf[5] = -FT(1.0 / 6.0);
        cf[6] = -FT(1.0 / 6.0); cf[7] = FT(5.0 / 6.0);  cf[8] = FT(1.0 / 3.0);
    }
}

// left/right_biased_interpolate at location loc along d (raw, no boundary fallback)
template <class FT>
OBD FT biased_raw(const Phys<FT>& P, int side, const FT* psi, Pt q, int d, int loc) {
    const GridD<FT>& g = P.g;
    int idx = q.i[d];                       // table index keeps the un-shifted index (:257-263)
    if (loc == OB_C) q = sh(g, q, d, 1);    // *_xᶜᵃᵃ(i) = *_xᶠᵃᵃ(i+1)
    long long s = g.st[d];
    const FT* f = psi + q.p;
    switch (P.scheme) {
        case ADV_WENO5: {
            FT cf[9];
            const FT* tab = P.wc[d][loc == OB_F ? 0 : 1];
#ifndef OB200_STRICT
            // `side` is per-thread data (the sign of the advecting velocity): both variants below evaluate ONE
            // reconstruction with the window / coefficients selected by `side`, so a warp with mixed signs does not
            // execute the reconstruction twice
            if (tab == nullptr) {
                const bool pos = side == SIDE_LEFT;
                const FT w0 = f[-3 * s], w1 = f[-2 * s], w2 = f[-s], w3 = f[0], w4 = f[s], w5 = f[2 * s];
                return P.zweno ? wf::weno_upwind<FT, true>(pos, w0, w1, w2, w3, w4, w5)
                               : wf::weno_upwind<FT, false>(pos, w0, w1, w2, w3, w4, w5);
            }
            {
                const int n2 = g.N[d] + 2;
                const FT* t0 = tab + ((long long)(side == SIDE_LEFT ? 1 : 0) * n2 + idx) * 3;
#pragma unroll
                for (int m = 0; m < 3; ++m)
#pragma unroll
                    for (int c = 0; c < 3; ++c) cf[3 * m + c] = t0[(long long)m * n2 * 3 + c];
                const FT* w = f + (side == SIDE_LEFT ? -3 : -2) * s;
                return weno5_core(side, P.zweno, w[0], w[s], w[2 * s], w[3 * s], w[4 * s], cf);
            }
#else
            if (tab == nullptr) {
                weno_uniform_coeffs(side, cf);
            } else {                       // retrieve_coeff :526-539: table[r+2][idx]
                int n2 = g.N[d] + 2;
                int r0 = side == SIDE_LEFT ? 1 : 0;     // p0 -> r=0 (left) / r=-1 (right)
#pragma unroll
                for (int m = 0; m < 3; ++m)
#pragma unroll
                    for (int c = 0; c < 3; ++c) cf[3 * m + c] = tab[((r0 + m) * n2 + idx) * 3 + c];
            }
            if (side == SIDE_LEFT)
                return weno5_core(side, P.zweno, f[-3 * s], f[-2 * s], f[-s], f[0], f[s], cf);
            return weno5_core(side, P.zweno, f[-2 * s], f[-s], f[0], f[s], f[2 * s], cf);
#endif
        }
        case ADV_U5:                       // upwind_biased_fifth_order.jl:24-46
            if (side == SIDE_LEFT)
                return div60((((-3 * f[s] + 27 * f[0]) + 47 * f[-s]) - 13 * f[-2 * s]) + 2 * f[-3 * s]);
            return div60((((2 * f[2 * s] - 13 * f[s]) + 47 * f[0]) + 27 * f[-s]) - 3 * f[-2 * s]);
        case ADV_U3:
            if (side == SIDE_LEFT) return div6((2 * f[0] + 5 * f[-s]) - f[-2 * s]);
            return div6((-f[s] + 5 * f[0]) + 2 * f[-s]);
        default:                           // ADV_U1
            return side == SIDE_LEFT ? f[-s] : f[0];
    }
}

template <class FT>
OBD FT sym_raw(const Phys<FT>& P, const FT* c, Pt q, int d, int loc) {
    if (P.scheme == ADV_C4 || P.scheme == ADV_U5 || P.scheme == ADV_WENO5) return sym4(P.g, c, q, d, loc);
    return I2(P.g, c, q, d, loc);
}

// ---- topologically_conditional_interpolation.jl:19-80 ------------------------------------
template <class FT>
OBD FT sym_c(const Phys<FT>& P, const FT* c, Pt q, int d, int loc) {
    const GridD<FT>& g = P.g;
    FT hi = sym_raw(P, c, q, d, loc);
    if (g.topo[d] != OB_BOUNDED) return hi;
    int i = q.i[d], N = g.N[d], NB = P.buffer;
    bool out = (i > NB) && (i < N + 1 - NB);
    return out ? hi : I2(g, c, q, d, loc);
}
template <class FT>
OBD FT biased_c(const Phys<FT>& P, int side, const FT* c, Pt q, int d, int loc) {
    const GridD<FT>& g = P.g;
    if (g.topo[d] != OB_BOUNDED) return biased_raw(P, side, c, q, d, loc);
    int i = q.i[d], N = g.N[d], NB = P.buffer;
    bool out = side == SIDE_LEFT ? ((i > NB) && (i < N + 1 - (NB - 1)))
                                 : ((i > NB - 1) && (i < N + 1 - NB));
    // the reference's ifelse evaluates both branches; the halo is wide enough for the
    // high-order one everywhere it is evaluated, so we may skip it when it is not selected.
    return out ? biased_raw(P, side, c, q, d, loc) : I2(g, c, q, d, loc);
}

// upwind_biased_advective_fluxes.jl:10
template <class FT> OBD FT upwind_product(FT u, FT pl, FT pr) {
    FT au = fabs(u);
    return ((u + au) * pl + (u - au) * pr) * FT(0.5);
}

// advection OF component B BY component A, evaluated at q (momentum); all fluxes include the area
template <class FT>
OBD FT momentum_flux(const Phys<FT>& P, int A, int B, const FT* Ua, const FT* psi, Pt q) {
    const GridD<FT>& g = P.g;
    int fl[3] = {OB_C, OB_C, OB_C};
    int ul, ud;
    if (A == B) { ul = OB_C; ud = A; }
    else { fl[A] = OB_F; fl[B] = OB_F; ul = OB_F; ud = B; }
    int pl = ul;
    if (P.scheme == ADV_C2) {          // centered_second_order.jl:16-26: ℑ(A_q U) * ℑ(ψ)
        int nat[3] = {OB_C, OB_C, OB_C};
        nat[A] = OB_F;
        FT t0, t1;
        if (g.topo[ud] == OB_FLAT) {
            t0 = areaA(g, A, q, nat[0], nat[1], nat[2]) * Ua[q.p];
        } else {
            Pt q1 = ul == OB_C ? q : sh(g, q, ud, -1);
            Pt q2 = sh(g, q1, ud, 1);
            t0 = FT(0.5) * (areaA(g, A, q1, nat[0], nat[1], nat[2]) * Ua[q1.p] +
                            areaA(g, A, q2, nat[0], nat[1], nat[2]) * Ua[q2.p]);
        }
        t1 = I2(g, psi, q, A, pl);
        return t0 * t1;
    }
    FT Ar = areaA(g, A, q, fl[0], fl[1], fl[2]);
    FT ut = sym_c(P, Ua, q, ud, ul);
    if (P.scheme >= ADV_U1) {          // upwind_biased_advective_fluxes.jl:18-97
#ifdef OB200_STRICT
        FT L = biased_c(P, SIDE_LEFT, psi, q, A, pl);
        FT R = biased_c(P, SIDE_RIGHT, psi, q, A, pl);
        return Ar * upwind_product(ut, L, R);
#else
        // ((u + |u|) L + (u - |u|) R) / 2 is EXACTLY u L for u > 0 and u R otherwise (one coefficient is 0, the
        // other 2u): only the upwind side is reconstructed, chosen per thread (no divergence: `side` is data)
        return Ar * (ut * biased_c(P, ut > FT(0) ? SIDE_LEFT : SIDE_RIGHT, psi, q, A, pl));
#endif
    }
    return (Ar * ut) * sym_c(P, psi, q, A, pl);     // centered_advective_fluxes.jl:15-27
}

template <class FT>
OBD FT tracer_flux(const Phys<FT>& P, int A, const FT* Ua, const FT* c, Pt q) {
    const GridD<FT>& g = P.g;
    int fl[3] = {OB_C, OB_C, OB_C};
    fl[A] = OB_F;
    FT Ar = areaA(g, A, q, fl[0], fl[1], fl[2]);
    if (P.scheme == ADV_C2) return (Ar * Ua[q.p]) * IF(g, c, q, A);
    if (P.scheme >= ADV_U1) {          // :103-128
#ifdef OB200_STRICT
        FT L = biased_c(P, SIDE_LEFT, c, q, A, OB_F);
        FT R = biased_c(P, SIDE_RIGHT, c, q, A, OB_F);
        return Ar * upwind_product(Ua[q.p], L, R);
#else
        const FT ua = Ua[q.p];
        return Ar * (ua * biased_c(P, ua > FT(0) ? SIDE_LEFT : SIDE_RIGHT, c, q, A, OB_F));
#endif
    }
    return (Ar * Ua[q.p]) * sym_c(P, c, q, A, OB_F);
}

// div_𝐯u/v/w (momentum_advection_operators.jl:52-86), B = advected component
template <class FT>
OBD FT div_Uu(const Phys<FT>& P, int B, const FT* const* U, const FT* psi, Pt q) {
    if (P.scheme == ADV_NONE) return FT(0);
    const GridD<FT>& g = P.g;
    FT t[3];
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        if (g.topo[A] == OB_FLAT) { t[A] = FT(0); continue; }
        if (A == B)    // δ to the Face location: f(i) - f(i-1)
            t[A] = momentum_flux(P, A, B, U[A], psi, q) - momentum_flux(P, A, B, U[A], psi, sh(g, q, A, -1));
        else           // δ to the Center location: f(i+1) - f(i)
            t[A] = momentum_flux(P, A, B, U[A], psi, sh(g, q, A, 1)) - momentum_flux(P, A, B, U[A], psi, q);
    }
    int l[3] = {OB_C, OB_C, OB_C};
    l[B] = OB_F;
    return (1 / volume(g, q, l[0], l[1], l[2])) * ((t[0] + t[1]) + t[2]);
}

// div_Uc (tracer_advection_operators.jl:31-35)
template <class FT>
OBD FT div_Uc(const Phys<FT>& P, const FT* const* U, const FT* c, Pt q) {
    if (P.scheme == ADV_NONE) return FT(0);
    const GridD<FT>& g = P.g;
    FT t[3];
#pragma unroll
    for (int A = 0; A < 3; ++A) {
        if (g.topo[A] == OB_FLAT) { t[A] = FT(0); continue; }
        t[A] = tracer_flux(P, A, U[A], c, sh(g, q, A, 1)) - tracer_flux(P, A, U[A], c, q);
    }
    return (1 / volume(g, q, OB_C, OB_C, OB_C)) * ((t[0] + t[1]) + t[2]);
}

// ---- ScalarDiffusivity: closure_kernel_operators.jl:22-48, abstract_scalar_diffusivity_closure.jl:172-207
// strain rates velocity_tracer_gradients.jl:25-43 (location of the strain given by (comp, dir))
template <class FT>
OBD FT strain(const GridD<FT>& g, int comp, int dir, const FT* const* U, Pt q) {
    if (comp == dir) return deriv(g, U[comp], q, comp, OB_C);            // Σ11, Σ22, Σ33 at ccc
    // Σ_ab = 0.5 (∂_b u_a + ∂_a u_b), both derivatives to the Face location
    int a = comp < dir ? comp : dir, b = comp < dir ? dir : comp;
    return FT(0.5) * (deriv(g, U[a], q, b, OB_F) + deriv(g, U[b], q, a, OB_F));
}

template <class FT>
OBD FT div_xy(const GridD<FT>& g, const FT* const* U, Pt q) {            // div_xyᶜᶜᶜ
    FT tx = g.topo[0] == OB_FLAT ? FT(0)
          : spacing(g, 1, OB_C, q.i[1]) * U[0][q.p + g.st[0]] - spacing(g, 1, OB_C, q.i[1]) * U[0][q.p];
    FT ty = g.topo[1] == OB_FLAT ? FT(0)
          : spacing(g, 0, OB_C, q.i[0]) * U[1][q.p + g.st[1]] - spacing(g, 0, OB_C, q.i[0]) * U[1][q.p];
    return (1 / (spacing(g, 0, OB_C, q.i[0]) * spacing(g, 1, OB_C, q.i[1]))) * (tx + ty);
}
template <class FT>
OBD FT zeta3(const GridD<FT>& g, const FT* const* U, Pt q) {             // ζ₃ᶠᶠᶜ
    FT a = g.topo[0] == OB_FLAT ? FT(0)
         : spacing(g, 1, OB_F, q.i[1]) * U[1][q.p] - spacing(g, 1, OB_F, q.i[1]) * U[1][q.p - g.st[0]];
    FT b = g.topo[1] == OB_FLAT ? FT(0)
         : spacing(g, 0, OB_F, q.i[0]) * U[0][q.p] - spacing(g, 0, OB_F, q.i[0]) * U[0][q.p - g.st[1]];
    return (a - b) / (spacing(g, 0, OB_F, q.i[0]) * spacing(g, 1, OB_F, q.i[1]));
}

// νᶜᶜᶜ / νᶠᶠᶜ / νᶠᶜᶠ / νᶜᶠᶠ of a cell-centred viscosity field (closure_kernel_operators.jl:84-90): at the location of the
// (comp, dir) stress; the double interpolations are outer(inner) = higher dimension of lower dimension
// (interpolation_operators.jl:60-71)
template <class FT>
OBD FT nu_at_stress(const GridD<FT>& g, const FT* nu, int comp, int dir, Pt q) {
    if (comp == dir) return nu[q.p];
    const int a = comp < dir ? comp : dir, b = comp < dir ? dir : comp;
    if (g.topo[b] == OB_FLAT) return IF(g, nu, q, a);
    return FT(0.5) * (IF(g, nu, sh(g, q, b, -1), a) + IF(g, nu, q, a));
}

// A * viscous_flux_{comp}{dir} at q
template <class FT>
OBD FT viscous_Aflux(const Phys<FT>& P, int comp, int dir, const FT* const* U, Pt q) {
    const GridD<FT>& g = P.g;
    int fl[3] = {OB_C, OB_C, OB_C};
    if (comp != dir) { fl[comp] = OB_F; fl[dir] = OB_F; }
    FT Ar = areaA(g, dir, q, fl[0], fl[1], fl[2]);
    FT fx = FT(0);
    if (P.vitd && dir == 2 && !(q.i[2] == 1 || q.i[2] == g.N[2] + 1)) {
        // vertically implicit diffusion on a Bounded z (abstract_scalar_diffusivity_closure.jl:232-249): away from the two
        // boundary indices only the part of the z flux that has no z derivative stays explicit: -ν ∂x w (u), -ν ∂y w (v), 0 (w)
        if (comp < 2) fx = -(P.nu * deriv(g, U[2], q, comp, OB_F));
        return Ar * fx;
    }
    if (P.closure == CLO_3D) {
        fx = -2 * (P.nu * strain(g, comp, dir, U, q));
    } else if (P.closure == CLO_SMAG || P.closure == CLO_AMD) {      // viscosity(closure, K) = K.νₑ (smagorinsky_lilly.jl:23, anisotropic_minimum_dissipation.jl:24)
        fx = -2 * (nu_at_stress(g, P.nue, comp, dir, q) * strain(g, comp, dir, U, q));
    } else if (P.closure == CLO_H) {
        if (comp < 2 && comp == dir) fx = -(P.nu * div_xy(g, U, q));
        else if (comp == 1 && dir == 0) fx = -(P.nu * zeta3(g, U, q));
        else if (comp == 0 && dir == 1) fx = P.nu * zeta3(g, U, q);
        else if (comp == 2 && dir < 2) fx = -(P.nu * deriv(g, U[2], q, dir, OB_F));
    } else if (P.closure == CLO_V) {
        if (dir == 2) fx = -(P.nu * deriv(g, U[comp], q, 2, comp == 2 ? OB_C : OB_F));
    }
    return Ar * fx;
}

template <class FT>
OBD FT div_tau(const Phys<FT>& P, int comp, const FT* const* U, Pt q) {
    if (P.closure == CLO_NONE) return FT(0);
    const GridD<FT>& g = P.g;
    FT t[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        if (g.topo[d] == OB_FLAT) { t[d] = FT(0); continue; }
        if (d == comp) t[d] = viscous_Aflux(P, comp, d, U, q) - viscous_Aflux(P, comp, d, U, sh(g, q, d, -1));
        else t[d] = viscous_Aflux(P, comp, d, U, sh(g, q, d, 1)) - viscous_Aflux(P, comp, d, U, q);
    }
    int l[3] = {OB_C, OB_C, OB_C};
    l[comp] = OB_F;
    return (1 / volume(g, q, l[0], l[1], l[2])) * ((t[0] + t[1]) + t[2]);
}

// `kappa`: the constant diffusivity (ScalarDiffusivity), the Prandtl number (SmagorinskyLilly); `ke`: the tracer's eddy
// diffusivity field (AnisotropicMinimumDissipation), else null
template <class FT>
OBD FT diffusive_Aflux(const Phys<FT>& P, int d, FT kappa, const FT* c, Pt q, const FT* ke = nullptr) {
    const GridD<FT>& g = P.g;
    int fl[3] = {OB_C, OB_C, OB_C};
    fl[d] = OB_F;
    FT Ar = areaA(g, d, q, fl[0], fl[1], fl[2]);
    if (P.closure == CLO_AMD)                // diffusivity(::AMD, K, id) = K.κₑ[id], κᶠᶜᶜ = ℑxᶠᵃᵃ(κₑ) (closure_kernel_operators.jl:88-90)
        return Ar * (-IF(g, ke, q, d) * deriv(g, c, q, d, OB_F));
    if (P.closure == CLO_SMAG) {             // κₑ = νₑ / Pr at cell centres, interpolated to the face (smagorinsky_lilly.jl:205-221)
        const FT k1 = P.nue[q.p] / kappa;
        const FT kl = g.topo[d] == OB_FLAT ? k1 : FT(0.5) * (P.nue[q.p - g.st[d]] / kappa + k1);
        return Ar * (-kl * deriv(g, c, q, d, OB_F));
    }
    bool active = P.closure == CLO_3D || (P.closure == CLO_H && d < 2) || (P.closure == CLO_V && d == 2);
    // vertically implicit diffusion: the explicit z flux only at k == 1 and k == Nz + 1 (:251-255)
    if (P.vitd && d == 2 && !(q.i[2] == 1 || q.i[2] == g.N[2] + 1)) active = false;
    return active ? Ar * (-kappa * deriv(g, c, q, d, OB_F)) : Ar * FT(0);
}
template <class FT>
OBD FT div_q(const Phys<FT>& P, FT kappa, const FT* c, Pt q, const FT* ke = nullptr) {
    if (P.closure == CLO_NONE) return FT(0);
    const GridD<FT>& g = P.g;
    FT t[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        if (g.topo[d] == OB_FLAT) { t[d] = FT(0); continue; }
        t[d] = diffusive_Aflux(P, d, kappa, c, sh(g, q, d, 1), ke) - diffusive_Aflux(P, d, kappa, c, q, ke);
    }
    return (1 / volume(g, q, OB_C, OB_C, OB_C)) * ((t[0] + t[1]) + t[2]);
}

// ---- SmagorinskyLilly eddy viscosity: calc_νᶜᶜᶜ (smagorinsky_lilly.jl:83-107, 146-153) ---------------------------------
// ∂z_b at ccf (buoyancy_tracer.jl:16, seawater_buoyancy.jl:166-171, no_buoyancy.jl:9)
template <class FT>
OBD FT dz_buoyancy(const GridD<FT>& g, const Buoy<FT>& B, Pt q) {
    switch (B.mode) {
        case BUOY_TRACER: return deriv(g, B.T, q, 2, OB_F);
        case BUOY_TS: return B.g * (B.alpha * deriv(g, B.T, q, 2, OB_F) - B.beta * deriv(g, B.S, q, 2, OB_F));
        case BUOY_T: return B.g * (B.alpha * deriv(g, B.T, q, 2, OB_F) - B.beta * FT(0));
        case BUOY_S: return B.g * (B.alpha * FT(0) - B.beta * deriv(g, B.S, q, 2, OB_F));
        default: return FT(0);
    }
}
template <class FT>
OBD FT smagorinsky_nu(const Phys<FT>& P, const Buoy<FT>& B, const FT* const* U, Pt q) {
    const GridD<FT>& g = P.g;
    auto sq = [&](int a, int b, Pt r) { FT s = strain(g, a, b, U, r); return s * s; };
    // ℑ_outer ᶜ(ℑ_inner ᶜ(Σ_ab²)) with Flat dimensions the identity
    auto avg2 = [&](int a, int b) {           // a < b: inner = a, outer = b
        auto inner = [&](Pt r) { return g.topo[a] == OB_FLAT ? sq(a, b, r) : FT(0.5) * (sq(a, b, r) + sq(a, b, sh(g, r, a, 1))); };
        return g.topo[b] == OB_FLAT ? inner(q) : FT(0.5) * (inner(q) + inner(sh(g, q, b, 1)));
    };
    const FT s11 = strain(g, 0, 0, U, q), s22 = strain(g, 1, 1, U, q), s33 = strain(g, 2, 2, U, q);
    const FT tr = (s11 * s11 + s22 * s22) + s33 * s33;
    const FT S2 = ((tr + 2 * avg2(0, 1)) + 2 * avg2(0, 2)) + 2 * avg2(1, 2);
    FT N2 = FT(0);
    if (B.mode) {
        const FT a = dz_buoyancy(g, B, q);
        const FT izc = g.topo[2] == OB_FLAT ? a : FT(0.5) * (a + dz_buoyancy(g, B, sh(g, q, 2, 1)));
        N2 = izc > FT(0) ? izc : FT(0);
    }
    const FT delta = cbrt((spacing(g, 0, OB_C, q.i[0]) * spacing(g, 1, OB_C, q.i[1])) * spacing(g, 2, OB_C, q.i[2]));
    if (S2 == FT(0)) return FT(0) * ((P.smagC * delta) * (P.smagC * delta)) * sqrt(2 * S2);
    FT sf = P.smagCb * N2 / S2;
    sf = sf < FT(1) ? sf : FT(1);
    const FT stab = sqrt(FT(1) - sf);
    const FT cd = P.smagC * delta;
    return (stab * (cd * cd)) * sqrt(2 * S2);
}

// ---- AnisotropicMinimumDissipation: calc_νᶜᶜᶜ / calc_κᶜᶜᶜ (anisotropic_minimum_dissipation.jl:180-220, 269-376;
//      normalised gradients velocity_tracer_gradients.jl:120-242).  Δᶠ at ANY location is 2 Δᶜ at the index passed (:255-267).
template <class FT, class F>
OBD FT avg_c(const GridD<FT>& g, int d, Pt q, F f) {          // ℑᶜ along d of a function of the position
    return g.topo[d] == OB_FLAT ? f(q) : FT(0.5) * (f(q) + f(sh(g, q, d, 1)));
}
template <class FT, class F>
OBD FT avg_cc(const GridD<FT>& g, int inner, int outer, Pt q, F f) {      // ℑ_outer ᶜ (ℑ_inner ᶜ f)
    return avg_c(g, outer, q, [&](Pt r) { return avg_c(g, inner, r, f); });
}
template <class FT>
struct AmdGrad {            // the normalised velocity gradients as functions of the position
    const GridD<FT>& g;
    const FT* const* U;
    OBD FT df(int d, Pt r) const { return 2 * spacing(g, d, OB_C, r.i[d]); }
    OBD FT xu(Pt r) const { return deriv(g, U[0], r, 0, OB_C); }
    OBD FT yv(Pt r) const { return deriv(g, U[1], r, 1, OB_C); }
    OBD FT zw(Pt r) const { return deriv(g, U[2], r, 2, OB_C); }
    OBD FT xv(Pt r) const { return df(0, r) / df(1, r) * deriv(g, U[1], r, 0, OB_F); }
    OBD FT yu(Pt r) const { return df(1, r) / df(0, r) * deriv(g, U[0], r, 1, OB_F); }
    OBD FT xw(Pt r) const { return df(0, r) / df(2, r) * deriv(g, U[2], r, 0, OB_F); }
    OBD FT zu(Pt r) const { return df(2, r) / df(0, r) * deriv(g, U[0], r, 2, OB_F); }
    OBD FT yw(Pt r) const { return df(1, r) / df(2, r) * deriv(g, U[2], r, 1, OB_F); }
    OBD FT zv(Pt r) const { return df(2, r) / df(1, r) * deriv(g, U[1], r, 2, OB_F); }
    OBD FT s12(Pt r) const { return FT(0.5) * (yu(r) + xv(r)); }
    OBD FT s13(Pt r) const { return FT(0.5) * (zu(r) + xw(r)); }
    OBD FT s23(Pt r) const { return FT(0.5) * (zv(r) + yw(r)); }
};
template <class FT>
OBD FT amd_delta2(const GridD<FT>& g, Pt q) {
    const FT fx = 2 * spacing(g, 0, OB_C, q.i[0]), fy = 2 * spacing(g, 1, OB_C, q.i[1]), fz = 2 * spacing(g, 2, OB_C, q.i[2]);
    return 3 / ((1 / (fx * fx) + 1 / (fy * fy)) + 1 / (fz * fz));
}
template <class FT>
OBD FT amd_nu(const Phys<FT>& P, const Buoy<FT>& B, const FT* const* U, Pt q) {
    const GridD<FT>& g = P.g;
    const AmdGrad<FT> G{g, U};
    auto sq = [](FT x) { return x * x; };
#define AXY(expr) avg_cc(g, 0, 1, q, [&](Pt r) { return expr; })
#define AXZ(expr) avg_cc(g, 0, 2, q, [&](Pt r) { return expr; })
#define AYZ(expr) avg_cc(g, 1, 2, q, [&](Pt r) { return expr; })
    const FT xu = G.xu(q), yv = G.yv(q), zw = G.zw(q);
    const FT xv2 = AXY(sq(G.xv(r))), yu2 = AXY(sq(G.yu(r))), xw2 = AXZ(sq(G.xw(r))), zu2 = AXZ(sq(G.zu(r))),
             yw2 = AYZ(sq(G.yw(r))), zv2 = AYZ(sq(G.zv(r)));
    // norm_tr_∇uᶜᶜᶜ (:315-328)
    const FT qn = (((((((xu * xu + yv * yv) + zw * zw) + xv2) + yu2) + xw2) + zu2) + yw2) + zv2;
    if (qn == FT(0)) return FT(0);
    // norm_uᵢₐ_uⱼₐ_Σᵢⱼᶜᶜᶜ (:269-313), term order kept (Σ₁₁ = ∂x u etc.)
    const FT t1 = ((((xu * (xu * xu) + yv * xv2) + zw * xw2) + 2 * xu * AXY(G.xv(r) * G.s12(r))) + 2 * xu * AXZ(G.xw(r) * G.s13(r)))
                  + 2 * AXY(G.xv(r)) * AXZ(G.xw(r)) * AYZ(G.s23(r));
    const FT t2 = ((((xu * yu2 + yv * (yv * yv)) + zw * yw2) + 2 * yv * AXY(G.yu(r) * G.s12(r)))
                   + 2 * AXY(G.yu(r)) * AYZ(G.yw(r)) * AXZ(G.s13(r))) + 2 * yv * AYZ(G.yw(r) * G.s23(r));
    const FT t3 = ((((xu * zu2 + yv * zv2) + zw * (zw * zw)) + 2 * AXZ(G.zu(r)) * AYZ(G.zv(r)) * AXY(G.s12(r)))
                   + 2 * zw * AXZ(G.zu(r) * G.s13(r))) + 2 * zw * AYZ(G.zv(r) * G.s23(r));
    const FT rr = (t1 + t2) + t3;
    FT cbz = FT(0);
    if (P.amdHasCb && B.mode) {        // Cb_norm_wᵢ_bᵢᶜᶜᶜ (:332-345) / Δᶠz
        auto db = [&](int d, Pt r) {   // ∂ᶠ of buoyancy_perturbation along d at r
            const FT del = buoyancy_at(B, r.p) - buoyancy_at(B, r.p - g.st[d]);
            if (g.topo[d] == OB_FLAT) return FT(0);
#ifndef OB200_STRICT
            if (g.regular[d]) return del * g.invd[d];
#endif
            return del / spacing(g, d, OB_F, r.i[d]);
        };
        const FT wx = (AXZ(G.xw(r)) * G.df(0, q)) * avg_c(g, 0, q, [&](Pt r) { return db(0, r); });
        const FT wy = (AYZ(G.yw(r)) * G.df(1, q)) * avg_c(g, 1, q, [&](Pt r) { return db(1, r); });
        const FT wz = (zw * G.df(2, q)) * avg_c(g, 2, q, [&](Pt r) { return db(2, r); });
        cbz = P.amdCb * ((wx + wy) + wz) / G.df(2, q);
    }
    const FT nu = -P.amdCnu * amd_delta2(g, q) * (rr - cbz) / qn;
    return nu > FT(0) ? nu : FT(0);
}
template <class FT>
OBD FT amd_kappa(const Phys<FT>& P, FT Ck, const FT* const* U, const FT* c, Pt q) {
    const GridD<FT>& g = P.g;
    const AmdGrad<FT> G{g, U};
    auto cx = [&](Pt r) { return G.df(0, r) * deriv(g, c, r, 0, OB_F); };
    auto cy = [&](Pt r) { return G.df(1, r) * deriv(g, c, r, 1, OB_F); };
    auto cz = [&](Pt r) { return G.df(2, r) * deriv(g, c, r, 2, OB_F); };
    const FT cx2 = avg_c(g, 0, q, [&](Pt r) { FT x = cx(r); return x * x; });
    const FT cy2 = avg_c(g, 1, q, [&](Pt r) { FT x = cy(r); return x * x; });
    const FT cz2 = avg_c(g, 2, q, [&](Pt r) { FT x = cz(r); return x * x; });
    const FT sigma = (cx2 + cy2) + cz2;                   // norm_θᵢ²ᶜᶜᶜ (:374-376)
    if (sigma == FT(0)) return FT(0);
    const FT icx = avg_c(g, 0, q, cx), icy = avg_c(g, 1, q, cy), icz = avg_c(g, 2, q, cz);
    // norm_uᵢⱼ_cⱼ_cᵢᶜᶜᶜ (:347-372); the second-last term of cy_uy interpolates norm_∂y_w with ℑxz as the reference does
    const FT a1 = (G.xu(q) * cx2 + AXY(G.xv(r)) * icx * icy) + AXZ(G.xw(r)) * icx * icz;
    const FT a2 = (AXY(G.yu(r)) * icy * icx + G.yv(q) * cy2) + AXZ(G.yw(r)) * icy * icz;
    const FT a3 = (AXZ(G.zu(r)) * icz * icx + AYZ(G.zv(r)) * icz * icy) + G.zw(q) * cz2;
    const FT theta = (a1 + a2) + a3;
    const FT ka = -Ck * amd_delta2(g, q) * theta / sigma;
    return ka > FT(0) ? ka : FT(0);
#undef AXY
#undef AXZ
#undef AYZ
}

// calc_νᶜᶜᶜ and calc_κᶜᶜᶜ of ALL tracers for one cell of a 3-D grid (no Flat dimension) from ONE evaluation of every normalised
// gradient: the 6 off-diagonal gradients at the 4 points of their averaging stencil (24 values), the 3 diagonal ones, the
// spacing ratios Δᶠ_a / Δᶠ_b once per distinct index pair.  Same expressions, the same order of operations inside each
// expression as amd_nu / amd_kappa above (which evaluate every gradient again at every use: 10 000 instructions and 550
// loads per cell); stretched spacings enter as reciprocals (one rounding of difference).
template <class FT>
OBD void amd_cell(const Phys<FT>& P, const Buoy<FT>& B, const FT* const* U, int ntr, const FT* const* c, Pt q, FT& nu_out,
                  FT* ka_out) {
    const GridD<FT>& g = P.g;
    const long long st[3] = {g.st[0], g.st[1], g.st[2]};
    FT f[3][2], iF[3][2], iC[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        f[d][0] = 2 * spacing(g, d, OB_C, q.i[d]);
        f[d][1] = g.regular[d] ? f[d][0] : 2 * spacing(g, d, OB_C, q.i[d] + 1);
        iF[d][0] = g.regular[d] ? g.invd[d] : 1 / spacing(g, d, OB_F, q.i[d]);
        iF[d][1] = g.regular[d] ? g.invd[d] : 1 / spacing(g, d, OB_F, q.i[d] + 1);
        iC[d] = g.regular[d] ? g.invd[d] : 1 / spacing(g, d, OB_C, q.i[d]);
    }
    // R[a][b] = Δᶠ_n(index + a) / Δᶠ_m(index + b)
    auto ratios = [&](int n, int m, FT (&R)[2][2]) {
        R[0][0] = f[n][0] / f[m][0];
        R[1][0] = g.regular[n] ? R[0][0] : f[n][1] / f[m][0];
        R[0][1] = g.regular[m] ? R[0][0] : f[n][0] / f[m][1];
        R[1][1] = g.regular[n] ? R[0][1] : (g.regular[m] ? R[1][0] : f[n][1] / f[m][1]);
    };
    FT Rxy[2][2], Ryx[2][2], Rxz[2][2], Rzx[2][2], Ryz[2][2], Rzy[2][2];
    ratios(0, 1, Rxy); ratios(1, 0, Ryx); ratios(0, 2, Rxz); ratios(2, 0, Rzx); ratios(1, 2, Ryz); ratios(2, 1, Rzy);
    // normalised gradient of component `comp` along `dd` at the point q + a * st[da] + b * st[db]; (da, db) = the two averaged
    // dimensions; the ratio and the reciprocal face spacing are the caller's
    auto grad = [&](int comp, int dd, long long p, FT ratio, FT inv) { return ratio * ((U[comp][p] - U[comp][p - st[dd]]) * inv); };
    auto avg4 = [](const FT (&F)[2][2]) { return FT(0.5) * (FT(0.5) * (F[0][0] + F[1][0]) + FT(0.5) * (F[0][1] + F[1][1])); };
    auto avg4p = [](const FT (&F)[2][2], const FT (&G2)[2][2]) {
        return FT(0.5) * (FT(0.5) * (F[0][0] * G2[0][0] + F[1][0] * G2[1][0]) + FT(0.5) * (F[0][1] * G2[0][1] + F[1][1] * G2[1][1]));
    };
    FT xv[2][2], yu[2][2], xw[2][2], zu[2][2], yw[2][2], zv[2][2], s12[2][2], s13[2][2], s23[2][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const long long pxy = q.p + a * st[0] + b * st[1], pxz = q.p + a * st[0] + b * st[2], pyz = q.p + a * st[1] + b * st[2];
            xv[a][b] = grad(1, 0, pxy, Rxy[a][b], iF[0][a]);
            yu[a][b] = grad(0, 1, pxy, Ryx[b][a], iF[1][b]);
            xw[a][b] = grad(2, 0, pxz, Rxz[a][b], iF[0][a]);
            zu[a][b] = grad(0, 2, pxz, Rzx[b][a], iF[2][b]);
            yw[a][b] = grad(2, 1, pyz, Ryz[a][b], iF[1][a]);
            zv[a][b] = grad(1, 2, pyz, Rzy[b][a], iF[2][b]);
            s12[a][b] = FT(0.5) * (yu[a][b] + xv[a][b]);
            s13[a][b] = FT(0.5) * (zu[a][b] + xw[a][b]);
            s23[a][b] = FT(0.5) * (zv[a][b] + yw[a][b]);
        }
    const FT xu = (U[0][q.p + st[0]] - U[0][q.p]) * iC[0], yv = (U[1][q.p + st[1]] - U[1][q.p]) * iC[1],
             zw = (U[2][q.p + st[2]] - U[2][q.p]) * iC[2];
    const FT xv2 = avg4p(xv, xv), yu2 = avg4p(yu, yu), xw2 = avg4p(xw, xw), zu2 = avg4p(zu, zu), yw2 = avg4p(yw, yw), zv2 = avg4p(zv, zv);
    const FT Axv = avg4(xv), Ayu = avg4(yu), Axw = avg4(xw), Azu = avg4(zu), Ayw = avg4(yw), Azv = avg4(zv);
    const FT delta2 = amd_delta2(g, q);
    // ---- viscosity (amd_nu) ----
    const FT qn = (((((((xu * xu + yv * yv) + zw * zw) + xv2) + yu2) + xw2) + zu2) + yw2) + zv2;
    FT nu = FT(0);
    if (qn != FT(0)) {
        const FT t1 = ((((xu * (xu * xu) + yv * xv2) + zw * xw2) + 2 * xu * avg4p(xv, s12)) + 2 * xu * avg4p(xw, s13))
                      + 2 * Axv * Axw * avg4(s23);
        const FT t2 = ((((xu * yu2 + yv * (yv * yv)) + zw * yw2) + 2 * yv * avg4p(yu, s12))
                       + 2 * Ayu * Ayw * avg4(s13)) + 2 * yv * avg4p(yw, s23);
        const FT t3 = ((((xu * zu2 + yv * zv2) + zw * (zw * zw)) + 2 * Azu * Azv * avg4(s12))
                       + 2 * zw * avg4p(zu, s13)) + 2 * zw * avg4p(zv, s23);
        const FT rr = (t1 + t2) + t3;
        FT cbz = FT(0);
        if (P.amdHasCb && B.mode) {
            const FT b0 = buoyancy_at(B, q.p);
            FT adb[3];
#pragma unroll
            for (int d = 0; d < 3; ++d)
                adb[d] = FT(0.5) * ((b0 - buoyancy_at(B, q.p - st[d])) * iF[d][0] + (buoyancy_at(B, q.p + st[d]) - b0) * iF[d][1]);
            const FT wx = (Axw * f[0][0]) * adb[0], wy = (Ayw * f[1][0]) * adb[1], wz = (zw * f[2][0]) * adb[2];
            cbz = P.amdCb * ((wx + wy) + wz) / f[2][0];
        }
        nu = -P.amdCnu * delta2 * (rr - cbz) / qn;
        nu = nu > FT(0) ? nu : FT(0);
    }
    nu_out = nu;
    // ---- diffusivities (amd_kappa) ----
    if (ntr > 0) {
        FT ywxz[2][2];          // ∂y w interpolated with ℑxz, as the reference's cy_uy does
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) ywxz[a][b] = grad(2, 1, q.p + a * st[0] + b * st[2], Ryz[0][b], iF[1][0]);
        const FT Aywxz = avg4(ywxz);
        for (int t = 0; t < ntr; ++t) {
            const FT* cc = c[t];
            const FT c0 = cc[q.p];
            FT cg[3][2];
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                cg[d][0] = f[d][0] * ((c0 - cc[q.p - st[d]]) * iF[d][0]);
                cg[d][1] = f[d][1] * ((cc[q.p + st[d]] - c0) * iF[d][1]);
            }
            const FT cx2 = FT(0.5) * (cg[0][0] * cg[0][0] + cg[0][1] * cg[0][1]), cy2 = FT(0.5) * (cg[1][0] * cg[1][0] + cg[1][1] * cg[1][1]),
                     cz2 = FT(0.5) * (cg[2][0] * cg[2][0] + cg[2][1] * cg[2][1]);
            const FT sigma = (cx2 + cy2) + cz2;
            FT ka = FT(0);
            if (sigma != FT(0)) {
                const FT icx = FT(0.5) * (cg[0][0] + cg[0][1]), icy = FT(0.5) * (cg[1][0] + cg[1][1]), icz = FT(0.5) * (cg[2][0] + cg[2][1]);
                const FT a1 = (xu * cx2 + Axv * icx * icy) + Axw * icx * icz;
                const FT a2 = (Ayu * icy * icx + yv * cy2) + Aywxz * icy * icz;
                const FT a3 = (Azu * icz * icx + Azv * icz * icy) + zw * cz2;
                const FT theta = (a1 + a2) + a3;
                ka = -P.amdCk[t] * delta2 * theta / sigma;
                ka = ka > FT(0) ? ka : FT(0);
            }
            ka_out[t] = ka;
        }
    }
}

// ---- tendencies: nonhydrostatic_tendency_kernel_functions.jl:44-232 (term order kept) -------
// comp 0,1,2 = u,v,w ; comp >= 3 = tracer (comp-3).  BG: the two background terms after the first advection term
template <class FT, bool BG = false>
OBD FT tendency(const Phys<FT>& P, int comp, const FT* const* U, const FT* psi, const FT* pHY,
                const Buoy<FT>& b, Pt q) {
    const GridD<FT>& g = P.g;
    if (comp >= 3) {
        FT G = -div_Uc(P, U, psi, q);
        if constexpr (BG) {          // - div_Uc(U_bg, c) - div_Uc(U, c_bg)   (:225-226)
            if (P.bgU[0]) G = G - div_Uc(P, P.bgU, psi, q);
            if (P.bg[comp]) G = G - div_Uc(P, U, P.bg[comp], q);
        }
        G = G - div_q(P, P.kappa[comp - 3], psi, q, P.kappae[comp - 3]);
        if (P.frc[comp].on) G = G + relaxation(P.frc[comp], q.i[0], q.i[1], q.i[2], psi[q.p]);     // + forcing (:231)
        return G;
    }
    FT G = -div_Uu(P, comp, U, psi, q);
    if constexpr (BG) {              // - div_𝐯u(U_bg, u) - div_𝐯u(U, u_bg)   (:62-63, :119-120, :173-174)
        if (P.bgU[0]) G = G - div_Uu(P, comp, P.bgU, psi, q);
        if (P.bg[comp]) G = G - div_Uu(P, comp, U, P.bg[comp], q);
    }
    if (comp == 0) {
        if (P.fplane) {          // x_f_cross_U = -f ℑxyᶠᶜᵃ(v) = -f ℑyᵃᶜᵃ(ℑxᶠᵃᵃ v)   (f_plane.jl:42)
            FT a0 = IF(g, U[1], q, 0);
            FT v = g.topo[1] == OB_FLAT ? a0 : FT(0.5) * (a0 + IF(g, U[1], sh(g, q, 1, 1), 0));
            G = G - (-P.f * v);
        }
        if (pHY) G = G - deriv(g, pHY, q, 0, OB_F);
    } else if (comp == 1) {
        if (P.fplane) {          // y_f_cross_U = f ℑxyᶜᶠᵃ(u) = f ℑyᵃᶠᵃ(ℑxᶜᵃᵃ u)       (f_plane.jl:43)
            FT a1 = IC(g, U[0], q, 0);
            FT u = g.topo[1] == OB_FLAT ? a1 : FT(0.5) * (IC(g, U[0], sh(g, q, 1, -1), 0) + a1);
            G = G - (P.f * u);
        }
        if (pHY) G = G - deriv(g, pHY, q, 1, OB_F);
    }
    G = G - div_tau(P, comp, U, q);
    if (comp < 2 && P.tilted && b.mode) G = G + P.ghat[comp] * buoyancy_at(b, q.p);      // x/y_dot_g_b (g_dot_b.jl:1-3)
    if (P.frc[comp].on) G = G + relaxation(P.frc[comp], q.i[0], q.i[1], q.i[2], psi[q.p]);     // + forcings.u/v/w (:71, :128, :180)
    return G;
}

}  // namespace ob
