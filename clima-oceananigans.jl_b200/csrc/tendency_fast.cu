// tendency_fast.cu -- specialised tendency (+ fused RK3/AB2 substep) kernel for the headline
// configuration: every non-Flat dimension Periodic, regular spacing, WENO5 with uniform
// coefficients (Z or JS weights), closure = nothing, optional FPlane and hydrostatic pressure.
// The tendency plan (capi.cu: plan_tendencies) sends 3-D grids to the TMA-staged kernel (tendency_tma.cu); the kernel
// here runs the 2-D grids (z Flat).
//
// Same quantities as physics.cuh (reference files cited there), reorganised for the FP64 pipe,
// which is what bounds this kernel on B200 (about 20-30 flop per byte of compulsory traffic):
//   * every face flux is evaluated ONCE and shared through shared memory; the one extra column
//     and row of faces a 32x8 tile needs are computed by two otherwise idle warps
//     (the reference evaluates every face twice, momentum_advection_operators.jl:52-56);
//   * only the UPWIND-side WENO reconstruction is evaluated: ((u+|u|) L + (u-|u|) R)/2 is exactly
//     u*L or u*R (upwind_biased_advective_fluxes.jl:10), chosen per thread by address selection of
//     a mirrored 5-point window (the reference always evaluates both sides);
//   * in Float64 the six divisions of the weight computation (:386-400) are folded into one
//     reciprocal:  sum_k w_k p_k = (sum_k g_k p_k) / (sum_k g_k),
//     g_k = C_k (E_k + tau^2) prod_{j != k} E_j,  E_k = (beta_k + eps)^2   (Z weights), which is
//     the same rational function evaluated with ~1e-16 relative differences.
// Parity with the oracle stays <= 1e-12 per step (tests/test_gpu_parity.py).
#include "internal.h"
#include "weno_fast.cuh"

namespace ob {

namespace fast {

template <class FT>
struct Ctx {
    const FT* U[2];
    const FT* psi;
    const FT* pHY;
    const FT* Gm;
    FT* Gn;
    FT* psi_new;
    long long s[3];
    FT area[2], invV, invd[2];
    FT f;
    int fplane;
    int N[2];
    Substep<FT> ss;
};

// (I(p) + I(p + s))/2 along stride s (see wf::interp4)
template <class FT>
__device__ __forceinline__ FT I4f(const FT* c, long long p, long long s) {
    return wf::interp4<FT>(c[p - s], c[p], c[p + s], c[p + 2 * s]);
}

// area * upwind flux of psi (component B, or tracer B = 3) in direction A (x or y) at position p
// (A == B: cell-centre index; otherwise face index along A)
template <class FT, bool ZW, int A, int B>
__device__ __forceinline__ FT flux_at(const Ctx<FT>& c, long long p) {
    const long long sA = c.s[A];
    FT ut;
    long long pf = p;
    if constexpr (B >= 2) {       // a tracer, or w, which is centred in the Flat z: U[A] is already at the face
        ut = c.U[A][p];
    } else if constexpr (A == B) {
        ut = I4f<FT>(c.U[A], p, sA);
        pf = p + sA;
    } else {
        const long long sB = c.s[B];
        ut = I4f<FT>(c.U[A], p - sB, sB);
    }
    // all six loads are issued independently of ut (no dependent second memory round trip);
    // the upwind window is then selected in registers
    const FT* q = c.psi + pf;
    const FT w0 = q[-3 * sA], w1 = q[-2 * sA], w2 = q[-sA], w3 = q[0], w4 = q[sA], w5 = q[2 * sA];
    FT rec = wf::weno_upwind<FT, ZW>(ut > FT(0), w0, w1, w2, w3, w4, w5);
    return c.area[A] * (ut * rec);
}

template <class FT, bool ZW, int B>
__global__ void __launch_bounds__(TX* TY, 2) tendency_fast_kernel(Ctx<FT> c) {
    __shared__ FT sFx[TY][TX + 1];
    __shared__ FT sFy[TY + 1][TX];
    const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * TX + tx;
    const int i0 = 1 + blockIdx.x * TX, j0 = 1 + blockIdx.y * TY;
    const int i = i0 + tx;
    const long long sx = c.s[0], sy = c.s[1], sz = c.s[2];
    // x: B == 0 needs F(i) - F(i-1) (extra column at i0-1), otherwise F(i+1) - F(i) (extra at i0+TX); y alike
    constexpr bool XLOW = (B == 0), YLOW = (B == 1);
    const long long p = i * sx + (j0 + ty) * sy + sz;       // the one level, k = 1
    // extra faces: warp 0 lanes 0..TY-1 -> x column ; warp 1 -> y row
    const bool xextra = tid < TY, yextra = tid >= 32 && tid < 32 + TX;
    const long long pxe = (XLOW ? (i0 - 1) : (i0 + TX)) * sx + (j0 + tid) * sy + sz;
    const long long pye = (i0 + (tid - 32)) * sx + (YLOW ? (j0 - 1) : (j0 + TY)) * sy + sz;

    const FT Fx = flux_at<FT, ZW, 0, B>(c, p);
    const FT Fy = flux_at<FT, ZW, 1, B>(c, p);
    sFx[ty][XLOW ? tx + 1 : tx] = Fx;
    sFy[YLOW ? ty + 1 : ty][tx] = Fy;
    if (xextra) sFx[tid][XLOW ? 0 : TX] = flux_at<FT, ZW, 0, B>(c, pxe);
    if (yextra) sFy[YLOW ? 0 : TY][tid - 32] = flux_at<FT, ZW, 1, B>(c, pye);
    __syncthreads();
    const FT dFx = XLOW ? (Fx - sFx[ty][tx]) : (sFx[ty][tx + 1] - Fx);
    const FT dFy = YLOW ? (Fy - sFy[ty][tx]) : (sFy[ty + 1][tx] - Fy);
    FT G = -(c.invV * (dFx + dFy));
    if (B == 0) {
        if (c.fplane) {      // - x_f_cross_U = + f * ℑxyᶠᶜᵃ(v)
            const FT* v = c.U[1];
            FT a0 = FT(0.5) * (v[p - sx] + v[p]), a1 = FT(0.5) * (v[p - sx + sy] + v[p + sy]);
            G = G - (-c.f * (FT(0.5) * (a0 + a1)));
        }
        if (c.pHY) G = G - (c.pHY[p] - c.pHY[p - sx]) * c.invd[0];
    } else if (B == 1) {
        if (c.fplane) {      // - y_f_cross_U = - f * ℑxyᶜᶠᵃ(u)
            const FT* u = c.U[0];
            FT a0 = FT(0.5) * (u[p - sy] + u[p + sx - sy]), a1 = FT(0.5) * (u[p] + u[p + sx]);
            G = G - (c.f * (FT(0.5) * (a0 + a1)));
        }
        if (c.pHY) G = G - (c.pHY[p] - c.pHY[p - sy]) * c.invd[1];
    }
    c.Gn[p] = G;
    if (c.ss.mode == SUB_RK3_FIRST) c.psi_new[p] = c.psi[p] + c.ss.c1 * G;
    else if (c.ss.mode == SUB_RK3) c.psi_new[p] = c.psi[p] + c.ss.dt * (c.ss.c1 * G + c.ss.c2 * c.Gm[p]);
    else if (c.ss.mode == SUB_AB2) c.psi_new[p] = c.psi[p] + c.ss.dt * (c.ss.c1 * G - c.ss.c2 * c.Gm[p]);
}

template <class FT, bool ZW>
void launch(const Ctx<FT>& c, int comp) {
    dim3 blk(TX, TY), grd(c.N[0] / TX, c.N[1] / TY);
    switch (comp) {
        case 0: tendency_fast_kernel<FT, ZW, 0><<<grd, blk, 0, stream()>>>(c); break;
        case 1: tendency_fast_kernel<FT, ZW, 1><<<grd, blk, 0, stream()>>>(c); break;
        case 2: tendency_fast_kernel<FT, ZW, 2><<<grd, blk, 0, stream()>>>(c); break;
        default: tendency_fast_kernel<FT, ZW, 3><<<grd, blk, 0, stream()>>>(c); break;
    }
    OB_LAUNCH_CHECK();
}

}  // namespace fast

template <class FT>
void launch_tendency_fast(const Phys<FT>& P, int comp, const FT* const U[3], const FT* psi,
                          const FT* pHY, FT* Gn, const FT* Gm, FT* psi_new, const Substep<FT>& ss) {
    const GridD<FT>& g = P.g;
    fast::Ctx<FT> c;
    for (int d = 0; d < 2; ++d) { c.U[d] = U[d]; c.N[d] = g.N[d]; c.invd[d] = 1 / g.d[d]; }
    for (int d = 0; d < 3; ++d) c.s[d] = g.st[d];
    c.psi = psi; c.pHY = pHY; c.Gm = Gm; c.Gn = Gn; c.psi_new = psi_new; c.ss = ss;
    c.area[0] = g.d[1] * g.d[2]; c.area[1] = g.d[0] * g.d[2];
    c.invV = 1 / ((g.d[0] * g.d[1]) * g.d[2]);
    c.f = P.f; c.fplane = P.fplane;
    if (P.zweno) fast::launch<FT, true>(c, comp); else fast::launch<FT, false>(c, comp);
}
template void launch_tendency_fast<float>(const Phys<float>&, int, const float* const[3], const float*,
                                          const float*, float*, const float*, float*, const Substep<float>&);
template void launch_tendency_fast<double>(const Phys<double>&, int, const double* const[3], const double*,
                                           const double*, double*, const double*, double*, const Substep<double>&);
}  // namespace ob
