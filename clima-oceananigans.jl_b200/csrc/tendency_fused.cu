// tendency_fused.cu -- ONE launch per stage for the tendencies + substep of u, v, w and the first tracer of the headline
// configuration (every non-Flat dimension Periodic or slab-decomposed, regular spacing, WENO5 with uniform
// coefficients, closure = nothing, optional FPlane / hydrostatic pressure).
//
// Replaces calculate_Gu!/Gv!/Gw!/Gc! (calculate_nonhydrostatic_tendencies.jl:155-180), rk3_substep_field!
// (runge_kutta_3.jl:204-218) / ab2_step_field! (quasi_adams_bashforth_2.jl:158-166) and store_field_tendencies!.
//
// Design (B200: 227 KB of shared memory per SM, TMA, 64 FP64 lanes and one 128 B/clk shared-memory port per SM):
//   * one PERSISTENT block per SM owns a 32 x R column tile and marches up in k.  Every state array is staged ONCE
//     per level by the Tensor Memory Accelerator (cp.async.bulk.tensor.3d, SASS UTMALDG) into an 8-slot ring of
//     (32+8) x (R+6) halo'd planes (levels k-3 .. k+3 live, k+4 in flight); the rings of u, v, w serve both as the
//     advected quantity of their own momentum equation and as the advecting velocities of all the others, so a
//     stage reads each state plane from HBM once instead of 3-4 times (one launch per field before);
//   * the warps form NG independent GROUPS that share the staged planes but own different FIELDS ((u, v) and
//     (w, c) with a tracer; u / v / w without): twice the warps on the same shared memory, each group with its own
//     named barrier, so one group's barrier drain is covered by the other's arithmetic.  In a group, warps 0..R-1
//     own one row of 32 cells (per level and field three face fluxes: x, y, z-top; the z face is carried in a
//     register along k, x / y faces are exchanged through shared memory) and warp R computes the extra column / row
//     of faces of the tile;
//   * a dedicated producer warp issues the TMA loads: `full` mbarriers (transaction counts) publish a level to the
//     groups, `done` mbarriers (one arrival per group and level) return the slot, so the groups may drift apart by
//     a level without a block-wide barrier;
//   * tiles are scheduled in LOCKSTEP (block b owns tiles b, b + G, ...; all blocks are at the same level at the same
//     time, so the halo rows / columns two neighbouring tiles share are read from HBM once and hit in L2 the second
//     time); the tiles left over after the last full round are split evenly over all blocks along z, so there is no
//     tail and no wave quantisation;
//   * shared-memory traffic is the second scarce resource (a warp-wide LDS.64 takes 2 cycles of the port, an FP64
//     instruction 0.5 cycles of the SM's FP64 lanes): faces whose advecting velocity is interpolated from the
//     advected field itself (u in x, v in y, w in z) take it from the six window values they load anyway; windows in
//     x and z are selected by ADDRESS (five loads, conflict-free in z, nearly so in x), windows in y by register
//     selects (the row pitch of 40 would make address selection a two-way bank conflict);
//   * constant factors (1/2 of the two-point averages, 1/12 of the fourth-order interpolant, face areas / volume) are
//     folded into three coefficients applied to the flux DIFFERENCES, and 4 eps into the smoothness-indicator FMA
//     (weno_fast.cuh: weno_face2): 170 FP64 instructions per cell and field against 193.
// Same rational functions of the same inputs as the reference (differences ~1e-16 relative); parity <= 1e-12 per
// step is tested against the oracle (tests/test_gpu_parity.py, tests/test_gpu_golden.py).
#include "internal.h"
#include "weno_fast.cuh"
#include "tma_util.cuh"
#include <algorithm>
#include <type_traits>

namespace ob {
namespace fz {

constexpr int COL0 = HALO + 1, BX = TX + 2 * HALO + 2, SLOTS = 8;      // TX, HALO: internal.h

template <int NT> struct Groups {          // field -> group map
    static constexpr int NF = 3 + NT;
    static constexpr int NG = NT == 0 ? 3 : 2;
    static constexpr int FPG = NT == 0 ? 1 : 2;      // fields per group
};

template <class FT, int R, int NF> struct Geo {
    static constexpr int BY = R + 2 * HALO;
    static constexpr int BOX_BYTES = BX * BY * (int)sizeof(FT);
    static constexpr int PLANE_BYTES = ((BOX_BYTES + 127) / 128) * 128;
    static constexpr int PE = PLANE_BYTES / (int)sizeof(FT);
    static constexpr int FXE = R * (TX + 1), FYE = (R + 1) * TX;       // exchange buffers per field (x faces, y faces)
    static constexpr int XE = NF * (FXE + FYE);                        // one set of exchange buffers
    static constexpr size_t SMEM = (size_t)NF * SLOTS * PLANE_BYTES + (size_t)XE * sizeof(FT);
};

template <class FT, int NF>
struct Args {
    CUtensorMap tm[NF];
    const FT* Gm[NF];
    FT* Gn[NF];
    FT* nw[NF];
    const FT* pHY;
    long long sy, sz;
    int O[3];
    int Ny, Nz, ntx, ntiles, chunk;
    int tile0, tsplit, tskip;      // tile t of this launch is tile t + tile0 (+ tskip for t >= tsplit) of the grid (part launches)
    FT cf[3];              // area[A] / V (further scaled per field class in the kernel)
    FT invdx, invdy, f;
    int fplane, do_sub;
    FT ca, cb;             // psi_new = psi + ca * G + cb * G^-
    // Bounded (stretched) z variant
    const FT* izC;         // 1 / Δz of cell k, 1 / Δz at face k (Julia index k)
    const FT* izF;
    const FT* tabF;        // packed WENO coefficient tables of z (Phys::wzp): reconstruction at Faces (u, v, c) / Centers (w)
    const FT* tabC;
    FT vh[2], v24;         // -24 ν / Δx, -24 ν / Δy, -24 ν    (viscous fluxes in the 24 x units of the momentum fluxes)
    FT th[2], t2;          // -2 κ / Δx, -2 κ / Δy, -2 κ       (diffusive fluxes of the tracer, 2 x units)
    FT fbb[NF], fbt[NF];   // constant Flux boundary conditions at the bottom / top (0: none)
};
// the forced instantiations (FRC) take the relaxation forcing of every field in addition; the unforced ones keep Args
template <class FT, int NF>
struct ArgsF : Args<FT, NF> {
    Relax<FT> frc[NF];
};
template <class FT, int NF, bool FRC> using KArgs = std::conditional_t<FRC, ArgsF<FT, NF>, Args<FT, NF>>;

// ---- work decomposition: whole tiles in lockstep rounds, then the leftover tiles split along z ----------------
// (all 32-bit and a pure function of blockIdx / gridDim / kernel parameters, so that the level index and the ring-slot
// offsets derived from it stay in UNIFORM registers)
struct Work {
    int Nz, G, b, full, round, pos, end;
    __device__ __forceinline__ Work(int ntiles, int Nz_, int chunk) : Nz(Nz_), G(gridDim.x), b(blockIdx.x), round(0) {
        full = ntiles / G;
        const int T2 = (ntiles - full * G) * Nz;        // leftover levels; `chunk` = ceil(T2 / G) from the host
        pos = min(T2, b * chunk);
        end = min(T2, pos + chunk);
    }
    __device__ __forceinline__ bool next(int& tile, int& kfirst, int& len) {
        if (round < full) {
            tile = round * G + b; kfirst = 0; len = Nz;
            ++round;
            return true;
        }
        if (pos >= end) return false;
        const int t2 = pos / Nz;
        tile = full * G + t2;
        kfirst = pos - t2 * Nz;
        len = min(Nz - kfirst, end - pos);
        pos += len;
        return true;
    }
};

__device__ __forceinline__ void named_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <class FT>
__device__ __forceinline__ FT interp12(FT cm, FT c0, FT c1, FT c2) {      // 12 x wf::interp4
    return fma(FT(7), c0 + c1, -(cm + c2));
}
// twice the upwind reconstruction from the six values around the face, selected in registers
template <class FT, bool ZW>
__device__ __forceinline__ FT weno_sel6(bool pos, FT w0, FT w1, FT w2, FT w3, FT w4, FT w5) {
    const FT c = pos ? w2 : w3;
    return wf::weno_face2<FT, ZW>(pos ? w0 : w5, pos ? w1 : w4, c, pos ? w3 : w2, pos ? w4 : w1, pos ? c : w5, pos ? c : w1);
}

// 24 x (momentum) or 2 x (tracers) the upwind flux ut * psi_face of field ring FB (component B, 3 = tracer) in
// direction A at plane element e, relative level NQ (A == B: cell-centre index; otherwise face index along A)
template <class FT, bool ZW, int A, int B, int NQ, int PE>
__device__ __forceinline__ FT flux(const FT* __restrict__ S, const int (&so)[SLOTS], int FB, int e) {
    constexpr int sA = A == 0 ? 1 : BX;
    if constexpr (B != 3 && A == B) {
        // the advecting velocity is the fourth-order interpolant of the advected component itself: values 1..4 of the window
        FT w[6];
        if constexpr (A < 2) {
            const FT* q = S + FB * SLOTS * PE + so[NQ + 3] + e + sA;
#pragma unroll
            for (int n = 0; n < 6; ++n) w[n] = q[(n - 3) * sA];
        } else {
            const FT* q = S + FB * SLOTS * PE + e;
#pragma unroll
            for (int n = 0; n < 6; ++n) w[n] = q[so[NQ + 1 + n]];          // levels NQ+1-3 .. NQ+1+2
        }
        const FT ut = interp12<FT>(w[1], w[2], w[3], w[4]);
        return ut * weno_sel6<FT, ZW>(ut > FT(0), w[0], w[1], w[2], w[3], w[4], w[5]);
    } else {
        FT ut;
        if constexpr (B == 3) {
            ut = S[A * SLOTS * PE + so[NQ + 3] + e];
        } else if constexpr (B < 2) {
            constexpr int sB = B == 0 ? 1 : BX;
            const FT* q = S + A * SLOTS * PE + so[NQ + 3] + e;
            ut = interp12<FT>(q[-2 * sB], q[-sB], q[0], q[sB]);
        } else {
            const FT* q = S + A * SLOTS * PE + e;
            ut = interp12<FT>(q[so[NQ + 1]], q[so[NQ + 2]], q[so[NQ + 3]], q[so[NQ + 4]]);
        }
        const bool pos = ut > FT(0);
        if constexpr (A == 1) {
            const FT* q = S + FB * SLOTS * PE + so[NQ + 3] + e;
            return ut * weno_sel6<FT, ZW>(pos, q[-3 * BX], q[-2 * BX], q[-BX], q[0], q[BX], q[2 * BX]);
        } else {
            FT a, b, c, d, g;
            if constexpr (A == 0) {
                const int base = FB * SLOTS * PE + so[NQ + 3] + e;
                const int A0 = pos ? base : base - 1, t = pos ? 1 : -1;
                a = S[A0 - 3 * t]; b = S[A0 - 2 * t]; c = S[A0 - t]; d = S[A0]; g = S[A0 + t];
            } else {
                const FT* q = S + FB * SLOTS * PE + e;
                const int oa = pos ? so[NQ] : so[NQ + 5], ob_ = pos ? so[NQ + 1] : so[NQ + 4],
                          oc = pos ? so[NQ + 2] : so[NQ + 3], od = pos ? so[NQ + 3] : so[NQ + 2],
                          og = pos ? so[NQ + 4] : so[NQ + 1];
                a = q[oa]; b = q[ob_]; c = q[oc]; d = q[od]; g = q[og];
            }
            return ut * wf::weno_face2<FT, ZW>(a, b, c, d, g, pos ? c : a, pos ? c : g);
        }
    }
}

// ---- Bounded, vertically stretched z (BASELINE config 3) ---------------------------------------------------------
// Same units and conventions as flux(); k is the level the block is at.  What changes against the periodic variant:
//   * interpolants along z fall back to the second-order average next to the walls
//     (topologically_conditional_interpolation.jl:19-80 with the buffer of WENO5 = 2: fourth-order symmetric for
//     2 < k < N-1, left-biased 2 < k < N, right-biased 1 < k < N-1);
//   * reconstructions along z use the stretched-grid coefficient tables (weno_fifth_order.jl:526-553) with the uniform
//     smoothness indicators (weno_fast.cuh weno_face_tab2: one arithmetic for both sides on the window ordered towards the
//     face, with the packed 80-byte table row of (index, side) fetched by five 16-byte loads);
//   * every face carries the viscous / diffusive flux of ScalarDiffusivity, -ν (∂_A u_B + ∂_B u_A) resp. -κ ∂_A c
//     (closure_kernel_operators.jl:22-48): the two differences are the central pairs of the windows that the advective
//     flux loads anyway (the advected field along A, the advecting velocity along B), so no extra shared-memory reads.
// twice the upwind reconstruction along z at index kq; (a .. g) = the window ordered towards the face, (x2, x0) as in
// weno_fast.cuh, i2 = the sum of the two values next to the face
template <class FT, bool ZW>
__device__ __forceinline__ FT zrecon2(const FT* __restrict__ tab, int N, int kq, bool pos, FT a, FT b, FT cc, FT d, FT g, FT x2,
                                      FT x0, FT i2) {
    const bool outL = kq > 2 && kq < N, outR = kq > 1 && kq < N - 1;
    if (!(outL || outR)) return i2;
    FT cf[10];
    if constexpr (sizeof(FT) == 8) {
        const double2* t = reinterpret_cast<const double2*>(tab) + (2 * kq + (pos ? 1 : 0)) * 5;
#pragma unroll
        for (int q = 0; q < 5; ++q) { const double2 v = __ldg(t + q); cf[2 * q] = v.x; cf[2 * q + 1] = v.y; }
    } else {
        const float2* t = reinterpret_cast<const float2*>(tab) + (2 * kq + (pos ? 1 : 0)) * 5;
#pragma unroll
        for (int q = 0; q < 5; ++q) { const float2 v = __ldg(t + q); cf[2 * q] = v.x; cf[2 * q + 1] = v.y; }
    }
    const FT r = wf::weno_face_tab2<FT, ZW>(a, b, cc, d, g, x2, x0, cf);
    if (outL && outR) return r;
    return (pos ? outL : outR) ? r : i2;
}

template <class FT, bool ZW, int A, int B, int NQ, int PE, int NF>
__device__ __forceinline__ FT fluxb(const Args<FT, NF>& c, int k, const FT* __restrict__ S, const int (&so)[SLOTS], int FB, int e) {
    constexpr int sA = A == 0 ? 1 : BX;
    const int kq = k + NQ;
    if constexpr (B != 3 && A == B) {
        FT w[6];
        if constexpr (A < 2) {
            const FT* q = S + FB * SLOTS * PE + so[NQ + 3] + e + sA;
#pragma unroll
            for (int n = 0; n < 6; ++n) w[n] = q[(n - 3) * sA];
            const FT ut = interp12<FT>(w[1], w[2], w[3], w[4]);
            const FT visc = (2 * c.vh[A]) * (w[3] - w[2]);
            return fma(ut, weno_sel6<FT, ZW>(ut > FT(0), w[0], w[1], w[2], w[3], w[4], w[5]), visc);
        } else {
            const FT* q = S + FB * SLOTS * PE + e;
#pragma unroll
            for (int n = 0; n < 6; ++n) w[n] = q[so[NQ + 1 + n]];          // levels kq-2 .. kq+3 (w faces around centre kq)
            const bool oc = kq > 2 && kq < c.Nz - 1;
            const FT i2 = w[2] + w[3];
            const FT ut = oc ? interp12<FT>(w[1], w[2], w[3], w[4]) : FT(6) * i2;
            const bool pos = ut > FT(0);
            const FT wc_ = pos ? w[2] : w[3];
            const FT rec = zrecon2<FT, ZW>(c.tabC, c.Nz, kq, pos, pos ? w[0] : w[5], pos ? w[1] : w[4], wc_, pos ? w[3] : w[2],
                                           pos ? w[4] : w[1], pos ? wc_ : w[5], pos ? wc_ : w[1], i2);
            const FT visc = ((2 * c.v24) * __ldg(c.izC + kq)) * (w[3] - w[2]);
            return fma(ut, rec, visc);
        }
    } else {
        FT ut, visc = FT(0);
        if constexpr (B == 3) {
            ut = S[A * SLOTS * PE + so[NQ + 3] + e];
        } else if constexpr (B < 2) {
            constexpr int sB = B == 0 ? 1 : BX;
            const FT* q = S + A * SLOTS * PE + so[NQ + 3] + e;
            const FT cm = q[-sB], c0 = q[0];
            ut = interp12<FT>(q[-2 * sB], cm, c0, q[sB]);
            visc = c.vh[B] * (c0 - cm);
        } else {            // w advected by u / v: the advecting velocity is interpolated along z at face level k
            const FT* q = S + A * SLOTS * PE + e;
            const FT cm = q[so[NQ + 2]], c0 = q[so[NQ + 3]];
            const bool oc = kq > 2 && kq < c.Nz - 1;
            ut = oc ? interp12<FT>(q[so[NQ + 1]], cm, c0, q[so[NQ + 4]]) : FT(6) * (cm + c0);
            visc = (c.v24 * __ldg(c.izF + kq)) * (c0 - cm);
        }
        const bool pos = ut > FT(0);
        if constexpr (A == 1) {
            const FT* q = S + FB * SLOTS * PE + so[NQ + 3] + e;
            const FT w2 = q[-BX], w3 = q[0];
            visc = fma(B == 3 ? c.th[1] : c.vh[1], w3 - w2, visc);
            return fma(ut, weno_sel6<FT, ZW>(pos, q[-3 * BX], q[-2 * BX], w2, w3, q[BX], q[2 * BX]), visc);
        } else if constexpr (A == 0) {
            const int base = FB * SLOTS * PE + so[NQ + 3] + e;
            const int A0 = pos ? base : base - 1, t = pos ? 1 : -1;
            const FT a = S[A0 - 3 * t], b = S[A0 - 2 * t], cc = S[A0 - t], d = S[A0], g = S[A0 + t];
            visc = fma(B == 3 ? c.th[0] : c.vh[0], pos ? d - cc : cc - d, visc);
            return fma(ut, wf::weno_face2<FT, ZW>(a, b, cc, d, g, pos ? cc : a, pos ? cc : g), visc);
        } else {            // z face at level kq of u, v or the tracer: natural windows kq-3 .. kq+1 (left) / kq-2 .. kq+2 (right)
            const FT* q = S + FB * SLOTS * PE + e;
            const int oa = pos ? so[NQ] : so[NQ + 5], ob_ = pos ? so[NQ + 1] : so[NQ + 4], oc = pos ? so[NQ + 2] : so[NQ + 3],
                      od = pos ? so[NQ + 3] : so[NQ + 2], og = pos ? so[NQ + 4] : so[NQ + 1];
            const FT a = q[oa], b = q[ob_], cc = q[oc], d = q[od], g = q[og];
            visc = fma((B == 3 ? c.t2 : c.v24) * __ldg(c.izF + kq), pos ? d - cc : cc - d, visc);     // levels kq-1, kq
            return fma(ut, zrecon2<FT, ZW>(c.tabF, c.Nz, kq, pos, a, b, cc, d, g, pos ? cc : a, pos ? cc : g, cc + d), visc);
        }
    }
}

template <class FT, bool ZW, int ZT, int A, int B, int NQ, int PE, int NF>
__device__ __forceinline__ FT fluxs(const Args<FT, NF>& c, int k, const FT* __restrict__ S, const int (&so)[SLOTS], int FB, int e) {
    if constexpr (ZT) return fluxb<FT, ZW, A, B, NQ, PE, NF>(c, k, S, so, FB, e);
    else return flux<FT, ZW, A, B, NQ, PE>(S, so, FB, e);
}

// one field of one level for a cell thread: first the faces that are exchanged (x, y), then the z-top face
template <class FT, bool ZW, int ZT, int B, int PE, int NF>
__device__ __forceinline__ void cell_fluxes_xy(const Args<FT, NF>& c, int k, const FT* S, const int (&so)[SLOTS], int FB, int e,
                                               bool first, FT& Fx, FT& Fy, FT& Fz) {
    constexpr int NQL = B == 2 ? -1 : 0;
    if (first) Fz = fluxs<FT, ZW, ZT, 2, B, NQL, PE, NF>(c, k, S, so, FB, e);
    Fx = fluxs<FT, ZW, ZT, 0, B, 0, PE, NF>(c, k, S, so, FB, e);
    Fy = fluxs<FT, ZW, ZT, 1, B, 0, PE, NF>(c, k, S, so, FB, e);
}
template <class FT, bool ZW, int ZT, int B, int PE, int NF>
__device__ __forceinline__ void cell_flux_z(const Args<FT, NF>& c, int k, const FT* S, const int (&so)[SLOTS], int FB, int e,
                                            FT& Fz, FT& dFz) {
    constexpr int NQH = B == 2 ? 0 : 1;
    const FT Fn = fluxs<FT, ZW, ZT, 2, B, NQH, PE, NF>(c, k, S, so, FB, e);
    dFz = Fn - Fz;
    Fz = Fn;
}

template <class FT, bool ZW, int ZT, int NT, bool HAS_GM, bool ACC, int R, int GRP, bool FRC>
__device__ __forceinline__ void group_main(const KArgs<FT, 3 + NT, FRC>& c, FT* S, FT* sX, unsigned long long* full,
                                           unsigned long long* done) {
    using GR = Groups<NT>;
    constexpr int NF = GR::NF, FPG = GR::FPG;
    using G_ = Geo<FT, R, NF>;
    constexpr int PE = G_::PE;
    constexpr int F0 = GRP * FPG;                 // first field of this group
    constexpr int GT = TX * (R + 1);              // threads of the group
    const int tx = threadIdx.x & 31, ty = (threadIdx.x >> 5) - GRP * (R + 1);
    const bool edge = ty == R;
    const unsigned sy = (unsigned)c.sy, sz = (unsigned)c.sz;
    const FT cmx = c.cf[0] * FT(1.0 / 24.0), cmy = c.cf[1] * FT(1.0 / 24.0), cmz = c.cf[2] * FT(1.0 / 24.0);
    const FT ctx_ = c.cf[0] * FT(0.5), cty = c.cf[1] * FT(0.5), ctz = c.cf[2] * FT(0.5);
    const int e = (ty + HALO) * BX + tx + COL0;
    unsigned git = 0;
    Work wk(c.ntiles, c.Nz, c.chunk);
    int tile, kfirst, len;
    while (wk.next(tile, kfirst, len)) {
        tile += c.tile0 + (tile >= c.tsplit ? c.tskip : 0);
        const int bx = tile % c.ntx, by = tile / c.ntx;
        const int i0 = 1 + bx * TX, j0 = 1 + by * R, k0 = 1 + kfirst;
        const int nrows = min(R, c.Ny - j0 + 1);
        const bool cell = !edge && ty < nrows;
        __syncthreads();                          // (all roles) the rings are refilled from scratch
        unsigned p = (unsigned)(i0 + tx) + (unsigned)(j0 + ty) * sy + (unsigned)k0 * sz;      // < 2^31 elements per field
        FT Fz[FPG];
#pragma unroll
        for (int s = 0; s < FPG; ++s) Fz[s] = FT(0);
        for (int it = 0; it < len; ++it, ++git) {
            const int k = k0 + it;
            int so[SLOTS];                        // element offset of the slot of level k + n, n = -3 .. 4
#pragma unroll
            for (int n = 0; n < SLOTS; ++n) so[n] = ((k + n - 3) & (SLOTS - 1)) * PE;
            FT* const sFx = sX;                               // [NF][R][TX + 1]
            FT* const sFy = sFx + NF * G_::FXE;               // [NF][R + 1][TX]
            // pointwise global operands, in flight while the fluxes are computed
            FT gm[FPG], ph = FT(0), phx = FT(0), phy = FT(0);
            if (cell) {
                if (HAS_GM) {
#pragma unroll
                    for (int s = 0; s < FPG; ++s) gm[s] = c.Gm[F0 + s][p];
                }
                if (F0 < 2 && c.pHY) {
                    ph = c.pHY[p];
                    if (F0 == 0) phx = c.pHY[p - 1];
                    if (F0 + FPG > 1) phy = c.pHY[p - sy];
                }
            }
            // the reads of the previous level's exchange buffers are ordered before this level's writes (warps parked at
            // bar.sync cost no issue slots: an mbarrier-polled exchange with early arrive / late wait measured 10 % slower)
            named_sync(1 + GRP, GT);
            tmau::mbar_wait(&full[git & 3], (git >> 2) & 1);

            FT Fx[FPG], Fy[FPG], dFz[FPG];
            if (cell) {
#pragma unroll
                for (int s = 0; s < FPG; ++s) {
                    const int f = F0 + s;
                    if (f == 0) cell_fluxes_xy<FT, ZW, ZT, 0, PE, NF>(c, k, S, so, 0, e, it == 0, Fx[s], Fy[s], Fz[s]);
                    else if (f == 1) cell_fluxes_xy<FT, ZW, ZT, 1, PE, NF>(c, k, S, so, 1, e, it == 0, Fx[s], Fy[s], Fz[s]);
                    else if (f == 2) cell_fluxes_xy<FT, ZW, ZT, 2, PE, NF>(c, k, S, so, 2, e, it == 0, Fx[s], Fy[s], Fz[s]);
                    else cell_fluxes_xy<FT, ZW, ZT, 3, PE, NF>(c, k, S, so, f, e, it == 0, Fx[s], Fy[s], Fz[s]);
                    sFx[f * G_::FXE + ty * (TX + 1) + (f == 0 ? tx + 1 : tx)] = Fx[s];
                    sFy[f * G_::FYE + (f == 1 ? ty + 1 : ty) * TX + tx] = Fy[s];
                    {
                        if (f == 0) cell_flux_z<FT, ZW, ZT, 0, PE, NF>(c, k, S, so, 0, e, Fz[s], dFz[s]);
                        else if (f == 1) cell_flux_z<FT, ZW, ZT, 1, PE, NF>(c, k, S, so, 1, e, Fz[s], dFz[s]);
                        else if (f == 2) cell_flux_z<FT, ZW, ZT, 2, PE, NF>(c, k, S, so, 2, e, Fz[s], dFz[s]);
                        else cell_flux_z<FT, ZW, ZT, 3, PE, NF>(c, k, S, so, f, e, Fz[s], dFz[s]);
                    }
                }
            } else if (edge) {
                // x faces of column -1 (u) / TX (others), rows 0 .. nrows-1; y faces of row -1 (v) / nrows (others)
                const int rx = (min(tx, nrows - 1) + HALO) * BX + COL0;
                const int ey = HALO * BX + tx + COL0;
#pragma unroll
                for (int s = 0; s < FPG; ++s) {
                    const int f = F0 + s;
                    FT ex, ey_;
                    if (f == 0) {
                        ex = fluxs<FT, ZW, ZT, 0, 0, 0, PE, NF>(c, k, S, so, 0, rx - 1);
                        ey_ = fluxs<FT, ZW, ZT, 1, 0, 0, PE, NF>(c, k, S, so, 0, ey + nrows * BX);
                    } else if (f == 1) {
                        ex = fluxs<FT, ZW, ZT, 0, 1, 0, PE, NF>(c, k, S, so, 1, rx + TX);
                        ey_ = fluxs<FT, ZW, ZT, 1, 1, 0, PE, NF>(c, k, S, so, 1, ey - BX);
                    } else if (f == 2) {
                        ex = fluxs<FT, ZW, ZT, 0, 2, 0, PE, NF>(c, k, S, so, 2, rx + TX);
                        ey_ = fluxs<FT, ZW, ZT, 1, 2, 0, PE, NF>(c, k, S, so, 2, ey + nrows * BX);
                    } else {
                        ex = fluxs<FT, ZW, ZT, 0, 3, 0, PE, NF>(c, k, S, so, f, rx + TX);
                        ey_ = fluxs<FT, ZW, ZT, 1, 3, 0, PE, NF>(c, k, S, so, f, ey + nrows * BX);
                    }
                    if (tx < nrows) sFx[f * G_::FXE + tx * (TX + 1) + (f == 0 ? 0 : TX)] = ex;
                    sFy[f * G_::FYE + (f == 1 ? 0 : nrows) * TX + tx] = ey_;
                }
            }
            named_sync(1 + GRP, GT);              // faces published; this group's stencil reads of the level are finished:
            if (edge && tx == 0) tmau::mbar_arrive(&done[git & 3]);     // the producer may refill the slot of level k-2 two levels on
            if (cell) {
#pragma unroll
                for (int s = 0; s < FPG; ++s) {
                    const int f = F0 + s;
                    const FT ox = sFx[f * G_::FXE + ty * (TX + 1) + (f == 0 ? tx : tx + 1)];
                    const FT oy = sFy[f * G_::FYE + (f == 1 ? ty : ty + 1) * TX + tx];
                    const FT dFx = f == 0 ? Fx[s] - ox : ox - Fx[s];
                    const FT dFy = f == 1 ? Fy[s] - oy : oy - Fy[s];
                    FT Gv;
                    if constexpr (ZT) {           // Az / V = 1 / Δz of the level (cell for u, v, c; face for w)
                        const FT iz = __ldg((f == 2 ? c.izF : c.izC) + k);
                        Gv = f < 3 ? -fma(cmx, dFx, fma(cmy, dFy, (iz * FT(1.0 / 24.0)) * dFz[s]))
                                   : -fma(ctx_, dFx, fma(cty, dFy, (iz * FT(0.5)) * dFz[s]));
                        if (f != 2) {             // apply_z_bcs! (apply_flux_bcs.jl:111-160): constant Flux BCs
                            if (k == 1) Gv = fma(c.fbb[f], iz, Gv);
                            if (k == c.Nz) Gv = fma(-c.fbt[f], iz, Gv);
                        }
                    } else {
                        Gv = f < 3 ? -fma(cmx, dFx, fma(cmy, dFy, cmz * dFz[s]))
                                   : -fma(ctx_, dFx, fma(cty, dFy, ctz * dFz[s]));
                    }
                    if (f == 0) {
                        if (c.fplane) {           // - x_f_cross_U = + f * ℑxyᶠᶜᵃ(v)   (f_plane.jl:42)
                            const FT* v = S + 1 * SLOTS * PE + so[3] + e;
                            FT a0 = FT(0.5) * (v[-1] + v[0]), a1 = FT(0.5) * (v[BX - 1] + v[BX]);
                            Gv = Gv - (-c.f * (FT(0.5) * (a0 + a1)));
                        }
                        if (c.pHY) Gv = Gv - (ph - phx) * c.invdx;
                    } else if (f == 1) {
                        if (c.fplane) {           // - y_f_cross_U = - f * ℑxyᶜᶠᵃ(u)   (f_plane.jl:43)
                            const FT* u = S + so[3] + e;
                            FT a0 = FT(0.5) * (u[-BX] + u[1 - BX]), a1 = FT(0.5) * (u[0] + u[1]);
                            Gv = Gv - (c.f * (FT(0.5) * (a0 + a1)));
                        }
                        if (c.pHY) Gv = Gv - (ph - phy) * c.invdy;
                    }
                    if constexpr (FRC) {          // + forcing, last in the sum (Relaxation at the field's own nodes)
                        if (c.frc[f].on) Gv = Gv + relaxation(c.frc[f], i0 + tx, j0 + ty, k, S[f * SLOTS * PE + so[3] + e]);
                    }
                    if constexpr (ACC) Gv = Gv + c.Gn[f][p];
                    c.Gn[f][p] = Gv;
                    if (c.do_sub) {
                        const FT ps = S[f * SLOTS * PE + so[3] + e];
                        FT nv = fma(c.ca, Gv, ps);
                        if (HAS_GM) nv = fma(c.cb, gm[s], nv);
                        c.nw[f][p] = nv;
                    }
                }
            }
            p += sz;
        }
    }
}

template <class FT, bool ZW, int ZT, int NT, bool HAS_GM, bool ACC, int R, bool FRC>
__global__ void __launch_bounds__(TX*(Groups<NT>::NG*(R + 1) + 1), 1)
tendency_fused_kernel(const __grid_constant__ KArgs<FT, 3 + NT, FRC> c) {
    using GR = Groups<NT>;
    constexpr int NF = GR::NF, NG = GR::NG;
    using G_ = Geo<FT, R, NF>;
    constexpr int PE = G_::PE;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long full[4], done[4];
    FT* const S = reinterpret_cast<FT*>(smem_raw);                  // rings: field f, slot s at (f * SLOTS + s) * PE
    FT* const sX = S + NF * SLOTS * PE;                             // exchange buffers
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int q = 0; q < 4; ++q) { tmau::mbar_init(&full[q], 1); tmau::mbar_init(&done[q], NG); }
        tmau::mbar_init_fence();
    }
    __syncthreads();
    if (warp == NG * (R + 1)) {
        // ---- producer warp -------------------------------------------------------------------------------
        unsigned git = 0;
        Work wk(c.ntiles, c.Nz, c.chunk);
        int tile, kfirst, len;
        const bool lead = (threadIdx.x & 31) == 0;
        while (wk.next(tile, kfirst, len)) {
            tile += c.tile0 + (tile >= c.tsplit ? c.tskip : 0);
            const int bx = tile % c.ntx, by = tile / c.ntx;
            const int i0 = 1 + bx * TX, j0 = 1 + by * R, k0 = 1 + kfirst;
            const int cx = i0 - HALO - 2 + c.O[0], cy = j0 - HALO - 1 + c.O[1], cz0 = c.O[2] - 1;
            __syncthreads();
            if (lead) {
                unsigned long long* pb = &full[git & 3];
                tmau::mbar_expect_tx(pb, 7u * NF * G_::BOX_BYTES);
                for (int L = k0 - 3; L <= k0 + 3; ++L)
#pragma unroll
                    for (int f = 0; f < NF; ++f)
                        tmau::tma_load_3d(S + (f * SLOTS + (L & (SLOTS - 1))) * PE, &c.tm[f], cx, cy, L + cz0, pb);
            }
            for (int it = 0; it < len; ++it, ++git) {
                if (lead && it + 1 < len) {       // the planes level k+1 adds: level k+4 into the slot of level k-4
                    const int k = k0 + it;
                    // its slot held level k-4: last read in iteration it-2 (it-1 for the bottom face of the first level)
                    if (it >= 1) { const unsigned w = it == 1 ? git - 1 : git - 2; tmau::mbar_wait(&done[w & 3], (w >> 2) & 1); }
                    unsigned long long* nb = &full[(git + 1) & 3];
                    tmau::mbar_expect_tx(nb, (unsigned)NF * G_::BOX_BYTES);
#pragma unroll
                    for (int f = 0; f < NF; ++f)
                        tmau::tma_load_3d(S + (f * SLOTS + ((k + 4) & (SLOTS - 1))) * PE, &c.tm[f], cx, cy, k + 4 + cz0, nb);
                }
            }
        }
        return;
    }
    const int grp = warp / (R + 1);
    if (grp == 0) group_main<FT, ZW, ZT, NT, HAS_GM, ACC, R, 0, FRC>(c, S, sX, full, done);
    else if (grp == 1) group_main<FT, ZW, ZT, NT, HAS_GM, ACC, R, 1, FRC>(c, S, sX, full, done);
    else if (NG > 2) group_main<FT, ZW, ZT, NT, HAS_GM, ACC, R, (NG > 2 ? 2 : 0), FRC>(c, S, sX, full, done);
}

// ---- host side --------------------------------------------------------------------------------
// Relaxation forcing of the fused fields as a pointwise pass into G^n (G^n = F, or G^n += F over the closure's part and / or
// the background terms), for the accumulate instantiations to add the rest: the forced FP64 variants with a tracer that would
// spill with the term in the epilogue (launch_frc).  The accumulate form adds G^n of EVERY field, so without precomputed terms
// the unforced fields' G^n are cleared here
template <class FT>
struct RelaxPass {
    int nf, acc;
    const FT* psi[FUSED_MAXF];
    FT* Gn[FUSED_MAXF];
    Relax<FT> frc[FUSED_MAXF];
    long long sy, sz;
    int N[3];
};
template <class FT>
__global__ void __launch_bounds__(128) relaxation_pass_kernel(const __grid_constant__ RelaxPass<FT> a) {
    const int i = 1 + blockIdx.x * blockDim.x + threadIdx.x, j = 1 + blockIdx.y * blockDim.y + threadIdx.y, k = 1 + blockIdx.z;
    if (i > a.N[0] || j > a.N[1]) return;
    const long long p = i + j * a.sy + k * a.sz;
    for (int f = 0; f < a.nf; ++f) {
        if (!a.frc[f].on) {
            if (!a.acc) a.Gn[f][p] = FT(0);
            continue;
        }
        const FT F = relaxation(a.frc[f], i, j, k, a.psi[f][p]);
        a.Gn[f][p] = a.acc ? a.Gn[f][p] + F : F;
    }
}
template <class FT, bool ZW, int ZT, int NT, bool HAS_GM, bool ACC, int R, bool FRC>
static void launch_variant(const Phys<FT>& P, const FusedFields<FT>& a, int part) {
    using GR = Groups<NT>;
    constexpr int NF = GR::NF;
    using G_ = Geo<FT, R, NF>;
    static_assert(G_::SMEM <= 227 * 1024 - 64, "shared memory budget");
    const GridD<FT>& g = P.g;
    KArgs<FT, NF, FRC> c;
    for (int f = 0; f < NF; ++f) {
        c.tm[f] = tmau::make_map<FT>(g, a.state[f] - g.off0, BX, G_::BY);
        c.Gm[f] = a.Gm[f]; c.Gn[f] = a.Gn[f]; c.nw[f] = a.nw[f];
        if constexpr (FRC) c.frc[f] = P.frc[f];
    }
    c.pHY = a.pHY;
    c.sy = g.st[1]; c.sz = g.st[2];
    for (int d = 0; d < 3; ++d) c.O[d] = g.O[d];
    c.Ny = g.N[1]; c.Nz = g.N[2];
    c.ntx = g.N[0] / TX;
    {
        const int nty = cdiv(g.N[1], R);
        c.ntiles = c.ntx * nty;
        c.tile0 = 0; c.tsplit = 1 << 30; c.tskip = 0;
        if (part) {
            // interior tile rows 1 .. nint; boundary tile rows 0 and the nb_hi at the high end
            const int nint = interior_tile_rows(g.N[1], R), nb_hi = nty - 1 - nint;
            if (part == 1) { c.tile0 = c.ntx; c.ntiles = nint * c.ntx; }
            else { c.ntiles = (1 + nb_hi) * c.ntx; c.tsplit = c.ntx; c.tskip = nint * c.ntx; }
        }
    }
    c.invdx = 1 / g.d[0]; c.invdy = 1 / g.d[1];
    if (ZT) {
        c.cf[0] = c.invdx; c.cf[1] = c.invdy; c.cf[2] = FT(0);
        c.izC = g.izC; c.izF = g.izF; c.tabF = P.wzp[0]; c.tabC = P.wzp[1];
        // with a.accumulate the closure's part is already in G^n: no viscous terms here
        const FT nu = (P.closure == CLO_3D && !a.accumulate) ? P.nu : FT(0), kap = (P.closure == CLO_3D && !a.accumulate) ? P.kappa[0] : FT(0);
        c.v24 = -24 * nu; c.vh[0] = c.v24 * c.invdx; c.vh[1] = c.v24 * c.invdy;
        c.t2 = -2 * kap; c.th[0] = c.t2 * c.invdx; c.th[1] = c.t2 * c.invdy;
        for (int f = 0; f < NF; ++f) {
            c.fbb[f] = a.fbc[f].kind[4] == 2 ? a.fbc[f].val[4] : FT(0);
            c.fbt[f] = a.fbc[f].kind[5] == 2 ? a.fbc[f].val[5] : FT(0);
        }
    } else {
        const FT invV = 1 / ((g.d[0] * g.d[1]) * g.d[2]);
        c.cf[0] = (g.d[1] * g.d[2]) * invV; c.cf[1] = (g.d[0] * g.d[2]) * invV; c.cf[2] = (g.d[0] * g.d[1]) * invV;
        c.izC = c.izF = c.tabF = c.tabC = nullptr;
    }
    c.f = P.f; c.fplane = P.fplane;
    const Substep<FT>& ss = a.ss;
    c.do_sub = ss.mode != SUB_NONE;
    c.ca = ss.mode == SUB_RK3_FIRST ? ss.c1 : ss.dt * ss.c1;
    c.cb = ss.mode == SUB_RK3 ? ss.dt * ss.c2 : (ss.mode == SUB_AB2 ? -(ss.dt * ss.c2) : FT(0));
    auto kern = tendency_fused_kernel<FT, ZW, ZT, NT, HAS_GM, ACC, R, FRC>;
    static bool attr_set = false;      // per instantiation
    if (!attr_set) {
        OB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G_::SMEM));
        attr_set = true;
    }
    const long long T = (long long)c.ntiles * c.Nz;
    if (T >= (1LL << 30)) throw Error("tendency_fused: grid too large for the 32-bit work decomposition");
    const int grid = (int)std::max(1LL, std::min((long long)tmau::sm_count(), T / 8));
    c.chunk = cdiv((long long)(c.ntiles - (c.ntiles / grid) * grid) * c.Nz, grid);
    kern<<<grid, TX * (GR::NG * (R + 1) + 1), G_::SMEM, stream()>>>(c);
    OB_LAUNCH_CHECK();
}

template <class FT, bool ZW, int ZT, int NT, int R, bool FRC>
static void launch_gm(const Phys<FT>& P, const FusedFields<FT>& a, int part) {
    const bool has_gm = a.ss.mode == SUB_RK3 || a.ss.mode == SUB_AB2;
    // the accumulate form (closure's part, backgrounds and / or the forcing precomputed into G^n) exists for the variants with
    // a tracer; the tendency plan gives the variant without one no precomputed terms
    if constexpr (NT == 1) {
        if (a.accumulate || a.gn_terms) {
            if (has_gm) launch_variant<FT, ZW, ZT, NT, true, true, R, FRC>(P, a, part);
            else launch_variant<FT, ZW, ZT, NT, false, true, R, FRC>(P, a, part);
            return;
        }
    }
    if (has_gm) launch_variant<FT, ZW, ZT, NT, true, false, R, FRC>(P, a, part);
    else launch_variant<FT, ZW, ZT, NT, false, false, R, FRC>(P, a, part);
}
// a model with a forced field among the fused ones takes the FRC instantiations (the term in the per-cell epilogue); every
// other keeps the unforced kernels.  The FP64 variants with a tracer are at the 72-register cap already and would spill
// 16-100 bytes more with the term (ptxas -v, sm_100a): there a pointwise pass writes the forcing into G^n and the
// accumulate instantiation adds the rest, one extra read and write of G^n and a read of the field per forced field
template <class FT, bool ZW, int ZT, int NT, int R>
static void launch_frc(const Phys<FT>& P, const FusedFields<FT>& a, int part) {
    constexpr int NF = 3 + NT;
    bool frc = false;
    for (int f = 0; f < NF; ++f) frc = frc || P.frc[f].on;
    if (!frc) return launch_gm<FT, ZW, ZT, NT, R, false>(P, a, part);
    if constexpr (sizeof(FT) == 4 || NT == 0) {
        launch_gm<FT, ZW, ZT, NT, R, true>(P, a, part);
    } else {
        const GridD<FT>& g = P.g;
        if (part != 2) {               // once per stage: before the first (or the only) part
            RelaxPass<FT> r;
            r.nf = NF; r.acc = (a.accumulate || a.gn_terms) ? 1 : 0;
            for (int f = 0; f < NF; ++f) { r.psi[f] = a.state[f]; r.Gn[f] = a.Gn[f]; r.frc[f] = P.frc[f]; }
            r.sy = g.st[1]; r.sz = g.st[2];
            for (int d = 0; d < 3; ++d) r.N[d] = g.N[d];
            dim3 blk(32, 4, 1), grd(cdiv(g.N[0], 32), cdiv(g.N[1], 4), g.N[2]);
            relaxation_pass_kernel<FT><<<grd, blk, 0, stream()>>>(r);
            OB_LAUNCH_CHECK();
        }
        FusedFields<FT> b = a;
        b.gn_terms = true;
        launch_gm<FT, ZW, ZT, NT, R, false>(P, b, part);
    }
}

// the z variant: ZT = 0 Periodic regular z, ZT = 1 Bounded z
template <class FT>
void launch(const Phys<FT>& P, const FusedFields<FT>& a, int part) {
#define GO(ZTV, NTV)                                                                                                   \
    {                                                                                                                  \
        if (P.zweno) launch_frc<FT, true, ZTV, NTV, rows_per_tile(NTV)>(P, a, part);                                   \
        else launch_frc<FT, false, ZTV, NTV, rows_per_tile(NTV)>(P, a, part);                                          \
    }
    if (P.g.topo[2] == OB_BOUNDED) GO(1, 1)
    else if (a.nf == 3) GO(0, 0)
    else GO(0, 1)
#undef GO
}
template void launch<float>(const Phys<float>&, const FusedFields<float>&, int);
template void launch<double>(const Phys<double>&, const FusedFields<double>&, int);

}  // namespace fz
}  // namespace ob
