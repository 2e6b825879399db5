// tendency_tma.cu -- TMA-staged variant of the specialised tendency (+ substep) kernel.
//
// Same arithmetic as tendency_fast.cu (one-sided WENO5, faces shared through registers / shared
// memory, single-reciprocal Float64 weights: weno_fast.cuh).  What changes is the data path: every operand
// of the stencils is staged in shared memory by the Tensor Memory Accelerator:
//   * a block of NW warps owns a 32 x (NW-1) column tile and marches in k; for every array it reads it keeps a
//     RING of (32+6) x (NW-1+6) halo'd planes in shared memory (psi: levels k-3..k+3, advecting velocities:
//     the 1-4 levels their interpolation needs);
//   * warps 0..NW-2 own one row of 32 cells each: three face fluxes per cell and level (x, y, z-top);
//   * warp NW-1 is the EDGE warp: its lane 0 issues `cp.async.bulk.tensor.3d` (SASS UTMALDG) for the planes of
//     level k+1 while all warps compute level k (completion tracked with two alternating mbarriers,
//     expect_tx / try_wait.parity, so no warp ever waits on a global load), and its lanes compute the one extra
//     column of x faces and the one extra row of y faces the tile needs (two flux evaluations against three in
//     the cell warps, so the block-wide barrier that publishes the faces is not held up by it: the first
//     version gave those edge faces to two of the cell warps, and ncu r1d showed 16 % of the stall samples
//     at that barrier);
//   * the z-direction stencil reads the ring, the x/y stencils read the level-k plane;
//   * the pointwise global operands (G^-, pHY') are loaded at the top of the level, before the flux
//     arithmetic, so their latency is hidden (36 % of the stall samples before).
// Tensor maps describe the padded internal layout (common.cuh): 3-D, box (40, NW+5, 1), no swizzle.
#include "internal.h"
#include "weno_fast.cuh"
#include "tma_util.cuh"
#include <cmath>

namespace ob {
namespace tma {

constexpr int TX = 32, NW = 8, HALO = 3, COL0 = HALO + 1;   // NW warps per block
template <class FT> struct Box {
    // The box must START on a 16-byte boundary in x (measured on B200: an odd FP64 start coordinate raises
    // "illegal instruction", tools/tma_probe4.cu), so it starts one column left of the halo: 1 + 3 + 32 + 3 + 1.
    static constexpr int R = NW - 1;                 // rows of cells
    static constexpr int BX = TX + 2 * HALO + 2, BY = R + 2 * HALO;
    static constexpr int PLANE_BYTES = ((BX * BY * (int)sizeof(FT) + 127) / 128) * 128;
    static constexpr int PE = PLANE_BYTES / (int)sizeof(FT);
};

// rings per advected component B: psi + auxiliary advecting velocities.
// aux a of B:      component            level range lo..hi      slots (power of two >= hi-lo+2)
//   B=0 (u):  v [0,0] 2,  w [0,1] 3          B=1 (v):  u [0,0] 2,  w [0,1] 3
//   B=2 (w):  u [-2,1] 5, v [-2,1] 5         B=3 (c):  u [0,0] 2,  v [0,0] 2,  w [0,1] 3
template <int B> struct Cfg {
    static constexpr int NA = B == 3 ? 3 : 2;
    __host__ __device__ static constexpr int comp(int a) {
        return B == 0 ? (a == 0 ? 1 : 2) : B == 1 ? (a == 0 ? 0 : 2) : B == 2 ? (a == 0 ? 0 : 1) : a;
    }
    __host__ __device__ static constexpr int lo(int a) { return B == 2 ? -2 : 0; }
    __host__ __device__ static constexpr int hi(int a) { return B == 2 ? 1 : (comp(a) == 2 ? 1 : 0); }
    // slots >= live levels + 1 prefetched level (any count: the slot index is a compile-time modulo)
    __host__ __device__ static constexpr int sl(int a) { return a >= NA ? 0 : (B == 2 ? 5 : (comp(a) == 2 ? 3 : 2)); }
};
constexpr int PSI_LO = -3, PSI_HI = 3, PSI_SL = 8;

template <class FT>
struct Ctx {
    CUtensorMap tm_psi, tm_aux[3];
    const FT* psi;        // Julia-(0,0,0) pointers for the pointwise (non-stencil) reads / writes
    const FT* pHY;
    const FT* Gm;
    const FT* cor;        // the velocity the Coriolis term interpolates (v for B = 0, u for B = 1)
    FT* Gn;
    FT* psi_new;
    long long s[3];
    int O[3];
    FT area[3], invV, invd[3], f;
    int fplane, Kc, Ny, Nz;
    Substep<FT> ss;
};

using tmau::mbar_init; using tmau::mbar_init_fence; using tmau::mbar_expect_tx; using tmau::mbar_wait; using tmau::tma_load_3d;

// position inside the staged data: level L (Julia k), tile row / column including the halo offset
struct P3 { int L, row, col; };
template <int D> __device__ __forceinline__ P3 shp(P3 q, int n) {
    if (D == 0) q.col += n; else if (D == 1) q.row += n; else q.L += n;
    return q;
}

template <class FT, int B>
struct Rings {
    const FT* psi;
    const FT* aux[3];
    __device__ __forceinline__ FT P(P3 q) const {
        return psi[((q.L + 8) & (PSI_SL - 1)) * Box<FT>::PE + q.row * Box<FT>::BX + q.col];
    }
    template <int COMP> __device__ __forceinline__ FT V(P3 q) const {
        if constexpr (COMP == B) return P(q);
        else {
            constexpr int a = Cfg<B>::comp(0) == COMP ? 0 : (Cfg<B>::comp(1) == COMP ? 1 : 2);
            return aux[a][((q.L + 60) % Cfg<B>::sl(a)) * Box<FT>::PE + q.row * Box<FT>::BX + q.col];
        }
    }
};

// (I(q) + I(q + 1))/2 along direction D of velocity component COMP (see wf::interp4)
template <class FT, int B, int COMP, int D>
__device__ __forceinline__ FT I4r(const Rings<FT, B>& r, P3 q) {
    return wf::interp4<FT>(r.template V<COMP>(shp<D>(q, -1)), r.template V<COMP>(q), r.template V<COMP>(shp<D>(q, 1)),
                           r.template V<COMP>(shp<D>(q, 2)));
}

// area * upwind flux of psi (component B or tracer) in direction A at position q
// (A == B: cell-centre index; otherwise face index along A)
template <class FT, bool ZW, int A, int B>
__device__ __forceinline__ FT flux_at(const Rings<FT, B>& r, const Ctx<FT>& c, P3 q) {
    FT ut;
    P3 pf = q;
    if constexpr (B == 3) {
        ut = r.template V<A>(q);
    } else if constexpr (A == B) {
        ut = I4r<FT, B, A, A>(r, q);
        pf = shp<A>(q, 1);
    } else {
        ut = I4r<FT, B, A, B>(r, shp<B>(q, -1));
    }
    const FT w0 = r.P(shp<A>(pf, -3)), w1 = r.P(shp<A>(pf, -2)), w2 = r.P(shp<A>(pf, -1)), w3 = r.P(pf),
             w4 = r.P(shp<A>(pf, 1)), w5 = r.P(shp<A>(pf, 2));
    FT rec = wf::weno_upwind<FT, ZW>(ut > FT(0), w0, w1, w2, w3, w4, w5);
    return c.area[A] * (ut * rec);
}

template <class FT, bool ZW, int B>
__global__ void __launch_bounds__(TX * NW, 3) tendency_tma_kernel(const __grid_constant__ Ctx<FT> c) {
    using BXs = Box<FT>;
    using CF = Cfg<B>;
    constexpr int R = BXs::R;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ FT sFx[2][R][TX + 1];
    __shared__ FT sFy[2][R + 1][TX];
    __shared__ __align__(8) unsigned long long bars[2];

    FT* ring_psi = reinterpret_cast<FT*>(smem_raw);
    FT* ring_aux[3];
    {
        FT* q = ring_psi + PSI_SL * BXs::PE;
#pragma unroll
        for (int a = 0; a < 3; ++a) { ring_aux[a] = q; q += CF::sl(a) * BXs::PE; }
    }
    const int tx = threadIdx.x, ty = threadIdx.y;
    const bool edge = ty == R, producer = edge && tx == 0;
    const int i0 = 1 + blockIdx.x * TX, j0 = 1 + blockIdx.y * R, k0 = 1 + blockIdx.z * c.Kc;
    const int nrows = min(R, c.Ny - j0 + 1);           // the last tile in y may be ragged
    const int Kc = min(c.Kc, c.Nz - k0 + 1);           // ... and so may the last chunk in z
    const int cx = i0 - HALO - 2 + c.O[0], cy = j0 - HALO - 1 + c.O[1], cz0 = c.O[2] - 1;   // array coords

    if (producer) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_init_fence();
    }
    __syncthreads();

    auto load_psi = [&](int L, unsigned long long* bar) {
        tma_load_3d(ring_psi + ((L + 8) & (PSI_SL - 1)) * BXs::PE, &c.tm_psi, cx, cy, L + cz0, bar);
    };
    auto load_aux = [&](int a, int L, unsigned long long* bar) {
        tma_load_3d(ring_aux[a] + ((L + 60) % CF::sl(a)) * BXs::PE, &c.tm_aux[a], cx, cy, L + cz0, bar);
    };
    if (producer) {
        // prologue: everything iteration 0 (and the carried z face) needs
        int planes = (PSI_HI - PSI_LO + 1);
#pragma unroll
        for (int a = 0; a < CF::NA; ++a) planes += CF::hi(a) - CF::lo(a) + 1;
        mbar_expect_tx(&bars[0], planes * BXs::BX * BXs::BY * (unsigned)sizeof(FT));
        for (int L = k0 + PSI_LO; L <= k0 + PSI_HI; ++L) load_psi(L, &bars[0]);
#pragma unroll
        for (int a = 0; a < CF::NA; ++a)
            for (int L = k0 + CF::lo(a); L <= k0 + CF::hi(a); ++L) load_aux(a, L, &bars[0]);
    }

    Rings<FT, B> Rg;
    Rg.psi = ring_psi;
    Rg.aux[0] = ring_aux[0]; Rg.aux[1] = ring_aux[1]; Rg.aux[2] = ring_aux[2];

    constexpr bool XLOW = (B == 0), YLOW = (B == 1), ZLOW = (B == 2);
    const bool cell = !edge && ty < nrows;
    const long long sx = c.s[0], sy = c.s[1], sz = c.s[2];
    long long p = (i0 + tx) * sx + (j0 + ty) * sy + k0 * sz;
    FT Fz_carry = FT(0);
    const int mode = c.ss.mode;
    const bool has_pHY = (B == 0 || B == 1) && c.pHY != nullptr, has_Gm = mode == SUB_RK3 || mode == SUB_AB2;
    const long long sB = B == 0 ? sx : sy;

    for (int it = 0; it < Kc; ++it) {
        const int k = k0 + it, buf = it & 1;
        if (producer && it + 1 < Kc) {      // prefetch the planes level k+1 adds
            unsigned long long* nb = &bars[(it + 1) & 1];
            mbar_expect_tx(nb, (1 + CF::NA) * BXs::BX * BXs::BY * (unsigned)sizeof(FT));
            load_psi(k + 1 + PSI_HI, nb);
#pragma unroll
            for (int a = 0; a < CF::NA; ++a) load_aux(a, k + 1 + CF::hi(a), nb);
        }
        // pointwise global operands, in flight while the fluxes are computed
        FT gm = FT(0), ph1 = FT(0), ph0 = FT(0);
        if (cell) {
            if (has_Gm) gm = c.Gm[p];
            if (has_pHY) { ph1 = c.pHY[p]; ph0 = c.pHY[p - sB]; }
        }
        mbar_wait(&bars[it & 1], (it >> 1) & 1);

        const P3 q{k, ty + HALO, tx + COL0};
        FT Fx = FT(0), Fy = FT(0), dFz = FT(0);
        if (cell) {
            if (it == 0) Fz_carry = flux_at<FT, ZW, 2, B>(Rg, c, ZLOW ? shp<2>(q, -1) : q);
            Fx = flux_at<FT, ZW, 0, B>(Rg, c, q);
            Fy = flux_at<FT, ZW, 1, B>(Rg, c, q);
            sFx[buf][ty][XLOW ? tx + 1 : tx] = Fx;
            sFy[buf][YLOW ? ty + 1 : ty][tx] = Fy;
            FT Fz_new = flux_at<FT, ZW, 2, B>(Rg, c, ZLOW ? q : shp<2>(q, 1));
            dFz = Fz_new - Fz_carry;
            Fz_carry = Fz_new;
        } else if (edge) {
            if (tx < nrows) {
                P3 e{k, tx + HALO, (XLOW ? -1 : TX) + COL0};
                sFx[buf][tx][XLOW ? 0 : TX] = flux_at<FT, ZW, 0, B>(Rg, c, e);
            }
            P3 e{k, (YLOW ? -1 : nrows) + HALO, tx + COL0};
            sFy[buf][YLOW ? 0 : nrows][tx] = flux_at<FT, ZW, 1, B>(Rg, c, e);
        }
        __syncthreads();
        if (cell) {
            FT dFx = XLOW ? (Fx - sFx[buf][ty][tx]) : (sFx[buf][ty][tx + 1] - Fx);
            FT dFy = YLOW ? (Fy - sFy[buf][ty][tx]) : (sFy[buf][ty + 1][tx] - Fy);
            FT G = -(c.invV * ((dFx + dFy) + dFz));
            if (B == 0) {
                if (c.fplane) {
                    const FT* v = c.cor;
                    FT a0 = FT(0.5) * (v[p - sx] + v[p]), a1 = FT(0.5) * (v[p - sx + sy] + v[p + sy]);
                    G = G - (-c.f * (FT(0.5) * (a0 + a1)));
                }
                if (has_pHY) G = G - (ph1 - ph0) * c.invd[0];
            } else if (B == 1) {
                if (c.fplane) {
                    const FT* u = c.cor;
                    FT a0 = FT(0.5) * (u[p - sy] + u[p + sx - sy]), a1 = FT(0.5) * (u[p] + u[p + sx]);
                    G = G - (c.f * (FT(0.5) * (a0 + a1)));
                }
                if (has_pHY) G = G - (ph1 - ph0) * c.invd[1];
            }
            c.Gn[p] = G;
            const FT ps = Rg.P(q);
            if (mode == SUB_RK3_FIRST) c.psi_new[p] = ps + c.ss.c1 * G;
            else if (mode == SUB_RK3) c.psi_new[p] = ps + c.ss.dt * (c.ss.c1 * G + c.ss.c2 * gm);
            else if (mode == SUB_AB2) c.psi_new[p] = ps + c.ss.dt * (c.ss.c1 * G - c.ss.c2 * gm);
        }
        p += sz;
    }
}

// ---- host side --------------------------------------------------------------------------------
using tmau::make_map;

template <class FT, bool ZW, int B>
static void launch_one(Ctx<FT>& c, const GridD<FT>& g, const FT* const U[3], const FT* psi) {
    using CF = Cfg<B>;
    using BXs = Box<FT>;
    c.tm_psi = make_map<FT>(g, psi - g.off0, BXs::BX, BXs::BY);
    int slots = PSI_SL;
    for (int a = 0; a < CF::NA; ++a) {
        slots += CF::sl(a);
        c.tm_aux[a] = make_map<FT>(g, U[CF::comp(a)] - g.off0, BXs::BX, BXs::BY);
    }
    size_t smem = (size_t)slots * BXs::PLANE_BYTES;
    auto kern = tendency_tma_kernel<FT, ZW, B>;
    static bool attr_set = false;      // one flag per kernel instantiation (function-local static of a template)
    if (!attr_set) {
        OB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
        attr_set = true;
    }
    // chunks of 32 levels in z (the last one may be shorter).  A wave-quantisation model (blocks as a multiple of the
    // resident block count, prologue of ~2 levels per chunk) picked 6 chunks at 256^3 and measured SLOWER than 8
    // (3.82 vs 3.74 ms per step), so the plain rule stays.
    c.Kc = cdiv(g.N[2], cdiv(g.N[2], 32));
    dim3 blk(TX, NW), grd(g.N[0] / TX, cdiv(g.N[1], BXs::R), cdiv(g.N[2], c.Kc));
    kern<<<grd, blk, smem, stream()>>>(c);
    OB_LAUNCH_CHECK();
}

// eligibility (3-D grid, Nx % 32 == 0, 16-byte row strides, field not forced) is decided by the tendency plan
// (capi.cu: plan_tendencies)
template <class FT>
void launch(const Phys<FT>& P, int comp, const FT* const U[3], const FT* psi, const FT* pHY, FT* Gn, const FT* Gm,
            FT* psi_new, const Substep<FT>& ss) {
    const GridD<FT>& g = P.g;
    Ctx<FT> c;
    c.psi = psi; c.pHY = pHY; c.Gm = Gm; c.Gn = Gn; c.psi_new = psi_new; c.ss = ss;
    c.cor = comp == 0 ? U[1] : U[0];
    for (int d = 0; d < 3; ++d) { c.s[d] = g.st[d]; c.O[d] = g.O[d]; c.invd[d] = 1 / g.d[d]; }
    c.area[0] = g.d[1] * g.d[2]; c.area[1] = g.d[0] * g.d[2]; c.area[2] = g.d[0] * g.d[1];
    c.invV = 1 / ((g.d[0] * g.d[1]) * g.d[2]);
    c.f = P.f; c.fplane = P.fplane;
    c.Ny = g.N[1]; c.Nz = g.N[2];
    c.Kc = g.N[2];
#define GO(ZWV)                                                         \
    switch (comp) {                                                     \
        case 0: launch_one<FT, ZWV, 0>(c, g, U, psi); break;            \
        case 1: launch_one<FT, ZWV, 1>(c, g, U, psi); break;            \
        case 2: launch_one<FT, ZWV, 2>(c, g, U, psi); break;            \
        default: launch_one<FT, ZWV, 3>(c, g, U, psi); break;           \
    }
    if (P.zweno) { GO(true) } else { GO(false) }
#undef GO
}
template void launch<float>(const Phys<float>&, int, const float* const[3], const float*, const float*, float*,
                            const float*, float*, const Substep<float>&);
template void launch<double>(const Phys<double>&, int, const double* const[3], const double*, const double*, double*,
                             const double*, double*, const Substep<double>&);
}  // namespace tma
}  // namespace ob
